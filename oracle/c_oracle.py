"""ctypes wrapper of oracle/coopsearch_oracle.c -- TEST INFRASTRUCTURE (see that file's header)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "liboracle.so")
META_WORDS = 8


class OfSpec(C.Structure):
    _fields_ = [("n", C.c_int32), ("m", C.c_int32), ("M", C.c_int32), ("R", C.c_int32), ("T", C.c_int32),
                ("agent_mode", C.c_int32), ("target_mode", C.c_int32), ("variant", C.c_int32), ("auto_reset", C.c_int32),
                ("v", C.c_double), ("detect_prob", C.c_double), ("safe_dist", C.c_double), ("force_dist", C.c_double),
                ("seed", C.c_uint32)]


class OsSpec(C.Structure):
    _fields_ = [("n", C.c_int32), ("m", C.c_int32), ("M", C.c_int32), ("R", C.c_int32), ("agent_mode", C.c_int32),
                ("target_mode", C.c_int32), ("auto_reset", C.c_int32), ("seed", C.c_uint32)]


def build(force=False):
    src = os.path.join(HERE, "coopsearch_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.run(["make", "-C", HERE, "-B", "liboracle.so"], check=True, capture_output=True)
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        for name in ("of_flight_reset", "of_flight_step", "of_flight_obs_state", "os_reset", "os_step", "os_views", "of_philox", "of_set_square"):
            getattr(_lib, name).restype = None
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


_threads = 1
_pool = None


def set_square(mode):
    """How the flight oracle squares coordinate differences: "pow" (default) = libm pow(v, 2.0), what Python's ** does in
    the reference; "mul" = v * v, what the CUDA kernels do (the two differ in the last bit for ~0.08 % of arguments)."""
    lib().of_set_square(C.c_int({"pow": 0, "mul": 1}[mode]))


def set_threads(k):
    """Host threads used to fan env blocks out (the C code is single-threaded; ctypes releases the GIL)."""
    global _threads, _pool
    k = max(1, int(k))
    if k != _threads:
        _threads = k
        if _pool is not None:
            _pool.shutdown()
        _pool = None


def _fanout(E, fn):
    """Calls fn(e0, e1) over contiguous blocks of [0, E) on the thread pool."""
    global _pool
    if _threads == 1 or E < 2 * _threads:
        fn(0, E)
        return
    if _pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _pool = ThreadPoolExecutor(max_workers=_threads)
    step = (E + _threads - 1) // _threads
    futs = [_pool.submit(fn, e0, min(E, e0 + step)) for e0 in range(0, E, step)]
    for f in futs:
        f.result()


def scaled_template(template, m, map_size):
    """[m][5] rows x, y, sx, sy, random with the a = map_size/10 scale applied (flight_env_easy.py:97-103)."""
    a = map_size / 10
    rows = np.zeros((m, 5))
    if template is not None:
        for j in range(m):
            rows[j] = [a * template["x"][j], a * template["y"][j], a * template["dx"][j], a * template["dy"][j],
                       1.0 if template["deter"][j] == "f" else 0.0]
    return rows


class FlightBatch:
    """E env instances of the flight_easy ("easy") or flight ("probmap") oracle, stepped in C."""

    def __init__(self, spec, template, seed, env_id_base, num_envs, auto_reset=False):
        self.spec = spec
        self.E = E = int(num_envs)
        self.base = int(env_id_base)
        n, m, M = spec.n_agents, spec.target_num, spec.map_size
        self.cs = OfSpec(n=n, m=m, M=M, R=spec.view_range, T=spec.time_limit, agent_mode=spec.agent_mode,
                         target_mode=spec.target_mode, variant=int(spec.variant == "probmap"), auto_reset=int(auto_reset),
                         v=float(spec.velocity), detect_prob=float(spec.detect_prob), safe_dist=float(spec.safe_dist),
                         force_dist=float(spec.force_dist), seed=int(seed) & 0xFFFFFFFF)
        self.tmpl = scaled_template(template, m, M)
        self.xy = np.zeros((E, n, 2))
        self.yaw = np.zeros((E, n))
        self.tgt = np.zeros((E, m, 2))
        self.meta = np.zeros((E, META_WORDS), np.uint32)
        self.meta[:, 4] = 0xFFFFFFFF                     # first reset opens episode 0
        self.map = np.zeros((E, M, M)) if spec.variant == "probmap" else None
        self.reward = np.zeros(E)
        self.terminated = np.zeros(E, np.uint8)
        self.win = np.zeros(E, np.uint8)
        self.touched = np.zeros(1, np.int64)

    def reset(self, targets=None, init=False, mask=None, keep_episode=False):
        if targets is not None:
            self.tgt[...] = targets
        m8 = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        f, sl = lib().of_flight_reset, self._sl

        def run(e0, e1):
            tc = np.zeros(1, np.int64)
            f(C.byref(self.cs), e1 - e0, self.base + e0, _p(self.tmpl), _p(sl(m8, e0, e1)), int(targets is not None),
              int(keep_episode), int(init), _p(self.xy[e0:e1]), _p(self.yaw[e0:e1]), _p(self.tgt[e0:e1]),
              _p(self.meta[e0:e1]), _p(sl(self.map, e0, e1)), _p(tc))
            self._tc.append(int(tc[0]))
        self._tc = []
        _fanout(self.E, run)
        self.touched[0] += sum(self._tc)

    def step(self, actions=None):
        a = None if actions is None else np.ascontiguousarray(actions, np.uint8)
        f, sl = lib().of_flight_step, self._sl

        def run(e0, e1):
            tc = np.zeros(1, np.int64)
            f(C.byref(self.cs), e1 - e0, self.base + e0, _p(self.tmpl), _p(sl(a, e0, e1)), _p(self.xy[e0:e1]),
              _p(self.yaw[e0:e1]), _p(self.tgt[e0:e1]), _p(self.meta[e0:e1]), _p(sl(self.map, e0, e1)),
              _p(self.reward[e0:e1]), _p(self.terminated[e0:e1]), _p(self.win[e0:e1]), _p(tc))
            self._tc.append(int(tc[0]))
        self._tc = []
        _fanout(self.E, run)
        self.touched[0] += sum(self._tc)
        return self.reward, self.terminated, self.win

    @staticmethod
    def _sl(arr, e0, e1):
        return None if arr is None else arr[e0:e1]

    def obs_state(self):
        n, m = self.spec.n_agents, self.spec.target_num
        obs = np.zeros((self.E, n, 4))
        state = np.zeros((self.E, 4 * n + 3 * m))
        f = lib().of_flight_obs_state
        _fanout(self.E, lambda e0, e1: f(C.byref(self.cs), e1 - e0, _p(self.xy[e0:e1]), _p(self.yaw[e0:e1]),
                                         _p(self.tgt[e0:e1]), _p(self.meta[e0:e1]), _p(obs[e0:e1]), _p(state[e0:e1])))
        return obs, state

    @property
    def found(self):
        return self.meta[:, 0]

    @property
    def out(self):
        return self.meta[:, 2]

    @property
    def time_step(self):
        return self.meta[:, 3]


class SearchBatch:
    """E env instances of the search_env oracle, stepped in C.  With auto_reset a terminating env is reset inside the
    step call, as the kernel does.  After step(): reward / terminated / target_find / terms describe that call's step (of
    the finished episode, where one ended); terms[e] = (-1, 1/freq of agents 0..n-1, 10 * targets found) are the reward's
    summands, zero for an env that did not step.  Everything else holds the state after the call."""

    def __init__(self, spec, seed, env_id_base, num_envs, auto_reset=False):
        self.spec = spec
        self.E = E = int(num_envs)
        self.base = int(env_id_base)
        n, m, M = spec.n_agents, spec.target_num, spec.map_size
        self.cs = OsSpec(n=n, m=m, M=M, R=spec.view_range, agent_mode=spec.agent_mode, target_mode=spec.target_mode,
                         auto_reset=int(auto_reset), seed=int(seed) & 0xFFFFFFFF)
        self.pos = np.zeros((E, n, 2), np.int32)
        self.cells = np.zeros((E, m, 2), np.int32)
        self.tmap = np.zeros((E, M, M), np.uint8)
        self.found = np.zeros((E, m), np.uint8)
        self.freq = np.zeros((E, M, M), np.int32)
        self.counters = np.zeros((E, 4), np.int32)
        self.counters[:, 3] = -1
        self.reward = np.zeros(E)
        self.terminated = np.zeros(E, np.uint8)
        self.target_find = np.zeros(E, np.int32)
        self.terms = np.zeros((E, n + 2))

    def reset(self, cells=None, mask=None):
        if cells is not None:
            self.cells[...] = cells
        m8 = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        f = lib().os_reset
        sl = lambda arr, e0, e1: None if arr is None else arr[e0:e1]
        _fanout(self.E, lambda e0, e1: f(C.byref(self.cs), e1 - e0, self.base + e0, _p(sl(m8, e0, e1)), int(cells is not None),
                                         _p(self.pos[e0:e1]), _p(self.cells[e0:e1]), _p(self.tmap[e0:e1]),
                                         _p(self.found[e0:e1]), _p(self.freq[e0:e1]), _p(self.counters[e0:e1])))

    def step(self, actions=None):
        a = None if actions is None else np.ascontiguousarray(actions, np.uint8)
        f = lib().os_step
        sl = lambda arr, e0, e1: None if arr is None else arr[e0:e1]
        _fanout(self.E, lambda e0, e1: f(C.byref(self.cs), e1 - e0, self.base + e0, _p(sl(a, e0, e1)), _p(self.pos[e0:e1]),
                                         _p(self.cells[e0:e1]), _p(self.tmap[e0:e1]), _p(self.found[e0:e1]),
                                         _p(self.freq[e0:e1]), _p(self.counters[e0:e1]), _p(self.reward[e0:e1]),
                                         _p(self.terminated[e0:e1]), _p(self.terms[e0:e1]), _p(self.target_find[e0:e1])))
        return self.reward, self.terminated

    def views(self, want_obs=True, want_state=True, envs=None):
        """(obs, state, avail) of every env, or of the envs listed in `envs` (in that order)."""
        s = self.spec
        n, M, S = s.n_agents, s.map_size, 2 * s.view_range - 1
        rows = np.arange(self.E) if envs is None else np.asarray(envs, np.int64).reshape(-1)
        pos = self.pos if envs is None else np.ascontiguousarray(self.pos[rows])
        tmap = self.tmap if envs is None else np.ascontiguousarray(self.tmap[rows])
        R = len(rows)
        obs = np.zeros((R, n, S * S + 2), np.float32) if want_obs else None
        state = np.zeros((R, 2 * M * M), np.float32) if want_state else None
        avail = np.zeros((R, n, 4), np.uint8)
        f = lib().os_views
        sl = lambda arr, e0, e1: None if arr is None else arr[e0:e1]
        _fanout(R, lambda e0, e1: f(C.byref(self.cs), e1 - e0, _p(pos[e0:e1]), _p(tmap[e0:e1]),
                                    _p(sl(obs, e0, e1)), _p(sl(state, e0, e1)), _p(avail[e0:e1])))
        return obs, state, avail

    def unfound_map(self):
        """[E, M, M] u8: target cells not found yet (the kernel's unfound bit rows)."""
        out = self.tmap.copy()
        e, k = np.nonzero(self.found)
        out[e, self.cells[e, k, 0], self.cells[e, k, 1]] = 0
        return out
