"""Batched discrete-grid search environment behind the reference's env protocol.

Mirrors ``SearchEnv`` (env/search_env.py): ``get_env_info, reset, step, get_obs, get_state,
get_avail_agent_actions, target_find, close`` with a leading ``num_envs`` axis.  The reference's ctor
opens a matplotlib figure (:49-53) and ``get_obs`` prints to stdout (:206,209); neither is reproduced.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import CoopSearchError
from .vec_flight import _wrap


class _Handle:
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            if self.ptr:
                _lib.load().cs_search_destroy(self.ptr)
                self.ptr = None
        except Exception:
            pass


class VecSearchEnv:
    """num_envs x SearchEnv (env/search_env.py)."""

    def __init__(self, args, circle_dict=None, targets_filename=None, num_envs=1, device=None, seed=0,
                 env_id_base=0, auto_reset=False, reset=True):
        if not torch.cuda.is_available():
            raise CoopSearchError("coopsearch_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.lib = _lib.load()
        self.args = args
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs = int(num_envs)
        self.map_size = int(args.map_size)
        self.target_num = int(args.target_num)
        self.target_mode = int(args.target_mode)
        self.agent_mode = int(args.agent_mode)
        self.n_agents = int(args.n_agents)
        self.view_range = int(args.view_range)
        self.obs_size = 2 * self.view_range - 1                       # search_env.py:27
        self.circle_dict = circle_dict
        self.targets_filename = targets_filename
        self.n_actions = 4
        self.seed = int(seed)
        self.env_id_base = int(env_id_base)
        if self.target_mode not in (0, 1, 2, 3):
            raise CoopSearchError('Unknown target mode')              # search_env.py:142-143
        if self.target_mode == 2 and not circle_dict:
            raise CoopSearchError('No circle dictionary')             # :124-125
        if self.target_mode == 3 and not targets_filename:
            raise CoopSearchError('No target file')                   # :139-140
        if self.target_mode in (2, 3) and auto_reset:
            # the layouts of modes 2 and 3 are placed from the host at reset(); an in-kernel auto-reset would redraw
            # uniform targets instead.  Step with auto_reset=False and call reset(mask=terminated).
            raise CoopSearchError('target_mode 2 / 3 need auto_reset=False (their target layouts are placed by reset())')
        cfg = _lib.SearchCfg(
            struct_size=C.sizeof(_lib.SearchCfg), num_envs=self.num_envs, n_agents=self.n_agents,
            target_num=self.target_num, map_size=self.map_size, view_range=self.view_range,
            agent_mode=self.agent_mode, target_mode=self.target_mode if self.target_mode in (0, 1) else 0,
            auto_reset=int(bool(auto_reset)), device=self.device.index, seed=self.seed & 0xFFFFFFFF,
            env_id_base=self.env_id_base & 0xFFFFFFFF)
        hp = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_create(C.byref(cfg), C.byref(hp)), "cs_search_create")
        self._h = _Handle(hp.value)
        b = _lib.SearchBuffers()
        _lib.check(self.lib.cs_search_buffers_get(self._h.ptr, C.byref(b)), "cs_search_buffers_get")
        E, n, M, W = self.num_envs, self.n_agents, self.map_size, b.words_per_row
        dev, own = self.device, self._h
        self.agent_pos = _wrap(b.pos, (E, n, 2), "<i4", dev, own)
        self.target_bits = _wrap(b.target_bits, (E, M, W), "<i4", dev, own)
        self.unfound_bits = _wrap(b.unfound_bits, (E, M, W), "<i4", dev, own)
        self.freq_map = _wrap(b.freq, (E, M, M), "<i4", dev, own)
        self.counters = _wrap(b.counters, (E, 4), "<i4", dev, own)
        self._obs = _wrap(b.obs, (E, n, self.obs_size ** 2 + 2), "<f4", dev, own)
        self._state = _wrap(b.state, (E, 2 * M * M), "<f4", dev, own)
        self._avail = _wrap(b.avail, (E, n, 4), "|u1", dev, own)
        self._reward = _wrap(b.reward, (E,), "<f4", dev, own)
        self._terminated = _wrap(b.terminated, (E,), "|u1", dev, own)
        self._target_find = _wrap(b.target_find, (E,), "<i4", dev, own)
        self._stats = _wrap(b.stats, (_lib.CS_NUM_STATS,), "<f8", dev, own)
        self._host = None
        self._fixed_cells = None
        self._reset_calls = 0
        if self.target_mode == 3:
            self._fixed_cells = self._cells_from_file(targets_filename)
        if reset:
            self.reset(init=True)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _cells_from_file(self, filename):
        """target_mode 3: one 'x y' pair per line (search_env.py:127-138); the same cells for every env."""
        cells = []
        with open(filename, "r") as fh:
            for line in fh:
                if line.strip():
                    x, y = [int(v) for v in line.split("\n")[0].split(" ")]
                    cells.append([x, y])
        if len(cells) != self.target_num:
            raise CoopSearchError("target file holds %d cells, target_num is %d" % (len(cells), self.target_num))
        self._check_cells(np.array(cells, np.int64)[None], "target file %s" % filename)
        return np.broadcast_to(np.array(cells, np.int32), (self.num_envs, self.target_num, 2)).copy()

    def _check_cells(self, cells, what):
        """Target cells [E,m,2] must lie on the map and be distinct within an env: the reference counts found targets per
        cell entry and would never reach target_num (search_env.py:263-271), while the bit rows hold one bit per cell."""
        M = self.map_size
        if cells.ndim != 3 or cells.shape[2] != 2:
            raise CoopSearchError("%s: cells must have shape (num_envs, target_num, 2)" % what)
        off = (cells < 0).any(-1) | (cells >= M).any(-1)
        if off.any():
            e, k = [int(v) for v in np.argwhere(off)[0]]
            raise CoopSearchError("%s: cell %s (env %d, target %d) lies off the %dx%d map"
                                  % (what, tuple(int(v) for v in cells[e, k]), e, k, M, M))
        key = np.sort(cells[..., 0] * M + cells[..., 1], axis=1)
        dup = key[:, 1:] == key[:, :-1]
        if dup.any():
            e, k = [int(v) for v in np.argwhere(dup)[0]]
            raise CoopSearchError("%s: env %d lists cell (%d, %d) more than once" % (what, e, key[e, k] // M, key[e, k] % M))

    def _cells_from_circles(self):
        """target_mode 2 (search_env.py:106-123): host-side sampling from the circle dictionary with a
        numpy Generator keyed by (seed, env id, reset count) -- a reset-time path, not part of the per-step hot path."""
        M, cd = self.map_size, self.circle_dict
        out = np.zeros((self.num_envs, self.target_num, 2), np.int32)
        for e in range(self.num_envs):
            rng = np.random.default_rng([self.seed, self.env_id_base + e, self._reset_calls])   # a fresh layout every reset (:106-123)
            taken, k = set(), 0
            for i, (cx, cy) in enumerate(cd['circle_center']):
                r = cd['circle_radius'][i]
                got = 0
                while got < cd['target_num'][i]:
                    x = int(rng.integers(max(cx - r, 0), min(cx + r, M)))
                    y = int(rng.integers(max(cy - r, 0), min(cy + r, M)))
                    if (x, y) not in taken:
                        taken.add((x, y)); out[e, k] = (x, y); k += 1; got += 1
        return out

    # ------------------------------------------------------------ reference API
    def get_env_info(self):
        """search_env.py:60-66 (+ n_envs)."""
        out = (C.c_int32 * 4)()
        _lib.check(self.lib.cs_search_env_info(self._h.ptr, out), "cs_search_env_info")
        return {"n_actions": out[0], "state_shape": out[1], "obs_shape": out[2], "episode_limit": out[3],
                "n_envs": self.num_envs}

    def reset(self, init=False, mask=None, cells=None):
        """reset (search_env.py:69-183).  `init` is accepted for signature parity; the freq map is never
        cleared either way (:39 vs :70-80).  cells: optional [E,m,2] int target cells to inject."""
        flags = 0
        if cells is not None:
            self._check_cells((cells.detach().cpu().numpy() if torch.is_tensor(cells) else np.asarray(cells)).astype(np.int64),
                              "reset(cells=...)")
        if cells is None and self.target_mode == 3:
            cells = self._fixed_cells
        if cells is None and self.target_mode == 2:
            cells = self._cells_from_circles()
            self._reset_calls += 1
        if cells is not None:
            c = torch.as_tensor(np.asarray(cells) if not torch.is_tensor(cells) else cells).to(
                device=self.device, dtype=torch.int32).contiguous()
            if tuple(c.shape) != (self.num_envs, self.target_num, 2):
                raise CoopSearchError("cells must have shape (num_envs, target_num, 2)")
            with torch.cuda.device(self.device):
                _lib.check(self.lib.cs_search_set_targets(self._h.ptr, C.c_void_p(c.data_ptr()), self._stream()),
                           "cs_search_set_targets")
            flags |= _lib.CS_RESET_KEEP_TARGETS
        mptr = None
        if mask is not None:
            mask = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            mptr = C.c_void_p(mask.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_reset(self._h.ptr, mptr, flags, self._stream()), "cs_search_reset")

    def step(self, actions):
        """step(act_list) (search_env.py:246-277) -> (reward [E] f32, terminated [E] u8, info '').
        An illegal move raises in the reference (:293); here it sets bit 1 of counters[:,2] for that env."""
        if torch.is_tensor(actions):
            a = actions.to(device=self.device, dtype=torch.uint8)
        else:
            a = torch.as_tensor(np.asarray(actions, dtype=np.uint8), device=self.device)
        if a.dim() == 1 and self.num_envs == 1:
            a = a.unsqueeze(0)
        if a.dim() != 2 or a.shape[0] != self.num_envs or a.shape[1] != self.n_agents:
            raise CoopSearchError('Act num mismatch agent')           # search_env.py:247-248
        a = a.contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_step(self._h.ptr, C.c_void_p(a.data_ptr()), self._stream()), "cs_search_step")
        return self._reward, self._terminated, ''

    def step_random(self, k=1):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_step_random(self._h.ptr, int(k), self._stream()), "cs_search_step_random")
        return self._reward, self._terminated, ''

    def get_obs(self):
        """[E,n,(2R-1)^2+2] (search_env.py:203-227)."""
        return self._obs

    def get_state(self):
        """[E,2*M*M], channels-last planes (search_env.py:186-200)."""
        return self._state

    def get_avail_agent_actions(self, agent_id):
        if agent_id >= self.n_agents:
            raise CoopSearchError('Agent id out of range')            # search_env.py:231-232
        return self._avail[:, agent_id]

    def get_avail_actions(self):
        return self._avail

    @property
    def target_find(self):
        return self._target_find

    @property
    def time_step(self):
        return self.counters[:, 1]

    @property
    def illegal(self):
        return (self.counters[:, 2] & 2) != 0

    def close(self):
        pass

    def render(self):
        raise CoopSearchError("render() is not part of the batched hot path")

    def stats(self):
        out = (C.c_double * _lib.CS_NUM_STATS)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_stats(self._h.ptr, out, self._stream()), "cs_search_stats")
        return dict(zip(_lib.STAT_NAMES, list(out)))

    @property
    def stats_tensor(self):
        return self._stats

    def host_buffers(self):
        if self._host is None:
            E, n, M = self.num_envs, self.n_agents, self.map_size
            pin = lambda *shape, dtype: torch.empty(shape, dtype=dtype).pin_memory()
            self._host = {
                "actions": pin(E, n, dtype=torch.uint8), "reward": pin(E, dtype=torch.float32),
                "terminated": pin(E, dtype=torch.uint8), "obs": pin(E, n, self.obs_size ** 2 + 2, dtype=torch.float32),
                "state": pin(E, 2 * M * M, dtype=torch.float32), "avail": pin(E, n, 4, dtype=torch.uint8),
            }
        return self._host

    def step_host(self, actions, want_obs=True, want_state=True):
        hb = self.host_buffers()
        a = np.asarray(actions, dtype=np.uint8)
        if a.shape != (self.num_envs, self.n_agents):
            raise CoopSearchError('Act num mismatch agent')
        hb["actions"].numpy()[...] = a
        io = _lib.SearchHostIO(
            actions=hb["actions"].data_ptr(), reward=hb["reward"].data_ptr(), terminated=hb["terminated"].data_ptr(),
            obs=hb["obs"].data_ptr() if want_obs else None, state=hb["state"].data_ptr() if want_state else None,
            avail=hb["avail"].data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_search_step_host(self._h.ptr, C.byref(io), self._stream()), "cs_search_step_host")
        return (hb["reward"].numpy(), hb["terminated"].numpy(), hb["obs"].numpy() if want_obs else None,
                hb["state"].numpy() if want_state else None, hb["avail"].numpy())
