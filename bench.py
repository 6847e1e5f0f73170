#!/usr/bin/env python
"""Benchmark of the env-step hot path (BASELINE.json metric: env-steps/s and agent-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5] [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] ("c2"): flight_easy 3a15t AM0TM0, 4096 envs per kernel launch.
4096 envs are ~2.6 MB of state+outputs, i.e. L2-resident, so the bench keeps 64 independent 4096-env batches
(~168 MB > the 126 MB L2) and steps them round-robin: one bench "step" is one env-step of every batch
(64 launches over 262144 env instances), and by the time a batch comes round again its lines have been evicted.
Under torchrun (N>1) every rank runs the same workload on its own GPU with its own global env ids (weak
scaling, no data-path collective); the only collective is the NCCL all-reduce of the 8-double episode-statistics
vector after the timed region.

The JSON line carries: value (device-resident inputs, CUDA-graph replay of the step launches), e2e (HOST
buffers through cs_flight_step_host: H2D actions + kernel + D2H reward/terminated/win/obs/state every step),
roofline of the step kernel against MEASURED_PEAKS.json, the CPU baseline (oracle port on the host cores) and
clocks sampled while the GPU was under this load.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

TEMPLATE = {  # flight_targets.txt of the reference (parsed as main.py:19-32 does); synthetic layout = the reference's own
    "x": [5, 2, 7.5, 2.8, 6.9, 5.5, 5.3, 1.8, 3, 4.5, 6.3, 8, 0.9, 9.4, 4.2],
    "y": [9.1, 7.5, 7, 8, 8.5, 8, 6.6, 6.8, 5.7, 5, 5.7, 6.7, 8.7, 9, 9.3],
    "deter": ["f", "t", "f", "f", "t", "f", "t", "t", "f", "f", "t", "f", "f", "t", "f"],
    "priority": [3, 3, 3, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1],
    "dx": [0.2, 0.3, 0.3, 0.27, 0.25, 0.25, 0.1, 0.28, 0.18, 0.23, 0.31, 0.29, 0.15, 0.21, 0.34],
    "dy": [0.2, 0.3, 0.26, 0.27, 0.25, 0.25, 0.12, 0.28, 0.18, 0.25, 0.30, 0.28, 0.16, 0.21, 0.33],
}

WORKLOADS = {
    # name: kind, n_agents, agent_mode, envs per launch, number of batches, description
    "c2": dict(kind="flight_easy", n=3, am=0, envs=4096, batches=64, grouped=True, lanes=1,
               desc="flight_easy 3a15t AM0TM0, 4096 batched envs per handle (BASELINE.json configs[1]); 64 independent handles "
                    "(rollout workers, 168 MB of state > L2) advance in ONE grouped launch (cs_flight_group_step)"),
    "c2s": dict(kind="flight_easy", n=3, am=0, envs=4096, batches=64,
                desc="flight_easy 3a15t AM0TM0, the same 64 handles x 4096 envs with one launch per handle (8 streams in a CUDA graph)"),
    "c3": dict(kind="flight_easy", n=5, am=2, envs=65536, batches=1, scaling="strong", total_envs=65536, policy="kernel",
               desc="flight_easy 5a15t AM2TM0, 65536 envs in total sharded over the N GPUs by global env id (BASELINE.json configs[2]); "
                    "uniform-random policy drawn in-kernel, keyed by the global env id"),
    "c4": dict(kind="flight", n=3, am=0, envs=16384, batches=1, map_overlap=True,
               desc="flight (probability map) 3a15t AM0TM0, 16384 envs per GPU (configs[3]); per env-step one step kernel and one "
                    "belief-map kernel, the map kernel on the handle's own stream (map_overlap: it runs concurrently with the next step kernel)"),
    "c2w": dict(kind="flight_easy", n=3, am=0, envs=1048576, batches=1,
                desc="flight_easy 3a15t AM0TM0, 1048576 envs in ONE launch (throughput asymptote of the c2 kernel)"),
    "c5": dict(kind="search", n=64, am=0, envs=131072, batches=1,
               desc="search_env 64 agents / 1000 targets / map 64, 131072 envs per GPU (BASELINE.json configs[4]: 1M envs across 8 GPUs, NCCL episode-stat all-reduce)"),
}


def flight_args(kind, n, am, m=15, M=50, R=7, T=200):
    return types.SimpleNamespace(env=kind, map_size=M, target_num=m, target_mode=0, agent_mode=am, n_agents=n, view_range=R,
                                 time_limit=T, detect_prob=0.9, safe_dist=1, agent_velocity=1, force_dist=3,
                                 turn_limit=np.pi / 4, wrong_alarm_prob=0.1)


def search_args(n=64, m=1000, M=64, R=7):
    return types.SimpleNamespace(env="search", map_size=M, target_num=m, target_mode=0, target_dir="./targets/", agent_mode=0,
                                 n_agents=n, view_range=R)


def algorithmic_bytes(kind, n, m=15, M=50, R=7, touched_per_step=0.0):
    """SURVEY.md section 8d contract figures (fp32 state, u8 actions), bytes per env-step."""
    if kind == "flight_easy":
        return 57 * n + 20 * m + 34
    if kind == "flight":
        return 57 * n + 20 * m + 34 + 8.0 * touched_per_step
    S = 2 * R - 1
    return 4 * n * (S * S + 2) + 8 * M * M + 16 * n + 8 * n + 3 * M * M // 8 + 8 * n


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.remove(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own env classes (unmodified copies staged under oracle/_ref by __graft_entry__.build()) on
# the host cores; the Python oracle port only where the staged reference is missing
# ----------------------------------------------------------------------------------------------------------------
def reference_kind():
    from oracle import refharness as rh
    if rh.reference_available():
        return "reference"
    print("bench.py: no reference checkout (COOPSEARCH_REFERENCE, BASELINE.json reference_path) and no staged oracle/_ref: "
          "the CPU baseline times the Python oracle port instead of the reference's own code", file=sys.stderr)
    return "port"


def _make_ref_env(kind, n, am):
    """An instance of the UNMODIFIED reference env class for this workload (oracle/_ref; SURVEY.md section 8d inputs)."""
    from oracle import refharness as rh
    ref = rh.import_reference()
    if kind in ("flight_easy", "flight"):
        args = rh.make_args(kind, n_agents=n, agent_mode=am)
        circle = rh.load_targets_reference_semantics(os.path.join(rh.REFERENCE_ROOT, "flight_targets.txt"))
        return rh.quiet(ref["FlightSearchEnvEasy" if kind == "flight_easy" else "FlightSearchEnv"], args, circle), args
    args = search_args() if n == 64 else search_args(n=n, m=15, M=50)
    return rh.quiet(ref["SearchEnv"], args), args


def _cpu_worker(job):
    """The loop common/rollout.py:43-63 runs on one env instance: reset, then per step get_obs, get_state, step under
    uniform-random (search: uniform-random legal) actions, for `seconds`.  impl "reference": the unmodified reference
    class; "port": oracle/py_envs.py."""
    import contextlib
    import io
    kind, n, am, seconds, wid, impl = job
    rng = np.random.default_rng(1000 + wid)
    np.random.seed(1000 + wid)
    if impl == "reference":
        env, _ = _make_ref_env(kind, n, am)
        reset = env.reset
    else:
        from oracle.py_envs import FlightOracle, FlightSpec, SearchOracle, SearchSpec
        if kind in ("flight_easy", "flight"):
            env = FlightOracle(FlightSpec(n_agents=n, agent_mode=am, variant="easy" if kind == "flight_easy" else "probmap"), TEMPLATE, 42, wid)
            reset = lambda: env.reset(init=False)
        else:
            env = SearchOracle(SearchSpec(n_agents=n, target_num=1000 if n == 64 else 15, map_size=64 if n == 64 else 50), 42, wid)
            reset = env.reset
    steps, limit = 0, (500 if kind == "search" else 10 ** 9)
    t0 = time.perf_counter()
    t_end = t0 + seconds
    with contextlib.redirect_stdout(io.StringIO()):              # the reference's search get_obs prints (search_env.py:206,209)
        while time.perf_counter() < t_end:
            reset()
            done, k = False, 0
            while not done and k < limit and time.perf_counter() < t_end:
                env.get_obs(); env.get_state()
                if kind == "search":
                    acts = [int(rng.choice(np.nonzero(env.get_avail_agent_actions(i))[0])) for i in range(n)]
                else:
                    acts = rng.integers(0, 3, size=n)
                _, done, _ = env.step(acts)
                steps += 1; k += 1
    return steps, time.perf_counter() - t0


def cpu_env_throughput(kind, n, am, seconds, procs, impl=None):
    """env-steps/s of `procs` independent single-threaded env loops (the reference is single-threaded; independent env
    instances are its embarrassingly-parallel upper bound, SURVEY.md section 8d).  Returns (env-steps/s, env-steps)."""
    import multiprocessing as mp
    impl = impl or reference_kind()
    jobs = [(kind, n, am, seconds, w, impl) for w in range(procs)]
    if procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with _pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    return sum(s / dt for s, dt in res), sum(s for s, _ in res)


class _pool:
    """One spawn-context process pool per bench run (start-up costs ~1 s per use otherwise)."""
    _shared = None

    def __init__(self, procs):
        import multiprocessing as mp
        if _pool._shared is None or _pool._shared[0] != procs:
            if _pool._shared is not None:
                _pool._shared[1].terminate()
            _pool._shared = (procs, mp.get_context("spawn").Pool(procs))
        self.pool = _pool._shared[1]

    def __enter__(self):
        return self.pool

    def __exit__(self, *exc):
        return False

    @staticmethod
    def close():
        if _pool._shared is not None:
            _pool._shared[1].terminate()
            _pool._shared = None


def rollout_worker_throughput(env_factory, n, seconds, seed=0):
    """BASELINE.json configs[0]: the reference's own RolloutWorker.generate_episode (common/rollout.py:22-141) with its
    Agents facade and alg=random (agent/agent.py:34-36), single process, driving `env_factory(args)`.  Returns
    (env-steps/s, episodes, env-steps, mean targets found per episode)."""
    import contextlib
    import io
    from oracle import refharness as rh
    rh.import_reference()
    with contextlib.redirect_stdout(io.StringIO()):
        from common.rollout import RolloutWorker
        from agent.agent import Agents
    args = rh.make_args("flight_easy", n_agents=n, agent_mode=0)
    env = env_factory(args)
    for k, v in env.get_env_info().items():
        if k != "n_envs":
            setattr(args, k, v)
    args.alg, args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = "random", 0, 0, 0, "step"
    args.last_action, args.reuse_network, args.cuda, args.evaluate_epoch = True, True, False, 20
    agents = rh.quiet(Agents, env, args)
    worker = rh.quiet(RolloutWorker, env, agents, args)
    np.random.seed(seed)
    rh.quiet(worker.generate_episode, 0)                         # warm-up episode
    steps = episodes = found = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        ep, _, _, tf = rh.quiet(worker.generate_episode, episodes + 1)
        steps += int((1 - ep["padded"][0]).sum())
        found += int(tf)
        episodes += 1
    dt = time.perf_counter() - t0
    return steps / dt, episodes, steps, found / max(1, episodes)


def c_port_throughput(kind, n, am, seconds, threads):
    """env-steps/s of the C oracle (oracle/coopsearch_oracle.c) incl. obs/state emission, `threads` host threads."""
    from oracle import c_oracle
    from oracle.py_envs import FlightSpec, SearchSpec
    c_oracle.set_threads(threads)
    E = 4096 * max(1, threads // 2)
    steps, t0 = 0, time.perf_counter()
    if kind in ("flight_easy", "flight"):
        spec = FlightSpec(n_agents=n, agent_mode=am, variant="easy" if kind == "flight_easy" else "probmap")
        if kind == "flight":
            E = 64 * threads
        b = c_oracle.FlightBatch(spec, TEMPLATE, 42, 0, E, auto_reset=True)
        b.reset(init=True)
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            b.step(None); b.obs_state()
            steps += E
    else:
        spec = SearchSpec(n_agents=n, target_num=1000 if n == 64 else 15, map_size=64 if n == 64 else 50)
        E = 16 * threads
        b = c_oracle.SearchBatch(spec, 42, 0, E)
        b.reset()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            b.step(None); b.views()
            steps += E
    dt = time.perf_counter() - t0
    c_oracle.set_threads(1)
    return steps / dt, steps


def cpu_baseline(kind, n, am, seconds_py, seconds_c):
    cores = os.cpu_count() or 1
    impl = reference_kind()
    v_all, steps_all = cpu_env_throughput(kind, n, am, seconds_py, cores, impl)
    v_one, _ = cpu_env_throughput(kind, n, am, min(seconds_py, 4.0), 1, impl)
    out = {
        "value": v_all, "unit": "env-steps/s", "cores": cores, "kind": impl,
        "sample": "%s: %d independent processes x %.0f s of reset/get_obs/get_state/step with uniform-random actions, %d env-steps in total"
                  % ("the UNMODIFIED reference env class (oracle/_ref, staged from the reference by __graft_entry__.build())" if impl == "reference"
                     else "Python oracle port (oracle/py_envs.py, the reference's scalar float64 loop)", cores, seconds_py, steps_all),
        "single_core": v_one, "cpu_model": _cpu_model(),
    }
    if impl == "reference":
        try:
            v_port, _ = cpu_env_throughput(kind, n, am, min(seconds_py, 4.0), 1, "port")
            out["port_single_core"] = v_port       # the oracle restatement beside the real thing
        except Exception as exc:
            out["port_single_core"] = repr(exc)
    try:
        v_c, _ = c_port_throughput(kind, n, am, seconds_c, cores)
        v_c1, _ = c_port_throughput(kind, n, am, min(seconds_c, 2.0), 1)
        out["c_port"] = {"value": v_c, "single_core": v_c1, "cores": cores,
                         "note": "plain-C oracle (oracle/coopsearch_oracle.c), same arithmetic, batched; not what the reference runs"}
    except Exception as exc:  # the C oracle needs gcc/make on the box
        print("C oracle unavailable: %s" % exc, file=sys.stderr)
    return out


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
def shard_envs(w, rank, world):
    """(first global env id, env count) of every batch of workload `w` on this rank.  Weak-scaled workloads give every
    GPU the same env count under its own global ids; strong-scaled ones (BASELINE.json configs[2]: 65536 envs over
    1/2/4/8 GPUs) split the global id range [0, total_envs) into contiguous blocks (dist.shard_range)."""
    if w.get("scaling") == "strong":
        total = w["total_envs"]
        base, rem = divmod(total, world)
        lo = rank * base + min(rank, rem)
        cnt = base + (1 if rank < rem else 0)
        return [(lo, cnt)]
    return [((rank * w["batches"] + b) * w["envs"], w["envs"]) for b in range(w["batches"])]


def make_envs(cs, w, device, rank, world=1, seed=42, count_touched=False):
    envs = []
    lpe = int(os.environ.get("CS_BENCH_LPE", str(w.get("lanes", 0))))      # 0 = the library's own choice
    for base, cnt in shard_envs(w, rank, world):
        if w["kind"] == "flight_easy":
            e = cs.VecFlightEasyEnv(flight_args("flight_easy", w["n"], w["am"]), TEMPLATE, num_envs=cnt, device=device,
                                    seed=seed, env_id_base=base, auto_reset=True, lanes_per_env=lpe)
        elif w["kind"] == "flight":
            e = cs.VecFlightEnv(flight_args("flight", w["n"], w["am"]), TEMPLATE, num_envs=cnt, device=device, seed=seed,
                                env_id_base=base, auto_reset=True, count_touched=count_touched, lanes_per_env=lpe,
                                map_overlap=bool(w.get("map_overlap")) and os.environ.get("CS_BENCH_MAP_OVERLAP", "1") != "0")
        else:
            e = cs.VecSearchEnv(search_args(), num_envs=cnt, device=device, seed=seed, env_id_base=base, auto_reset=True)
        envs.append(e)
    return envs


def silence(fn, *a, **k):
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


MIN_TIMED_MS = 60.0       # the host-buffer (e2e) blocks are repeated until they last at least this long
DUMP_BYTES = 60 << 20     # --dump-outputs data: with the .npy headers under 64 MB (64e6 bytes) in all
SPREAD_REPLAYS = 5        # untimed replays after the timed one whose min / max show how much one replay varies


def dump_outputs(torch, envs, kind, directory):
    """Writes what the last step left in the env buffers -- reward, terminated, win (flight), target_find, get_obs(),
    get_state() and, for search, the action masks -- as <directory>/<name>.npy in float32, one row per env in global env
    id order.  When all rows would exceed DUMP_BYTES, every array keeps the same fixed, seeded sample of env rows."""
    cat = lambda get: torch.cat([get(e).float() for e in envs])
    arrays = {"reward": cat(lambda e: e._reward), "terminated": cat(lambda e: e._terminated)}
    if kind != "search":
        arrays["win"] = cat(lambda e: e.win_flag)
    arrays.update(target_find=cat(lambda e: e.target_find), obs=cat(lambda e: e.get_obs()), state=cat(lambda e: e.get_state()))
    if kind == "search":
        arrays["avail"] = cat(lambda e: e.get_avail_actions())
    rows = arrays["reward"].shape[0]
    row_bytes = sum(4 * a[0].numel() for a in arrays.values())
    if rows * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(rows, DUMP_BYTES // row_bytes, replace=False))
        idx = torch.from_numpy(keep).to(arrays["reward"].device)
        arrays = {k: a.index_select(0, idx) for k, a in arrays.items()}
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a.cpu().numpy())


def run_gpu_workload(cs, torch, name, steps, warmup, device, rank, world, want_e2e=True, burn_in_steps=6000, dump_dir=None):
    """One workload on this rank.  The `steps` bench steps are captured into ONE CUDA graph; the timed region is one
    replay of it, bracketed by CUDA events on the launching stream.  Before it, untimed: `warmup` steps, then
    `burn_in_steps` rounded up to whole replays, queued back to back so that clocks have ramped under this load and
    the timed replay starts while the GPU is still busy (no launch gap in the region).  Every count is fixed, so the
    same arguments step the envs through the same sequence; `dump_dir` receives what the last timed step computed."""
    w = WORKLOADS[name]
    n = w["n"]
    A = 4 if w["kind"] == "search" else 3
    envs = silence(make_envs, cs, w, device, rank, world)
    POOL = 8
    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    if w["kind"] == "search" or w.get("policy") == "kernel":
        actions = None          # the uniform-random (search: legal) policy is drawn in-kernel, keyed by the global env id
    else:
        actions = [[torch.randint(0, A, (e.num_envs, n), generator=gen, device=device, dtype=torch.uint8) for e in envs]
                   for _ in range(POOL)]

    side = torch.cuda.Stream(device=device)
    nstreams = max(1, min(int(os.environ.get("CS_BENCH_STREAMS", "8")), len(envs)))
    forks = [torch.cuda.Stream(device=device) for _ in range(nstreams)] if nstreams > 1 else []
    grouped = None
    if w.get("grouped") and len(envs) > 1 and os.environ.get("CS_BENCH_GROUPED", "1") != "0":
        grouped = cs.DeviceStepper(envs)          # all batches advance in ONE launch (cs_flight_group_step)
        nstreams, forks = 1, []

    def one_step(k):
        """One env-step of every batch.  The batches are independent env sets (rollout workers): either one grouped
        launch steps them all, or their launches are forked over `nstreams` streams (captured as parallel branches of
        the CUDA graph) and joined again."""
        if grouped is not None:
            with torch.cuda.stream(side):
                grouped.step(actions[k % POOL])
            return
        if forks:
            for f in forks:
                f.wait_stream(side)
        for b, e in enumerate(envs):
            with torch.cuda.stream(forks[b % nstreams] if forks else side):
                if actions is None:
                    e.step_random(1)
                else:
                    e.step(actions[k % POOL][b])
        for f in forks:
            side.wait_stream(f)

    def join_maps():
        """map_overlap handles run their belief-map kernels on their own stream: joined before a capture begins / ends"""
        for e in envs:
            if getattr(e, "map_overlap", False):
                with torch.cuda.stream(side):
                    e.sync_map()

    torch.cuda.synchronize(device)
    lib = cs.load_library()
    with torch.cuda.stream(side):
        k0 = lib.cs_launch_count()
        one_step(0)
        kernels_per_step = int(lib.cs_launch_count() - k0)     # kernels of OUR library one step launches (graph replays repeat them)
        join_maps()
        torch.cuda.synchronize(device)
        gsteps = torch.cuda.CUDAGraph()                        # exactly `steps` bench steps
        with torch.cuda.graph(gsteps, stream=side):
            for k in range(steps):
                one_step(k)
            join_maps()
        for k in range(warmup):
            one_step(k)
        join_maps()
    torch.cuda.synchronize(device)
    if world > 1:
        torch.distributed.barrier()
    burn_in_replays = -(-burn_in_steps // steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(side):
        for _ in range(burn_in_replays):
            gsteps.replay()
        e0.record()
        gsteps.replay()                                        # the timed region: exactly `steps` steps
        e1.record()
    torch.cuda.synchronize(device)
    if world > 1:
        torch.distributed.barrier()
    ms = e0.elapsed_time(e1)
    if dump_dir is not None:
        dump_outputs(torch, envs, w["kind"], dump_dir)
    # noise check, not part of the timed figure: SPREAD_REPLAYS more replays of the same graph, each bracketed by events
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(SPREAD_REPLAYS + 1)]
    with torch.cuda.stream(side):
        evs[0].record()
        for r in range(SPREAD_REPLAYS):
            gsteps.replay()
            evs[r + 1].record()
    torch.cuda.synchronize(device)
    spread = [evs[r].elapsed_time(evs[r + 1]) for r in range(SPREAD_REPLAYS)]
    launches = steps * (1 if grouped is not None else len(envs))
    env_count = sum(e.num_envs for e in envs)
    out = dict(grouped=grouped is not None, ms_total=ms, ms_per_step=ms / steps, env_steps_per_step=env_count, launches=launches, streams=nstreams,
               kernels=kernels_per_step * steps, burn_in_steps=burn_in_replays * steps, check_replays_ms=[min(spread), max(spread)],
               us_per_launch=1000.0 * ms / launches, lanes_per_env=getattr(envs[0], "lanes_per_env", None),
               envs_per_launch=env_count if grouped is not None else envs[0].num_envs)

    # ---- end to end through the host-buffer C-ABI call -----------------------------------------------------
    if want_e2e:
        e2e_steps = max(3, min(steps, 50))
        rng = np.random.default_rng(7)
        streams = [torch.cuda.Stream(device=device) for _ in range(min(4, len(envs)))]

        def time_blocks(host_step):
            for k in range(3):
                host_step(k)
            torch.cuda.synchronize(device)
            blocks = []
            if world > 1:
                torch.distributed.barrier()
            t_region = time.perf_counter()
            while True:                                   # repeat the e2e_steps block until >= MIN_TIMED_MS, median block
                t0 = time.perf_counter()
                for k in range(e2e_steps):
                    host_step(k)
                torch.cuda.synchronize(device)
                blocks.append(time.perf_counter() - t0)
                if ((time.perf_counter() - t_region) * 1000.0 >= MIN_TIMED_MS and len(blocks) >= 3) or len(blocks) >= 200:
                    break
            return sorted(blocks)[len(blocks) // 2] / e2e_steps, len(blocks)

        if w["kind"] == "search":
            for e in envs:
                e.host_buffers()["avail"].copy_(e.get_avail_actions().cpu())

            def host_step(k):
                for b, e in enumerate(envs):
                    av = e.host_buffers()["avail"].numpy()
                    # first legal move of every agent, computed on the host from the previous step's D2H avail mask
                    e.step_host(av.argmax(axis=2).astype(np.uint8))
            dt, nblocks = time_blocks(host_step)
            hb = envs[0].host_buffers()
            out.update(e2e_s_per_step=dt, e2e_steps=e2e_steps, e2e_blocks=nblocks, e2e_form="cs_search_step_host per batch",
                       h2d_bytes_per_step=sum(e.host_buffers()["actions"].numel() for e in envs),
                       d2h_bytes_per_step=sum(sum(v.numel() * v.element_size() for kname, v in e.host_buffers().items() if kname != "actions") for e in envs))
        else:
            # this step's actions are in PINNED host memory (two alternating sets); one library call steps every batch and
            # returns when every batch's results are in host memory.  Two forms of the same call are timed, the faster
            # one is the e2e figure: "compact" (pooled buffers: 16 + 16n bytes per env over PCIe -- the 16-byte records in
            # one flat copy, the agent rows written in place into the reference-shaped host rows by one strided copy; host
            # threads update result arrays and find flags) and "slab" (the whole output slab of every batch, batches
            # pipelined over a few streams).
            host_actions = [[rng.integers(0, A, size=(e.num_envs, n), dtype=np.uint8) for e in envs] for _ in range(2)]
            pinned = [[torch.from_numpy(a).pin_memory() for a in host_actions[k]] for k in range(2)]
            pooled_actions = [torch.from_numpy(np.concatenate(host_actions[k], axis=0)).pin_memory() for k in range(2)]
            use_graph = os.environ.get("CS_BENCH_E2E_GRAPH", "1") != "0"
            forms = {}
            # slab first: the compact form's pooled buffers stay attached to the envs afterwards
            for form in ("slab", "compact"):
                if form == "compact":
                    stepper = cs.HostStepper(envs, streams, graph=False, compact=True)      # six enqueues per step: no graph needed
                    if stepper._pool is None:
                        raise RuntimeError("the env batches of workload %s did not pool" % name)
                    dt, nblocks = time_blocks(lambda k: stepper.step(actions=pooled_actions[k % 2]))
                else:
                    steppers = [cs.HostStepper(envs, streams, actions=pinned[k], graph=use_graph, compact=False) for k in range(2)]
                    dt, nblocks = time_blocks(lambda k: steppers[k % 2].step())
                forms[form] = dict(s_per_step=dt, blocks=nblocks, d2h=sum(int(e.host_buffers(form == "compact")["d2h_bytes"]) for e in envs))
            best = min(forms, key=lambda f: forms[f]["s_per_step"])
            out.update(e2e_s_per_step=forms[best]["s_per_step"], e2e_steps=e2e_steps, e2e_blocks=forms[best]["blocks"], e2e_form=best,
                       e2e_forms={f: {"env_steps_per_s": env_count / v["s_per_step"], "d2h_bytes_per_step": v["d2h"]} for f, v in forms.items()},
                       h2d_bytes_per_step=sum(e.host_buffers()["actions"].numel() for e in envs), d2h_bytes_per_step=forms[best]["d2h"])
    # statistics of the finished episodes on this GPU (all-reduced by the caller)
    stats = torch.zeros(8, dtype=torch.float64, device=device)
    for e in envs:
        stats += torch.tensor(list(e.stats().values()), dtype=torch.float64, device=device)
    out["stats"] = stats
    return out


def shard_invariance_stats(cs, torch, dist, name, device, rank, world, steps=400):
    """Hardware proof that sharding does not change results: a FRESH set of handles for this rank's shard of a
    strong-scaled workload runs exactly `steps` steps under the in-kernel random policy (keyed by the global env id);
    the NCCL all-reduced episode statistics must be identical for every world size."""
    w = dict(WORKLOADS[name])
    envs = silence(make_envs, cs, w, device, rank, world)
    for e in envs:
        e.step_random(steps)
    stats = torch.zeros(8, dtype=torch.float64, device=device)
    for e in envs:
        stats += torch.tensor(list(e.stats().values()), dtype=torch.float64, device=device)
    stats = dist.allreduce_stats(stats)
    return dict(zip(cs._lib.STAT_NAMES, [float(x) for x in stats.tolist()]))


def measure_obs_full(cs, torch, device, peak):
    """Reference-shaped flight observation (flight_env.py:223-230): 4*M*M read + 4n(M*M+4) written per env."""
    w = dict(WORKLOADS["c4"])
    env = silence(make_envs, cs, w, device, 0)[0]
    env.step_random(3)
    out = {}
    for kind in ("tma", "plain"):
        env.set_obs_kernel(kind)
        for _ in range(5):
            env.get_obs()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            env.get_obs()
        e1.record()
        torch.cuda.synchronize(device)
        us = 1000.0 * e0.elapsed_time(e1) / 20
        M2 = env.map_size ** 2
        nbytes = env.num_envs * (4 * M2 + 4 * env.n_agents * (M2 + 4))
        out[kind] = {"us_per_launch": us, "achieved": nbytes / (us * 1e-6) / 1e9, "frac": nbytes / (us * 1e-6) / 1e9 / peak,
                     "bytes_per_env": nbytes // env.num_envs}
    return out


def measure_spread(cs, torch, device, peak, E=1048576, n=3, m=3, K=20):
    """simple_spread (env/simple_spread.py; SURVEY 8f rank 4): env-steps/s of the batched step on E envs, K steps per CUDA
    graph replayed until >= 60 ms, auto-reset, pre-generated device actions; and the unmodified reference class on one core."""
    import types
    args = types.SimpleNamespace(env="simple_spread", n_agents=n, target_num=m, map_size=50)
    env = silence(cs.VecSimpleSpreadEnv, args, num_envs=E, device=device, seed=42, auto_reset=True)
    gen = torch.Generator(device=device).manual_seed(3)
    acts = [torch.randint(0, 5, (E, n), generator=gen, device=device, dtype=torch.uint8) for _ in range(4)]
    side = torch.cuda.Stream(device=device)
    with torch.cuda.stream(side):
        for k in range(5):
            env.step(acts[k % 4])
        torch.cuda.synchronize(device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for k in range(K):
                env.step(acts[k % 4])
        torch.cuda.synchronize(device)
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize(device)
        times, t_region = [], time.perf_counter()
        while True:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record()
            torch.cuda.synchronize(device)
            times.append(e0.elapsed_time(e1))
            if (time.perf_counter() - t_region) * 1000.0 >= MIN_TIMED_MS and len(times) >= 3:
                break
    us = 1000.0 * sorted(times)[len(times) // 2] / K
    obs_dim = 2 + 2 * (n - 1) + 4 * m
    # read: coordinates 16(n+m), meta 16, episode reward 8, actions n; write: agent coordinates 16n, obs 4*n*obs_dim,
    # state 8(n+m), occupied m, reward 4+8, terminated 1, meta 16, episode reward 8
    per_env = (16 * (n + m) + 24 + n) + (16 * n + 4 * n * obs_dim + 8 * (n + m) + m + 13 + 24)
    out = {"workload": "simple_spread %da%dt map 50, %d envs in one launch, auto-reset" % (n, m, E), "kernel": "spread_kernel<STEP> (one warp per env)",
           "value": E / (us * 1e-6), "unit": "env-steps/s", "agent_steps_per_s": n * E / (us * 1e-6), "us_per_launch": us,
           "roofline": {"bound": "hbm", "achieved": per_env * E / (us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": per_env * E / (us * 1e-6) / 1e9 / peak, "algorithmic_bytes_per_env_step": per_env, "traffic": load_traffic("spread")}}
    try:                                                   # the unmodified reference class, one core, bounded sample
        from oracle import refharness as rh
        ref = rh.import_reference()["SimpleSpreadEnv"]
        renv = rh.quiet(ref, args)
        renv.reset()
        rng = np.random.default_rng(1)
        t0, steps = time.perf_counter(), 0
        while time.perf_counter() - t0 < 2.0:
            for _ in range(100):
                renv.step([int(a) for a in rng.integers(0, 5, size=n)]); renv.get_obs(); renv.get_state()
            steps += 100
            if steps % 1000 == 0:
                renv.reset()
        out["reference_one_core"] = {"value": steps / (time.perf_counter() - t0), "unit": "env-steps/s",
                                     "sample": "2 s of step/get_obs/get_state on the unmodified reference class (oracle/_ref)"}
    except Exception as exc:                               # the staged reference is absent: no CPU figure
        out["reference_one_core"] = {"error": repr(exc)}
    return out


def measure_policy(cs, torch, device, n=3, iters=30):
    """Batched agent network + action choice (csrc/policy.cu, policy_tc.cuh; SURVEY 8f rank 1) on random-init weights of the
    reference's architecture (in 10 -> 64 -> GRU 64 -> 64 -> 3): rows/s of one choose_actions launch for the tensor-core
    kernel and the fp32 kernel at 4096 envs and at the c2 workload's 262144 envs (786432 rows), and the closed device loop
    get_obs -> choose_actions -> step (one CUDA graph per step) on 262144 flight_easy envs."""
    torch.manual_seed(0)
    in_dim = 4 + 3 + n
    sd = {"fc1.weight": torch.randn(64, in_dim) * 0.1, "fc1.bias": torch.zeros(64), "rnn.weight_ih": torch.randn(192, 64) * 0.1,
          "rnn.weight_hh": torch.randn(192, 64) * 0.1, "rnn.bias_ih": torch.zeros(192), "rnn.bias_hh": torch.zeros(192),
          "fc2.0.weight": torch.randn(64, 64) * 0.1, "fc2.0.bias": torch.zeros(64), "fc2.2.weight": torch.randn(3, 64) * 0.1,
          "fc2.2.bias": torch.zeros(3)}
    flop = 2 * (in_dim * 64 + 2 * 64 * 192 + 64 * 64 + 64 * 3)
    out = {"workload": "agent network + greedy action choice, random-init weights, synthetic obs", "flop_per_row": flop, "runs": []}
    for E in (4096, 262144):
        for precision in ("bf16", "fp32"):
            agents = cs.BatchedRNNAgents(sd, num_envs=E, n_agents=n, device=device, precision=precision)
            obs = torch.rand(E, n, 4, device=device) * 2 - 1
            for _ in range(5):
                agents.choose_actions(obs)
            torch.cuda.synchronize(device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                agents.choose_actions(obs)
            e1.record()
            torch.cuda.synchronize(device)
            us = 1000.0 * e0.elapsed_time(e1) / iters
            rows = E * n
            # per row: obs 16 B + last action 1 B read, hidden 256 B read + 256 B written, q 12 B + action 1 B written
            out["runs"].append({"kernel": agents.kernel_name, "rows": rows, "us_per_launch": us, "agent_steps_per_s": rows / (us * 1e-6),
                                "tflops": rows * flop / (us * 1e-6) / 1e12, "hbm_gbs": rows * 542 / (us * 1e-6) / 1e9})
            del agents
    # closed loop on the device
    E = 262144
    env = silence(cs.VecFlightEasyEnv, flight_args("flight_easy", n, 0), TEMPLATE, num_envs=E, device=device, seed=3, auto_reset=True)
    agents = cs.BatchedRNNAgents(sd, num_envs=E, n_agents=n, device=device)
    side = torch.cuda.Stream(device=device)
    with torch.cuda.stream(side):
        for _ in range(3):
            env.step(agents.choose_actions(env.get_obs()))
        torch.cuda.synchronize(device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(10):
                env.step(agents.choose_actions(env.get_obs()))
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            g.replay()
        e1.record()
        torch.cuda.synchronize(device)
    us = 1000.0 * e0.elapsed_time(e1) / 200
    out["device_loop"] = {"what": "get_obs -> choose_actions (tensor cores) -> step, 262144 flight_easy 3a15t envs, 10 steps per CUDA graph",
                          "us_per_step": us, "env_steps_per_s": E / (us * 1e-6), "agent_steps_per_s": E * n / (us * 1e-6)}
    return out


def measure_touched(cs, torch, device, steps=200):
    """Exact mean number of probability-map cells updated per env-step on the c4 workload (separate, untimed pass)."""
    w = dict(WORKLOADS["c4"]); w["envs"] = 2048
    envs = silence(make_envs, cs, w, device, 0, count_touched=True)
    e = envs[0]
    base = e.stats()["map_cells_touched"]
    e.step_random(steps)
    torch.cuda.synchronize(device)
    return (e.stats()["map_cells_touched"] - base) / (steps * w["envs"])


def measure_c1(cs, torch, device, seconds=4.0):
    """BASELINE.json configs[0] (flight_easy 1a15t AM0TM0, single env, random policy via common/rollout.py): the
    reference's own RolloutWorker + Agents(alg=random) driving (i) the reference env on one host core and (ii) our
    E=1 SingleEnvAdapter (one kernel launch per call: the latency floor of the drop-in, not a throughput figure)."""
    from oracle import refharness as rh
    if not rh.reference_available():
        return {"unavailable": "no reference checkout (COOPSEARCH_REFERENCE, BASELINE.json reference_path) and no staged oracle/_ref"}
    ref = rh.import_reference()
    circle = rh.load_targets_reference_semantics(os.path.join(rh.REFERENCE_ROOT, "flight_targets.txt"))
    v_ref, eps, steps, found = rollout_worker_throughput(lambda a: rh.quiet(ref["FlightSearchEnvEasy"], a, circle), 1, seconds)
    out = {"workload": "flight_easy 1a15t AM0TM0, single env, reference RolloutWorker.generate_episode + alg=random (common/rollout.py:22-141)",
           "reference_env": {"value": v_ref, "unit": "env-steps/s", "episodes": eps, "env_steps": steps, "mean_targets_found": found, "cores": 1}}
    mk = lambda a: cs.SingleEnvAdapter(silence(cs.VecFlightEasyEnv, a, circle, num_envs=1, device=device, seed=7))
    v_ad, eps, steps, found = rollout_worker_throughput(mk, 1, seconds)
    out["adapter_e1"] = {"value": v_ad, "unit": "env-steps/s", "episodes": eps, "env_steps": steps, "mean_targets_found": found,
                         "note": "unmodified reference RolloutWorker on SingleEnvAdapter(VecFlightEasyEnv, num_envs=1): every protocol call is a device round trip"}
    return out


def kernel_name(w, lanes, grouped=False):
    """The dominant kernel of a workload (csrc/flight_*.cu, csrc/search.cu)."""
    if w["kind"] == "search":
        return "search_kernel<STEP>"
    if grouped:
        return "flight_tpe_group_kernel<N=%d,K=%d>" % (w["n"], lanes)
    if w["kind"] == "flight":
        if lanes == 8:
            return "flight_fused_kernel<N=%d,STEP> (step + belief map of an env in one launch, 8 lanes per env)" % w["n"]
        if lanes in (1, 4):
            return "flight_map_tile_kernel (after flight_tpe_kernel<N=%d,K=%d,STEP,MAP>; two launches per env-step)" % (w["n"], lanes)
        return "flight_kernel<LPE=%s,STEP> + flight_map_generic_kernel" % lanes
    return ("flight_tpe_kernel<N=%d,K=%d,STEP>" % (w["n"], lanes)) if lanes and lanes <= 4 else "flight_kernel<LPE=%s,STEP>" % lanes


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(key):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(key)
    return None


def config_for(name, world):
    """The `config` object of the JSON line: a pure function of the workload and the world size, so that both arms
    (`--impl ours`, `--impl reference`) print the same one."""
    w = WORKLOADS[name]
    grouped = bool(w.get("grouped")) and os.environ.get("CS_BENCH_GROUPED", "1") != "0"
    if w.get("scaling") == "strong":
        per_gpu, handles = w["total_envs"] // world, 1
    else:
        per_gpu, handles = w["envs"] * w["batches"], w["batches"]
    return {
        "workload": w["desc"], "envs_per_handle": per_gpu // handles, "handles_per_gpu": handles,
        "envs_per_launch": per_gpu if (grouped or handles == 1) else per_gpu // handles, "launches_per_step": 1 if grouped else handles,
        "env_instances_per_gpu": per_gpu, "auto_reset": True,
        "actions": "uniform-random policy: pre-generated u8 tensors resident in HBM (flight) / drawn in-kernel with Philox (search, shard-invariance runs)",
        "launch": "the --steps bench steps are captured into one CUDA graph; one step = " +
                  ("ONE grouped launch that steps every handle (cs_flight_group_step)" if grouped else "one launch per handle"),
        "timing": "the timed region is one replay of the K-step graph, bracketed by CUDA events on the launching stream and queued behind the untimed "
                  "burn-in replays; its duration / K is ms_per_step (max over ranks); synchronize + barrier before the burn-in and after the region; "
                  "%d more replays after it, untimed for the result, give timed.check_replays_ms_min_max (raise --steps where they spread)" % SPREAD_REPLAYS,
        "l2": "working set of all batches exceeds the 126 MB L2; batches are revisited round-robin, no flush",
        "parallelism": "dp%d (env instances sharded by global id, no data-path collective)" % world,
    }


def reference_arm(args, w, rank):
    """`--impl reference`: the reference's own CPU implementation of the path -- the UNMODIFIED env classes staged under
    oracle/_ref (the Python oracle port where that is missing) -- on every host core.  One bench step = a bounded sample:
    every core runs the reset / get_obs / get_state / step loop on its own env instance for a fixed slice of time."""
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    impl = reference_kind()
    total = args.steps + args.warmup
    per_step_seconds = max(0.05, min(8.0, 110.0 / max(1, total)))
    for _ in range(args.warmup):
        cpu_env_throughput(w["kind"], w["n"], w["am"], per_step_seconds, cores, impl)
    vals, total_steps = [], 0
    for _ in range(args.steps):
        v, s_ = cpu_env_throughput(w["kind"], w["n"], w["am"], per_step_seconds, cores, impl)
        vals.append(v); total_steps += s_
    _pool.close()
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "env-steps/s", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * per_step_seconds, "higher_is_better": True,
        "scaling": WORKLOADS[args.workload].get("scaling", "weak"), "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(args.workload, int(os.environ.get("WORLD_SIZE", "1"))),
        "agent_steps_per_s": v * w["n"],
        "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": impl,
                         "sample": "%d env-steps of reset/get_obs/get_state/step under uniform-random actions: %d steps x %.2f s on %d processes, each with its own instance of %s"
                                   % (total_steps, args.steps, per_step_seconds, cores,
                                      "the unmodified reference env class (oracle/_ref)" if impl == "reference" else "the Python oracle port (oracle/py_envs.py)"),
                         "cpu_model": _cpu_model()},
        "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def extra_entry(cs, torch, name, r, peak, device, with_touched=True):
    ww = WORKLOADS[name]
    tch = measure_touched(cs, torch, device) if (ww["kind"] == "flight" and with_touched) else None
    pu = algorithmic_bytes(ww["kind"], ww["n"], touched_per_step=tch or 0.0) if ww["kind"] != "search" else \
        algorithmic_bytes("search", 64, m=1000, M=64, R=7)
    v = r["env_steps_per_step"] / (r["ms_per_step"] / 1000.0)
    gbs = pu * r["envs_per_launch"] / (1e-6 * r["us_per_launch"]) / 1e9
    out = {"workload": ww["desc"], "kernel": kernel_name(ww, r["lanes_per_env"], r["grouped"]), "value": v, "unit": "env-steps/s",
           "agent_steps_per_s": v * ww["n"], "us_per_launch": r["us_per_launch"], "timed_region_ms": r["ms_total"],
           "check_replays_ms_min_max": r["check_replays_ms"],
           "roofline": {"achieved": gbs, "peak": peak, "frac": gbs / peak, "unit": "GB/s", "algorithmic_bytes_per_env_step": pu,
                        "env_steps_per_launch": r["envs_per_launch"], "map_cells_touched_per_env_step": tch, "traffic": load_traffic(name)}}
    if "e2e_s_per_step" in r:
        out["e2e_value"] = r["env_steps_per_step"] / r["e2e_s_per_step"]
        out["e2e_form"] = r.get("e2e_form")
        out["e2e_forms"] = r.get("e2e_forms")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the supplementary workloads / CPU baseline")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy "
                                                         "(rank 0's envs; float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return reference_arm(args, w, rank)

    import torch
    import coopsearch_b200 as cs
    from coopsearch_b200 import dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: the product has no CPU path")
    rank, local, world = dist.init_from_env("nccl" if world > 1 else None, bind_cpus=True)
    device = torch.device("cuda", local if world > 1 else 0)
    torch.cuda.set_device(device)
    lib = cs.load_library()
    launches0 = lib.cs_launch_count()

    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    res = run_gpu_workload(cs, torch, args.workload, args.steps, args.warmup, device, rank, world,
                           dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None

    ms_max = dist.max_over_ranks(res["ms_total"], device=device)
    e2e_max = dist.max_over_ranks(res["e2e_s_per_step"], device=device)
    t0 = time.perf_counter()
    stats = dist.allreduce_stats(res["stats"])          # NCCL all-reduce of the episode statistics
    torch.cuda.synchronize(device)
    allreduce_us = 1e6 * (time.perf_counter() - t0)

    # supplementary workloads that run on EVERY rank (max over ranks, like the headline): configs[2] strong-scaled over
    # the N GPUs with the cross-N shard-invariance statistics, configs[4] at its stated 131072 envs per GPU
    extra = {}
    peak, peak_src = load_peaks()
    if not args.no_extra:
        for name in ("c3", "c5"):
            if name == args.workload:
                continue
            try:
                k = min(args.steps, 60 if name != "c5" else 20)
                # (no host-buffer leg for c5 at its full size: 131072 envs x 80 KB of observations / state planes per step)
                r = run_gpu_workload(cs, torch, name, k, 5, device, rank, world, want_e2e=(world == 1 and name != "c5"), burn_in_steps=2000)
                r["ms_per_step"] = dist.max_over_ranks(r["ms_per_step"], device=device)
                r["us_per_launch"] = dist.max_over_ranks(r["us_per_launch"], device=device)
                st = dist.allreduce_stats(r["stats"])
                r["env_steps_per_step"] = r["env_steps_per_step"] * world if WORKLOADS[name].get("scaling") != "strong" else WORKLOADS[name]["total_envs"]
                ent = extra_entry(cs, torch, name, r, peak, device)
                ent["n_gpus"] = world
                ent["scaling"] = WORKLOADS[name].get("scaling", "weak")
                ent["episode_stats_allreduced"] = dict(zip(cs._lib.STAT_NAMES, [float(x) for x in st.tolist()]))
                if WORKLOADS[name].get("scaling") == "strong":
                    ent["shard_invariance"] = {
                        "what": "fresh handles, exactly 400 steps of the in-kernel random policy over the SAME 65536 global env ids, NCCL all-reduced statistics: identical for every N",
                        "stats": shard_invariance_stats(cs, torch, dist, name, device, rank, world)}
                extra[name] = ent
            except Exception as exc:  # supplementary only: never lose the headline line
                extra[name] = {"error": repr(exc)}
    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
        return 0

    env_steps = res["env_steps_per_step"] * world * args.steps
    value = env_steps / (ms_max / 1000.0)
    e2e_value = res["env_steps_per_step"] * world / e2e_max
    touched = None
    if w["kind"] == "flight":
        touched = measure_touched(cs, torch, device)
    per_unit = algorithmic_bytes(w["kind"], w["n"], touched_per_step=touched or 0.0) if w["kind"] != "search" else \
        algorithmic_bytes("search", 64, m=1000, M=64, R=7)
    bytes_per_launch = per_unit * res["envs_per_launch"]
    sec_per_launch = (res["ms_total"] / 1000.0) / res["launches"]
    achieved = bytes_per_launch / sec_per_launch / 1e9
    cfg = config_for(args.workload, world)
    line = {
        "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": w.get("scaling", "weak"), "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "timed": {"steps": args.steps, "region_ms": res["ms_total"], "burn_in_steps": res["burn_in_steps"],
                  "check_replays_ms_min_max": res["check_replays_ms"], "lanes_per_env": res["lanes_per_env"], "streams": res["streams"]},
        "agent_steps_per_s": value * w["n"],
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": res["h2d_bytes_per_step"],
                "d2h_bytes_per_step": res["d2h_bytes_per_step"], "agent_steps_per_s": e2e_value * w["n"],
                "steps": res["e2e_steps"], "blocks": res["e2e_blocks"], "form": res.get("e2e_form"), "forms": res.get("e2e_forms"),
                "path": "HostStepper.step(): one library call for all batches, its device side captured in one CUDA graph.  compact form (cs_flight_host_pool_step): pinned host actions of all batches -> ONE H2D copy -> one (grouped) step launch -> one pack launch -> two D2H copies into pinned host memory (16-byte records; the agent rows of all envs written in place into the reference-shaped state rows by a strided copy) -> host threads update reward / terminated / win / target_find and the find flags, rewrite target coordinates of reset envs -- all inside the timed region, synchronised every step.  slab form (cs_flight_step_host_many): per batch H2D -> step kernel -> D2H of the whole output slab, batches pipelined over 4 streams (search: cs_search_step_host per batch); median block of %d steps, blocks repeated until >= %d ms" % (res["e2e_steps"], MIN_TIMED_MS)},
        "gpu_launches": int(res["kernels"]),
        "gpu_launches_process_total": int(lib.cs_launch_count() - launches0),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": load_traffic(args.workload), "peak_source": peak_src,
                     "kernel": kernel_name(w, res["lanes_per_env"], res["grouped"]),
                     "algorithmic_bytes_per_env_step": per_unit, "env_steps_per_launch": res["envs_per_launch"],
                     "us_per_launch": 1e6 * sec_per_launch, "map_cells_touched_per_env_step": touched,
                     "note": "duration = timed K-step replay / launches; launches of independent batches overlap when streams > 1"},
        "clocks": clocks,
        "episode_stats_allreduced": dict(zip(cs._lib.STAT_NAMES, [float(x) for x in stats.tolist()])),
        "stats_allreduce_us": allreduce_us,
    }
    if not args.no_extra:
        if world == 1:
            for name in ("c2s", "c2w", "c4"):
                if name == args.workload:
                    continue
                try:
                    r = run_gpu_workload(cs, torch, name, min(args.steps, 60), 5, device, 0, 1, want_e2e=True, burn_in_steps=2000)
                    extra[name] = extra_entry(cs, torch, name, r, peak, device)
                except Exception as exc:
                    extra[name] = {"error": repr(exc)}
            try:
                extra["c4_obs"] = {"workload": "flight get_obs(): prob_map || features for 16384 envs x 3 agents (656 MB per call)",
                                   "unit": "GB/s", "peak": peak, **measure_obs_full(cs, torch, device, peak)}
            except Exception as exc:
                extra["c4_obs"] = {"error": repr(exc)}
            try:
                extra["policy"] = measure_policy(cs, torch, device)
            except Exception as exc:
                extra["policy"] = {"error": repr(exc)}
            try:
                extra["spread"] = measure_spread(cs, torch, device, peak)
            except Exception as exc:
                extra["spread"] = {"error": repr(exc)}
            try:
                extra["c1"] = measure_c1(cs, torch, device)
            except Exception as exc:
                extra["c1"] = {"error": repr(exc)}
            line["cpu_baseline"] = cpu_baseline(w["kind"], w["n"], w["am"], args.cpu_seconds, 4.0)
            _pool.close()
        line["extra"] = extra
    print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
