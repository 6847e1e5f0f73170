"""CPU-side checks of the product package: the C-ABI library loads and exports every symbol the header
declares, the host-built heading table reproduces libm bit for bit, host logic (sharding, error paths)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_of_the_header():
    import coopsearch_b200 as cs
    from coopsearch_b200 import _lib
    lib = cs.load_library()
    header = open(os.path.join(ROOT, "include", "coopsearch.h")).read()
    declared = set(re.findall(r"\b(cs_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 28
    for name in sorted(declared):
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(_lib.SIGNATURES), "ctypes table and header disagree: %s" % (declared ^ set(_lib.SIGNATURES))
    assert lib.cs_version() == 2
    assert lib.cs_launch_count() == 0          # nothing launched by loading


def test_struct_sizes_match_the_header(tmp_path):
    """A C translation unit including the header reports the struct sizes the ctypes mirrors must have."""
    from coopsearch_b200 import _lib
    src = r'''
    #include <stdio.h>
    #include "coopsearch.h"
    int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(cs_flight_cfg), sizeof(cs_flight_buffers),
        sizeof(cs_flight_host_io), sizeof(cs_search_cfg), sizeof(cs_search_buffers), sizeof(cs_search_host_io),
        sizeof(cs_episode_buffers), sizeof(cs_policy_cfg), sizeof(cs_policy_weights), sizeof(cs_policy_io),
        sizeof(cs_spread_cfg), sizeof(cs_spread_buffers), sizeof(cs_flight_host_views)); return 0; }
    '''
    exe = str(tmp_path / "cs_sizes")
    subprocess.run(["gcc", "-x", "c", "-I", os.path.join(ROOT, "include"), "-o", exe, "-"], input=src.encode(), check=True)
    got = [int(v) for v in subprocess.run([exe], capture_output=True, check=True).stdout.split()]
    want = [C.sizeof(t) for t in (_lib.FlightCfg, _lib.FlightBuffers, _lib.FlightHostIO, _lib.SearchCfg,
                                  _lib.SearchBuffers, _lib.SearchHostIO, _lib.EpisodeBuffers, _lib.PolicyCfg,
                                  _lib.PolicyWeights, _lib.PolicyIO, _lib.SpreadCfg, _lib.SpreadBuffers, _lib.FlightHostViews)]
    assert got == want


def reachable_headings(depth):
    a, two_pi, pi, three_pi = np.pi / 18, 2 * np.pi, np.pi, 3 * np.pi
    seen = set()
    for start in (np.pi / 2, 0.0, np.pi):
        s, frontier = {start}, {start}
        for _ in range(depth):
            new = set()
            for h in frontier:
                for d in (0.0, a, -a):
                    g = h + d
                    if g > two_pi:
                        g -= two_pi
                    elif g < 0:
                        g += two_pi
                    new.add(g)
                    new.add(pi - g if g <= pi else three_pi - g)
            frontier = new - s
            s |= frontier
        seen |= s
    return np.array(sorted(seen))


@pytest.mark.parametrize("time_limit", [200, 500])
def test_heading_table_is_libm_bit_for_bit(time_limit):
    """Every heading reachable within `time_limit` steps (flight_env_easy.py:259-266,281-284) is served from the
    table, and the table holds exactly numpy's (= the reference's) sin/cos."""
    import coopsearch_b200 as cs
    lib = cs.load_library()
    vals = reachable_headings(time_limit)
    so, co, ft = np.zeros_like(vals), np.zeros_like(vals), np.zeros(len(vals), np.int32)
    P = lambda x, t: x.ctypes.data_as(C.POINTER(t))
    entries = lib.cs_debug_heading_lut(time_limit, P(vals, C.c_double), len(vals), P(so, C.c_double), P(co, C.c_double),
                                       P(ft, C.c_int32))
    assert entries > 0 and ft.all()
    assert np.array_equal(so, np.sin(vals)) and np.array_equal(co, np.cos(vals))
    # off-lattice headings take the fallback
    odd = np.array([0.3, 1.0, 2.5, 6.0])
    lib.cs_debug_heading_lut(time_limit, P(odd, C.c_double), 4, P(so, C.c_double), P(co, C.c_double), P(ft, C.c_int32))
    assert not ft[:4].any()


def test_create_rejects_bad_configs_without_a_gpu():
    """Argument validation happens before any CUDA call, with the reference's messages."""
    import coopsearch_b200 as cs
    from coopsearch_b200 import _lib
    lib = cs.load_library()
    cfg = _lib.FlightCfg(struct_size=C.sizeof(_lib.FlightCfg), num_envs=4, n_agents=3, target_num=15, map_size=50,
                         view_range=7, time_limit=200, agent_mode=9, target_mode=0, variant=0, device=0,
                         velocity=1, detect_prob=0.9, safe_dist=1, force_dist=3)
    h = C.c_void_p()
    assert lib.cs_flight_create(C.byref(cfg), C.byref(h)) == -1
    assert b"No such agent mode" in lib.cs_last_error()
    cfg.agent_mode, cfg.target_mode = 0, 4
    assert lib.cs_flight_create(C.byref(cfg), C.byref(h)) == -1
    assert b"No such target mode" in lib.cs_last_error()
    cfg.target_mode, cfg.struct_size = 0, 8
    assert lib.cs_flight_create(C.byref(cfg), C.byref(h)) == -1
    assert b"ABI mismatch" in lib.cs_last_error()
    scfg = _lib.SearchCfg(struct_size=C.sizeof(_lib.SearchCfg), num_envs=1, n_agents=3, target_num=15, map_size=50,
                          view_range=7, agent_mode=3, target_mode=0)
    assert lib.cs_search_create(C.byref(scfg), C.byref(h)) == -1
    assert b"Unknown agent mode" in lib.cs_last_error()


def test_env_construction_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import types
    import coopsearch_b200 as cs
    args = types.SimpleNamespace(map_size=50, target_num=15, target_mode=1, agent_mode=0, n_agents=3, view_range=7,
                                 time_limit=200, detect_prob=0.9, safe_dist=1, agent_velocity=1, force_dist=3)
    with pytest.raises(cs.CoopSearchError, match="no CPU fallback"):
        cs.VecFlightEasyEnv(args, None, num_envs=2)
    with pytest.raises(cs.CoopSearchError, match="no CPU fallback"):
        cs.VecSearchEnv(args, num_envs=2)


def test_load_targets_parses_like_main_py(tmp_path):
    import coopsearch_b200 as cs
    import golden_util as gu
    p = tmp_path / "t.txt"
    lines = ["position(X10^5m)    determinacy    priority        dx             dy\r\n"]
    for j in range(15):
        lines.append("%s    %s\t\t%s\t   %d      %s     %s\r\n" % (gu.TEMPLATE["x"][j], gu.TEMPLATE["y"][j], gu.TEMPLATE["deter"][j],
                                                                  gu.TEMPLATE["priority"][j], gu.TEMPLATE["dx"][j], gu.TEMPLATE["dy"][j]))
    lines.append("\r\n")
    p.write_text("".join(lines))
    got = cs.load_targets(str(p))
    assert got == {k: [float(v) if k in ("x", "y", "dx", "dy") else v for v in gu.TEMPLATE[k]] for k in gu.TEMPLATE}


def test_shard_range_partitions_exactly():
    from coopsearch_b200 import dist
    for total in (1, 7, 4096, 65536, 1048576, 1000003):
        for world in (1, 2, 3, 4, 8):
            spans = [dist.shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        dist.shard_range(10, 2, 2)


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import torch
    import torch.distributed as td
    from coopsearch_b200 import dist
    import golden_util as gu
    from oracle import c_oracle
    from oracle.py_envs import FlightSpec
    r, _, w = dist.init_from_env(backend="gloo")
    # each rank steps ITS shard of 64 global envs on the CPU oracle (the shard logic is what is under test)
    lo, hi = dist.shard_range(64, r, w)
    spec = FlightSpec(n_agents=3, time_limit=30)
    b = c_oracle.FlightBatch(spec, gu.TEMPLATE, 5, lo, hi - lo, auto_reset=True)
    b.reset(init=True)
    stats = np.zeros(8)
    for t in range(60):
        rew, term, win = b.step(None)
        stats[5] += hi - lo
        stats[0] += term.sum()
        stats[3] += win[term.astype(bool)].sum()
    total = dist.allreduce_stats(stats)
    slow = dist.max_over_ranks(float(r + 1))
    q.put((r, total.tolist(), slow, b.found.tolist()))
    td.destroy_process_group()


def test_two_rank_gloo_stat_allreduce_and_shard_invariance():
    """world_size 2 over gloo: the summed statistics equal the single-process run, and the concatenated
    per-rank states equal the unsharded state (global-id keyed draws)."""
    import multiprocessing as mp
    import golden_util as gu
    from oracle import c_oracle
    from oracle.py_envs import FlightSpec
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 300
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    spec = FlightSpec(n_agents=3, time_limit=30)
    b = c_oracle.FlightBatch(spec, gu.TEMPLATE, 5, 0, 64, auto_reset=True)
    b.reset(init=True)
    stats = np.zeros(8)
    for t in range(60):
        rew, term, win = b.step(None)
        stats[5] += 64
        stats[0] += term.sum()
        stats[3] += win[term.astype(bool)].sum()
    assert outs[0][1] == outs[1][1] == stats.tolist()
    assert outs[0][2] == outs[1][2] == 2.0
    assert outs[0][3] + outs[1][3] == b.found.tolist()
