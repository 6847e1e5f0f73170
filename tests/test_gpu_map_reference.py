"""The belief-map kernels (csrc/flight_map.cuh) judged call by call against the float64 reference oracle/map_ref.py.

Every sensing call is checked on every env and every cell of the reference-shaped map: the map the kernel exported
before the call, the positions it sensed from (agent_xy after the step) and the targets it found (the new-found meta
word) go into the reference; corner counts, touched set, untouched cells, found cells and p = 1 cells must come out
exact, the touched-cell statistic must grow by the reference's count, and every other cell must lie within the bound
of the kernel's fp32 arithmetic plus the term of its fp32-pair q.  The padding cells of the tiled layout (rows and columns
>= M) are not part of that map and are not asserted on.

(a) the benchmark's shape, 400+ calls, tiled form with and without map_overlap; (b) a geometry x form x detect_prob
grid; (c) placements that put corners exactly on, and one ulp off, R^2, fp32 interval ends on both sides of the
1e-3 guard band, agents on corner rows 0 and M and at y = 63 with M = 63; (d) the benchmark's own configuration and
stepping (auto-reset, map_overlap, replays of a CUDA graph) for 6000 + 60 steps against the C oracle; (e) the
end-to-end margin against the 1e-5 bar at lower detect_prob on a crowded map, split into what q = 1 - d rounded to
fp32 would explain and the rest.  Each test prints its largest ratio / relative error."""
import os

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import c_oracle, map_ref
from oracle.py_envs import FlightSpec
from test_gpu_flight_easy import make_args, cpu

pytestmark = pytest.mark.gpu
META_NEWFOUND = 1
MAP_RTOL, MAP_ATOL = 1e-5, 1e-37


def _env(spec, E, lanes=0, seed=3, template=None, **kw):
    import coopsearch_b200 as cs
    return cs.VecFlightEnv(make_args(dict(spec.__dict__)), template, num_envs=E, seed=seed, env_id_base=500,
                           count_touched=True, lanes_per_env=lanes, **kw)


def _touched(env):
    return int(env.stats()["map_cells_touched"])


def checked_call(env, spec, fn, worst, mask=None):
    """Runs fn() (one step or reset(mask)) and checks the map update it made on every env (or on the envs of mask)."""
    before = env.prob_map.clone()
    t0 = _touched(env)
    fn()
    after = env.prob_map
    xy = env.agent_xy.clone()
    newf = env._meta_word(META_NEWFOUND).clone()
    tgt = env.tgt_xy.clone()
    if mask is not None:
        idx = mask.nonzero().flatten()
        others = mask == 0
        assert torch.equal(after[others].view(torch.int32), before[others].view(torch.int32)), \
            "a reset changed the map of an env it did not reset"
        before, after, xy, newf, tgt = before[idx], after[idx], xy[idx], newf[idx], tgt[idx]
    return map_ref.check_call(after, before, xy, spec.map_size, spec.view_range, spec.detect_prob, tgt, newf,
                              touched_delta=_touched(env) - t0, worst=worst)


def random_map(E, M, gen, ones=0.03):
    m = torch.rand(E, M, M, generator=gen, device="cuda") ** 4
    m[torch.rand(E, M, M, generator=gen, device="cuda") < ones] = 1.0
    return m


def run_checked(env, spec, calls, worst, seed=0):
    """`calls` steps with uniform-random actions; finished envs are reset by reset(mask=terminated) (one sensing job
    per call, the map carries over), and that reset is checked as a call of its own."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for t in range(calls):
        a = torch.randint(0, 3, (env.num_envs, spec.n_agents), generator=gen, device="cuda", dtype=torch.uint8)
        out = {}
        checked_call(env, spec, lambda: out.update(term=env.step(a)[1].clone()), worst)
        term = out["term"]
        if bool(term.any()):
            checked_call(env, spec, lambda: env.reset(mask=term), worst, mask=term)


def _print(tag, worst):
    print("\n%s: largest |error| / bound %.4f (rounding terms alone %.4f), pow/mul disagreements %d of %d corners "
          "within %d ulp of R^2, %d calls" % (tag, worst.get("total", 0), worst.get("rounding", 0), worst.get("pow_diff", 0),
                                               worst.get("pow_checked", 0), map_ref.POW_WINDOW, worst.get("calls", 0)))


# ------------------------------------------------------------------------------------------------------------- (a)
@pytest.mark.parametrize("overlap", [False, True])
def test_c4_shape_every_call(overlap):
    spec = FlightSpec(n_agents=3, target_num=15, map_size=50, view_range=7, detect_prob=0.9, variant="probmap")
    env = _env(spec, 16384, template=gu.TEMPLATE, seed=42, map_overlap=overlap)
    worst = {}
    run_checked(env, spec, 400, worst, seed=1)
    _print("(a) c4 shape, 16384 envs, map_overlap=%s" % overlap, worst)
    assert worst["calls"] >= 400


# ------------------------------------------------------------------------------------------------------------- (b)
MS = [5, 16, 17, 50, 62, 63, 64, 100]
RS = [1, 2, 7, 9, 15]
NS = [1, 3, 8, 9]
DS = [0.9, 0.5, 0.1, 0.0, 1.0]


@pytest.mark.parametrize("lanes", [0, 8, 16])
@pytest.mark.parametrize("M", MS)
def test_geometry_grid_every_call(M, lanes):
    """Every view range at every map size and form; agent count and detect_prob rotate through their lists so that
    each (M, R) pair meets a different n and d in each form (R = 15 covers a disc larger than the map for M <= 17)."""
    worst = {}
    k = MS.index(M)
    for i, R in enumerate(RS):
        n = NS[(k + i + lanes // 8) % len(NS)]
        d = DS[(k + 2 * i + lanes // 8) % len(DS)]
        spec = FlightSpec(n_agents=n, target_num=6, map_size=M, view_range=R, detect_prob=d, agent_mode=(i + k) % 4,
                          target_mode=1, variant="probmap", time_limit=25)
        env = _env(spec, 192, lanes=lanes, seed=7 + i)
        gen = torch.Generator(device="cuda").manual_seed(k * 10 + i)
        env.prob_map = random_map(env.num_envs, M, gen)
        run_checked(env, spec, 40, worst, seed=i)
    _print("(b) M=%d lanes=%d" % (M, lanes), worst)


# ------------------------------------------------------------------------------------------------------------- (c)
def adversarial_cases(M, R):
    """Sensed positions [cases, n=3, 2], agents of a case > force_dist + 1.01 v = 4.01 apart."""
    up, dn = np.nextafter(10.0, 11.0), np.nextafter(10.0, 9.0)
    far = lambda x, y: [[x, y], [x + 4.5, y + 0.25], [x + 0.25, y + 4.75]]      # three overlapping discs
    cases = [
        far(10.0, 10.0),                   # corners exactly at R^2 (axis-aligned; 3-4-5 with R = 5), union of ties
        far(up, 10.0), far(dn, 10.0),      # one ulp inside / outside R^2
        far(10.0, up), far(10.0, dn),
    ]
    for base in (20.0, 7.0):
        for frac in (1e-3, 1.0 - 1e-3):
            for dlt in (2e-6, -2e-6, 2e-5, -2e-5):   # fp32 interval ends 1e-3 +- delta from an integer: both sides of the band
                cases.append(far(10.0, base + frac + dlt))
                cases.append(far(10.5, base + frac + dlt))
    cases.append(far(0.0, 10.0))           # agent on corner row 0 (x) and column 0 (y) below
    cases.append(far(10.0, 0.0))
    cases.append([[float(M), 10.0], [float(M) - 4.5, 10.25], [float(M), 14.75]])      # corner row M
    cases.append([[10.0, float(M)], [14.5, float(M)], [10.25, float(M) - 4.75]])      # corner column M (bit M)
    cases.append([[20.0, float(M) - 0.1], [24.5, float(M)], [20.25, float(M) - 4.75]])
    return np.array(cases, dtype=np.float64)


@pytest.mark.parametrize("lanes", [0, 8, 16])
@pytest.mark.parametrize("M,R", [(50, 7), (50, 5), (63, 7), (40, 5), (64, 5)])
def test_adversarial_placements(M, R, lanes):
    """Each case is placed on its own env: pre-step positions = sensed - (v, 0), heading 0, action 0 (turns by 0),
    so the step kernel senses from exactly the intended point.  The agents of a case stay more than force_dist + 1.01 v
    apart, so no repulsion moves them.  Positions that the move takes just outside [0, M] are clamped onto the edge."""
    sensed = adversarial_cases(M, R)
    E, n = sensed.shape[0], sensed.shape[1]
    spec = FlightSpec(n_agents=n, target_num=6, map_size=M, view_range=R, detect_prob=0.9, target_mode=1, variant="probmap",
                      time_limit=500)
    env = _env(spec, E, lanes=lanes, seed=9)
    gen = torch.Generator(device="cuda").manual_seed(M + R)
    env.prob_map = random_map(E, M, gen, ones=0.1)
    pre = sensed.copy()
    pre[:, :, 0] -= 1.0
    edge = sensed[:, :, 0] >= M                        # reached by a move that ends just past M: clamped to M
    pre[edge, 0] = M - 1.0 + 1e-12
    env.agent_xy.copy_(torch.from_numpy(pre).cuda())
    env.agent_yaw.zero_()
    # targets placed onto agents' cells so that some are found this call (detect_prob 0.9)
    tg = np.repeat(sensed[:, :1], 6, axis=1) + np.linspace(-0.4, 0.4, 6)[None, :, None]
    env.tgt_xy.copy_(torch.from_numpy(tg).cuda())
    worst = {}
    zero = torch.zeros(E, n, dtype=torch.uint8, device="cuda")
    for t in range(4):                                 # the placed call, then onward from there
        out = {}
        checked_call(env, spec, lambda: out.update(term=env.step(zero)[1].clone()), worst)
        if t == 0:
            got = cpu(env.agent_xy)
            want = np.clip(sensed, 0, M)
            assert np.array_equal(got, want), np.argwhere(got != want)
            ties = map_ref.corner_sums(torch.from_numpy(want).cuda(), M) == float(R * R)
            assert bool(ties.any())
        term = out["term"]
        if bool(term.any()):                           # an env that found all its targets is not sensed again until reset
            checked_call(env, spec, lambda: env.reset(mask=term), worst, mask=term)
    _print("(c) M=%d R=%d lanes=%d" % (M, R, lanes), worst)


# ------------------------------------------------------------------------------------------------------------- (d)
def _relerr(got, want):
    """largest |got - want| / |want| over cells with |want| > atol; and whether rtol/atol holds everywhere"""
    want32 = want.astype(np.float32).astype(np.float64)
    ok = np.abs(got - want32) <= MAP_ATOL + MAP_RTOL * np.abs(want32)
    big = np.abs(want) > MAP_ATOL
    rel = np.abs(got.astype(np.float64) - want)[big] / np.abs(want[big])
    return (float(rel.max()) if rel.size else 0.0), bool(ok.all())


def test_benchmark_horizon_against_c_oracle(oracle_squares_by_multiplication):
    """c4 as bench.py builds it -- 16384 envs, auto_reset, map_overlap, steps replayed from a K-step CUDA graph with a
    pool of 8 device action tensors -- for 6000 + 60 steps.  A 512-env slice is stepped by the C oracle (multiplication
    squares); the device's per-step discrete outputs of that slice are recorded inside the graph."""
    import coopsearch_b200 as cs
    E, S, K, POOL = 16384, 512, 10, 8
    STEPS = 6060
    spec = FlightSpec(n_agents=3, target_num=15, map_size=50, view_range=7, detect_prob=0.9, variant="probmap")
    env = cs.VecFlightEnv(make_args(dict(spec.__dict__)), gu.TEMPLATE, num_envs=E, seed=42, env_id_base=0,
                          auto_reset=True, map_overlap=True)
    orc = c_oracle.FlightBatch(spec, gu.TEMPLATE, 42, 0, S, auto_reset=True)
    c_oracle.set_threads(max(1, min(16, os.cpu_count() or 1)))
    try:
        orc.reset(init=True)
        np.testing.assert_allclose(cpu(env.tgt_xy[:S]), orc.tgt, rtol=0, atol=1e-9)
        orc.tgt[...] = cpu(env.tgt_xy[:S])
        assert _relerr(cpu(env.prob_map[:S]).astype(np.float64), orc.map)[1]
        gen = torch.Generator(device="cuda").manual_seed(1234)
        pool = [torch.randint(0, 3, (E, 3), generator=gen, device="cuda", dtype=torch.uint8) for _ in range(POOL)]
        pool_np = [cpu(a[:S]) for a in pool]
        hist = {k: torch.zeros((K, S), dtype=torch.int64, device="cuda") for k in ("found", "term", "win", "time", "reward")}
        side = torch.cuda.Stream()

        def record(k):
            hist["found"][k].copy_(env.found_mask[:S])
            hist["term"][k].copy_(env._terminated[:S])
            hist["win"][k].copy_(env.win_flag[:S])
            hist["time"][k].copy_(env.time_step[:S])
            hist["reward"][k].copy_(env._reward[:S].to(torch.int64))

        worst_rel, worst_at = 0.0, -1
        with torch.cuda.stream(side):
            env.step(pool[0]); env.sync_map()                  # the eager step bench.py takes before its capture
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for k in range(K):
                    env.step(pool[k % POOL])
                    record(k)
                env.sync_map()
        torch.cuda.synchronize()
        r, t, w = orc.step(pool_np[0])
        assert np.array_equal(cpu(env.found_mask[:S]).astype(np.uint32), orc.found)
        done = 1
        while done < STEPS:
            with torch.cuda.stream(side):
                g.replay()
            torch.cuda.synchronize()
            h = {k: cpu(v) for k, v in hist.items()}
            for k in range(K):
                r, t, w = orc.step(pool_np[k % POOL])
                where = "step %d" % (done + k)
                assert np.array_equal(h["found"][k].astype(np.uint32), orc.found.astype(np.int64).astype(np.uint32)), where
                assert np.array_equal(h["term"][k], t.astype(np.int64)) and np.array_equal(h["win"][k], w.astype(np.int64)), where
                assert np.array_equal(h["time"][k], orc.time_step.astype(np.int64)), where
                assert np.array_equal(h["reward"][k], r.astype(np.int64)), where
            done += K
            # device-drawn targets (Box-Muller with CUDA log / sincos, ~1e-15 from glibc's) into the oracle
            np.testing.assert_allclose(cpu(env.tgt_xy[:S]), orc.tgt, rtol=0, atol=1e-9)
            orc.tgt[...] = cpu(env.tgt_xy[:S])
            if (done - 1) % 500 == 0 or done >= STEPS:
                np.testing.assert_array_equal(cpu(env.agent_xy[:S]), orc.xy, err_msg="step %d" % done)
                rel, ok = _relerr(cpu(env.prob_map[:S]).astype(np.float64), orc.map)
                if rel > worst_rel:
                    worst_rel, worst_at = rel, done
                assert ok, "map outside rtol %g / atol %g after %d steps (largest relative error %.3g)" % (MAP_RTOL, MAP_ATOL, done, rel)
        print("\n(d) c4 as benchmarked, %d steps, 512-env slice: largest map relative error %.3g (after %d steps)" %
              (done, worst_rel, worst_at))
    finally:
        c_oracle.set_threads(1)


# ------------------------------------------------------------------------------------------------------------- (e)
@pytest.mark.parametrize("d", [0.5, 0.2, 0.05])
def test_detect_prob_sweep_margin(d, oracle_squares_by_multiplication):
    """M = 16, 8 agents, R = 7: nearly every cell is in view at every call, so a cell stays above atol for ~ -85/ln(q)
    calls.  Compared end to end with the C oracle (per-step discrete outputs exact, map within rtol 1e-5 / atol 1e-37).
    The largest relative error is split with float64 shadow maps evolved by map_ref from the device's own positions
    and found targets: q = 1 - d (the reference), q = qf + ql (the fp32 pair the kernels carry) and q = fl32(1 - d)
    (what the kernels carried before)."""
    E, T = 256, 2000
    spec = FlightSpec(n_agents=8, target_num=15, map_size=16, view_range=7, detect_prob=d, target_mode=1, variant="probmap")
    env = _env(spec, E, seed=13, reset=False)
    orc = c_oracle.FlightBatch(spec, None, 13, 500, E)
    c_oracle.set_threads(max(1, min(16, os.cpu_count() or 1)))
    try:
        orc.reset(init=True)
        env.reset(init=True, targets=orc.tgt)
        q32 = float(np.float32(1.0 - d))
        shadow = {k: torch.from_numpy(orc.map.copy()).cuda() for k in ("q", "pair", "fp32")}
        assert _relerr(cpu(env.prob_map).astype(np.float64), orc.map)[1]
        rng = np.random.default_rng(int(d * 100))
        worst = {"e2e": 0.0, "shadow": 0.0, "pair_part": 0.0, "fp32_part": 0.0, "rest": 0.0}

        def shadow_call(idx=None):
            xy, tgt, newf = env.agent_xy.clone(), env.tgt_xy.clone(), env._meta_word(META_NEWFOUND).clone()
            sel = slice(None) if idx is None else idx
            s = map_ref.sense(xy[sel], 16, 7, tgt[sel], newf[sel])
            shadow["q"][sel] = map_ref.update(shadow["q"][sel], s, d)["want"]
            shadow["pair"][sel] = map_ref.update(shadow["pair"][sel], s, d)["want_qf"]
            shadow["fp32"][sel] = map_ref.update(shadow["fp32"][sel], s, d, qk=q32)["want_qf"]

        for t in range(T):
            a = rng.integers(0, 3, size=(E, 8), dtype=np.uint8)
            _, term, _ = env.step(a)
            r, ot, ow = orc.step(a)
            shadow_call()
            where = "d=%g step %d" % (d, t)
            assert np.array_equal(cpu(env.found_mask).astype(np.uint32), orc.found), where
            assert np.array_equal(cpu(term), ot), where
            if ot.any():
                m = torch.from_numpy(ot).cuda()
                env.reset(mask=m)
                orc.reset(mask=ot)
                np.testing.assert_allclose(cpu(env.tgt_xy), orc.tgt, rtol=0, atol=1e-9, err_msg=where)
                orc.tgt[...] = cpu(env.tgt_xy)
                shadow_call(m.nonzero().flatten())
            if t % 100 == 99 or t == T - 1:
                got = cpu(env.prob_map).astype(np.float64)
                rel, ok = _relerr(got, orc.map)
                worst["e2e"] = max(worst["e2e"], rel)
                sq = cpu(shadow["q"])
                worst["shadow"] = max(worst["shadow"], _relerr(sq, orc.map)[0])
                worst["pair_part"] = max(worst["pair_part"], _relerr(cpu(shadow["pair"]), sq)[0])
                worst["fp32_part"] = max(worst["fp32_part"], _relerr(cpu(shadow["fp32"]), sq)[0])
                worst["rest"] = max(worst["rest"], _relerr(got, cpu(shadow["pair"]))[0])
                assert ok, "%s: map outside rtol %g (largest relative error %.3g)" % (where, MAP_RTOL, rel)
        print("\n(e) d=%g, M=16 n=8 R=7, %d steps: largest map relative error %.3g; q as fp32 alone would explain %.3g, "
              "q as the fp32 pair %.3g; the rest (device against the pair's float64 map) %.3g; shadow map against the "
              "C oracle %.3g" % (d, T, worst["e2e"], worst["fp32_part"], worst["pair_part"], worst["rest"], worst["shadow"]))
    finally:
        c_oracle.set_threads(1)
