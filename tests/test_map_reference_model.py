"""The float64 belief-map reference (oracle/map_ref.py) checked on its own, on any box.

1. With pow squares and the reference's operation order it reproduces the committed flight fixtures bit for bit (maps
   after every sampled step, the final map and the second episode's map), evolving its own float64 map call by call.
2. It equals the C oracle's map update on random inputs, bit for bit, including the touched count.
3. An fp32 emulation of belief_f4 (flight_map.cuh) with a correctly rounded reciprocal lies inside its bound on random
   and adversarial cells.
4. Plausible kernel mistakes, restated on that emulation or on the corner classification, land outside the bound or
   break an exact requirement."""
import math

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import c_oracle, map_ref
from oracle.py_envs import FlightSpec

FLAG_DONE = 2


def _sensing_now(orc, M, R, square="pow"):
    xy = torch.from_numpy(orc.xy.copy())
    tgt = torch.from_numpy(orc.tgt.copy())
    newf = torch.from_numpy(orc.meta[:, 1].astype(np.int64))
    return map_ref.sense(xy, M, R, tgt, newf, square=square)


def _apply(shadow, s, d, live):
    u = map_ref.update(shadow, s, d, arith="reference")
    return torch.where(torch.from_numpy(live).view(-1, 1, 1), u["want"], shadow)


@pytest.mark.parametrize("name", gu.FLIGHT_FIXTURES)
def test_reproduces_reference_fixtures_bit_for_bit(name):
    g = gu.load(name)
    kw, base, seed = gu.flight_spec_kwargs(g, "probmap")
    spec = FlightSpec(**kw)
    M, R, d = spec.map_size, spec.view_range, spec.detect_prob
    T, E = g["reward"].shape
    orc = c_oracle.FlightBatch(spec, None, seed, base, E)          # positions and found targets only
    orc.reset(targets=g["tgt_xy"], init=True)
    shadow = _apply(torch.full((E, M, M), 0.5, dtype=torch.float64), _sensing_now(orc, M, R), d, np.ones(E, bool))
    assert np.array_equal(shadow.numpy(), g["init_map"])
    for t in range(T):
        live = (orc.meta[:, 5] & FLAG_DONE) == 0                  # a finished env is not sensed again
        orc.step(g["actions"][t])
        assert np.array_equal(orc.xy, g["xy"][t]) and np.array_equal(orc.found, g["found"][t])
        shadow = _apply(shadow, _sensing_now(orc, M, R), d, live)
        if (t + 1) in g["map_steps"]:
            assert np.array_equal(shadow.numpy(), g["maps"][list(g["map_steps"]).index(t + 1)]), (name, t)
    assert np.array_equal(shadow.numpy(), g["final_map"])
    orc.meta[:, 5] &= ~np.uint32(FLAG_DONE)
    orc.reset(targets=g["ep2_tgt_xy"], init=False)
    shadow = _apply(shadow, _sensing_now(orc, M, R), d, np.ones(E, bool))
    for t in range(g["ep2_actions"].shape[0]):
        live = (orc.meta[:, 5] & FLAG_DONE) == 0
        orc.step(g["ep2_actions"][t])
        assert np.array_equal(orc.found, g["ep2_found"][t])
        shadow = _apply(shadow, _sensing_now(orc, M, R), d, live)
    assert np.array_equal(shadow.numpy(), g["ep2_map"])


@pytest.mark.parametrize("square", ["pow", "mul"])
@pytest.mark.parametrize("d", [0.9, 0.5, 0.1, 0.0, 1.0])
@pytest.mark.parametrize("M,R,n", [(20, 5, 3), (17, 7, 8), (9, 15, 2), (40, 2, 5)])
def test_equals_c_oracle_on_random_inputs(M, R, n, d, square):
    rng = np.random.default_rng(M * 100 + R * 10 + n + int(d * 1000))
    E = 64
    spec = FlightSpec(n_agents=n, map_size=M, view_range=R, detect_prob=d, variant="probmap", target_mode=1, time_limit=1000)
    c_oracle.set_square(square)
    try:
        orc = c_oracle.FlightBatch(spec, None, 7, 100, E)
        orc.reset(init=True)
        for call in range(6):
            # random positions (half of the envs on integer points, where corners tie with R^2), random maps with cells
            # at exactly 1 and 0, targets near the agents so that some are found
            xy = rng.uniform(-1, M + 1, size=(E, n, 2))
            xy[: E // 2] = np.round(xy[: E // 2])
            orc.xy[...] = xy
            orc.yaw[...] = rng.uniform(0, 2 * np.pi, size=(E, n))
            pm = rng.uniform(0, 1, size=(E, M, M)) ** 3
            pm[rng.uniform(size=pm.shape) < 0.05] = 1.0
            pm[rng.uniform(size=pm.shape) < 0.02] = 0.0
            orc.map[...] = pm
            orc.tgt[...] = xy[:, rng.integers(0, n, size=spec.target_num)] + rng.normal(0, 2, size=(E, spec.target_num, 2))
            orc.meta[:, 0] = 0
            orc.meta[:, 5] = 0                                       # not finished: every env senses
            t0 = int(orc.touched[0])
            orc.step(rng.integers(0, 3, size=(E, n), dtype=np.uint8))
            s = _sensing_now(orc, M, R, square)
            got = map_ref.update(torch.from_numpy(pm), s, d, arith="reference")["want"].numpy()
            assert np.array_equal(got, orc.map, equal_nan=True), call
            assert int(s.n_touched.sum()) == int(orc.touched[0]) - t0
    finally:
        c_oracle.set_square("pow")


# ---------------------------------------------------------------------------------------------------- fp32 emulation
def fma32(a, b, c):
    """fp32 fma: a*b is exact in float64 (48 bits), the sum rounds in float64 and then to fp32 (double rounding stays
    within 2^-53 of the single rounding, inside the reference's slack)"""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def rcp_exact(x):
    return (1.0 / x.astype(np.float64)).astype(np.float32)


def rcp_bf16(x):
    return torch.from_numpy(rcp_exact(x)).to(torch.bfloat16).to(torch.float32).numpy()


def belief_emul(p, counts, found, d, rcp=rcp_exact, q_of=lambda d: 1.0 - d, pair=True, one_case=True, found_mode="touched"):
    """belief_f4 / belief_cell (flight_map.cuh, flight_common.cuh) in numpy fp32, then the found-cell store.
    pair=False: q rounded to fp32 alone (ql = 0), as the kernels did before they carried q as a pair.
    found_mode: "touched" (the kernel: found and touched -> 1), "always" (mistake: found -> 1 even untouched),
    "never" (mistake: the store is lost)"""
    p = p.astype(np.float32)
    q = q_of(d)
    qf = np.float32(q)
    ql = np.float32(q - np.float64(qf)) if pair else np.float32(0)
    w = np.float32(0.25) * counts.astype(np.float32)       # build_cell_lut
    u = (counts == 0).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        qp = fma32(np.full_like(p, qf), p, ql * p)
        num, keep = w * qp, u * p
        den = qp + (np.float32(1.0) - p)
        res = fma32(num, rcp(den), keep)
    if qf == 0:
        res = np.where(u != 0, p, res)
    elif one_case:
        res = np.where((p == 1) & (u == 0), np.float32(0.25) * counts.astype(np.float32), res)
    if found_mode == "touched":
        res = np.where(found & (counts > 0), np.float32(1), res)
    elif found_mode == "always":
        res = np.where(found, np.float32(1), res)
    return res


def adversarial_cells(rng, N):
    """p, counts, found: log-uniform p down to the smallest subnormal, and the edges (0, 1, 1/2, 1 - 2^-24, subnormal
    boundaries, p whose num = c*p is subnormal)"""
    e = rng.uniform(0, 150, size=N)
    p = (2.0 ** -e) * rng.uniform(0.5, 1, size=N)
    special = np.array([0.0, 1.0, 0.5, 1 - 2.0 ** -24, 1 - 2.0 ** -23, 2.0 ** -149, 2.0 ** -126, 2.0 ** -127,
                        3 * 2.0 ** -149, 2.0 ** -124, 0.9999, 1e-38, 1e-30, 0.25, 0.75])
    p[: special.size * 5] = np.repeat(special, 5)
    p = p.astype(np.float32)
    counts = rng.integers(0, 5, size=N)
    counts[: special.size * 5] = np.tile(np.arange(5), special.size)
    found = rng.uniform(size=N) < 0.05
    return p, counts, found


def _judge(res, p, counts, found, d):
    s = map_ref.Sensing.from_counts(torch.from_numpy(counts).view(1, -1, 1), torch.from_numpy(found).view(1, -1, 1))
    u = map_ref.update(torch.from_numpy(p).view(1, -1, 1), s, d)
    got = torch.from_numpy(res).view(1, -1, 1)
    total = map_ref.bound_ratio(got, u["want"], u["bound"] + u["bound_q"], u["exact"])
    rounding = map_ref.bound_ratio(got, u["want_qf"], u["bound"], u["exact"])
    return total.flatten(), rounding.flatten(), u


DS = [0.9, 0.5, 0.2, 0.1, 0.05, 0.0, 1.0, 0.999, 1e-6, 1 / 3]


@pytest.mark.parametrize("d", DS)
def test_fp32_emulation_within_bound(d):
    rng = np.random.default_rng(int(d * 1e6) + 3)
    p, counts, found = adversarial_cells(rng, 200_000)
    total, rounding, u = _judge(belief_emul(p, counts, found, d), p, counts, found, d)
    assert float(total.max()) <= 1.0 and float(rounding.max()) <= 1.0
    nonexact = ~u["exact"].flatten()
    print("d=%g: largest |error| / bound %.3f (rounding terms alone, against F(qf + ql): %.3f) over %d cells" %
          (d, float(total.max()), float(rounding[nonexact].max()), int(nonexact.sum())))


def _report(name, ratio, affected):
    r = ratio[affected]
    r = r[torch.isfinite(r)]
    inf = int((~torch.isfinite(ratio[affected])).sum())
    med = float(r.median()) if r.numel() else float("inf")
    mn = float(r.min()) if r.numel() else float("inf")
    print("%-44s cells changed %6d  exact requirement broken %6d  finite ratio median %.3g min %.3g" %
          (name, int(affected.sum()), inf, med, mn))
    return inf, mn


@pytest.mark.parametrize("d", [0.05, 0.2])
def test_q_pair_keeps_long_lived_cells_within_the_bar(d):
    """A cell in full view at every call, from 0.5 until it drops below atol 1e-37 (~1700 calls at d = 0.05).  With q
    rounded to fp32 alone every call shifts the cell by |fl32(q) - q| / q in the same direction and the sum passes the
    maps' rtol 1e-5 at d = 0.05; with q carried as an fp32 pair what remains is the rounding walk."""
    q = 1.0 - d
    p64, worst = np.array([0.5]), {True: 0.0, False: 0.0}
    p32 = {True: np.array([0.5], np.float32), False: np.array([0.5], np.float32)}
    four, none = np.array([4]), np.array([False])
    while p64[0] > 1e-37:
        p64 = q * p64 / (q * p64 + (1 - p64))
        for pair in (True, False):
            p32[pair] = belief_emul(p32[pair], four, none, d, pair=pair)
            worst[pair] = max(worst[pair], abs(float(p32[pair][0]) - p64[0]) / p64[0])
    print("d=%g: largest relative error, q as fp32 pair %.3g, q as fp32 %.3g" % (d, worst[True], worst[False]))
    assert worst[True] < 1e-5
    if d == 0.05:
        assert worst[False] > 1e-5


@pytest.mark.parametrize("mutant", ["rcp_bf16", "q_is_d", "no_exact_one", "found_untouched", "found_lost"])
def test_update_mistakes_fall_outside_the_bound(mutant):
    # with a correctly rounded reciprocal, fl(fl(count qf / 4) fl(1 / qf)) happens to equal count / 4 for most d, so the
    # p = 1 case shows at a d where it does not (the device's 1-ulp rcp.approx may miss it at others)
    d = 0.15 if mutant == "no_exact_one" else 0.9
    rng = np.random.default_rng(11)
    p, counts, found = adversarial_cells(rng, 200_000)
    kw = {"rcp_bf16": dict(rcp=rcp_bf16), "q_is_d": dict(q_of=lambda d: d), "no_exact_one": dict(one_case=False),
          "found_untouched": dict(found_mode="always"), "found_lost": dict(found_mode="never")}[mutant]
    good = belief_emul(p, counts, found, d)
    bad = belief_emul(p, counts, found, d, **kw)
    total, _, u = _judge(bad, p, counts, found, d)
    changed = torch.from_numpy(good.view(np.uint32) != bad.view(np.uint32))
    assert bool(changed.any())
    _report(mutant, total, changed)
    assert float(total.max()) > 1.0
    # every changed cell in the normal range is caught; below it the absolute subnormal term of the bound can hide a
    # relative mistake.  A bf16 reciprocal is exact or nearly so for some denominators: most cells, not all, show it.
    normal = changed & (u["want"].flatten().abs() >= 2.0 ** -100)
    caught = (total[normal] > 1).float().mean().item()
    print("%s: %.4f of the changed normal-range cells out of bound" % (mutant, caught))
    assert caught >= (0.75 if mutant == "rcp_bf16" else 1.0), caught


# ------------------------------------------------------------------------------------------ classification mistakes
def _tie_geometry(E=48, M=24, R=5, n=3, seed=5):
    """Agents on integer and half-integer points (3-4-5 ties with R = 5, axis-aligned ties), targets in view"""
    rng = np.random.default_rng(seed)
    xy = rng.integers(0, M + 1, size=(E, n, 2)).astype(np.float64)
    xy[E // 2:] += rng.choice([0.0, 0.5, 0.25], size=(E - E // 2, n, 2))
    tgt = xy[:, rng.integers(0, n, size=6)] + rng.uniform(-3, 3, size=(E, 6, 2))
    tgt[:, 0] = np.floor(tgt[:, 0]) + 0.6                            # round and trunc disagree here
    newf = rng.integers(0, 64, size=E)
    return torch.from_numpy(xy), torch.from_numpy(tgt), torch.from_numpy(newf), M, R


def _counts_from(c):
    c = c.to(torch.int32)
    return c[:, :-1, :-1] + c[:, 1:, :-1] + c[:, :-1, 1:] + c[:, 1:, 1:]


@pytest.mark.parametrize("mutant", ["le", "per_agent", "round_hit", "tile_last_row", "transposed"])
def test_classification_mistakes_break_exact_parts(mutant):
    xy, tgt, newf, M, R = _tie_geometry()
    s = map_ref.sense(xy, M, R, tgt, newf)
    sums = map_ref.corner_sums(xy, M)
    counts, found = s.counts.clone(), s.found.clone()
    if mutant == "le":
        counts = _counts_from((sums <= R * R).any(1))
    elif mutant == "per_agent":
        counts = sum(_counts_from(sums[:, a] < R * R) for a in range(xy.shape[1])).clamp(max=4)
    elif mutant == "round_hit":
        E, m = tgt.shape[:2]
        ci = torch.round(tgt[:, :, 0]).clamp(max=M - 1).long()
        cj = torch.round(tgt[:, :, 1]).clamp(max=M - 1).long()
        bits = (newf.view(E, 1) >> torch.arange(m).view(1, m)) & 1
        ok = (bits != 0) & (ci >= 0) & (cj >= 0)
        found = torch.zeros(E, M * M, dtype=torch.bool)
        found[torch.arange(E).view(E, 1).expand(E, m)[ok], (ci * M + cj)[ok]] = True
        found = found.view(E, M, M)
    elif mutant == "tile_last_row":
        c = s.corners.to(torch.int32)
        lower = c[:, 1:].clone()
        lower[:, 3::4] = c[:, 3:-1:4]                                  # cell row 4k+3 reads corner row i, not i+1
        counts = c[:, :-1, :-1] + lower[:, :, :-1] + c[:, :-1, 1:] + lower[:, :, 1:]
    elif mutant == "transposed":
        counts = s.counts.transpose(1, 2).contiguous()
    rng = np.random.default_rng(2)
    E = xy.shape[0]
    p = (rng.uniform(0, 1, size=(E, M, M)) ** 2).astype(np.float32)
    p[rng.uniform(size=p.shape) < 0.05] = 1.0
    d = 0.9
    good = belief_emul(p, s.counts.numpy(), s.found.numpy(), d)
    bad = belief_emul(p, counts.numpy(), found.numpy(), d)
    assert not (torch.equal(counts, s.counts) and torch.equal(found, s.found)), "mistake invisible on these inputs"
    total, _, _ = _judge(bad.ravel(), p.ravel(), s.counts.numpy().ravel(), s.found.numpy().ravel(), d)
    changed = torch.from_numpy((good.view(np.uint32) != bad.view(np.uint32)).ravel())
    _report(mutant, total, changed)
    assert bool((total[changed] > 1).all()) and bool(changed.any())


def test_le_mistake_needs_ties():
    """`<=` instead of `<` only differs where a corner lies exactly at R^2: on the tie geometry it does, on random
    non-integer positions it does not -- why the GPU tests place agents on such points on purpose"""
    xy, _, _, M, R = _tie_geometry()
    sums = map_ref.corner_sums(xy, M)
    assert bool(((sums == R * R).any(1)).any())
    rnd = torch.from_numpy(np.random.default_rng(1).uniform(0, M, size=(48, 3, 2)))
    s2 = map_ref.corner_sums(rnd, M)
    assert not bool((s2 == R * R).any())


def test_pow_recheck_counts_disagreements():
    """pow(v, 2.0) and v * v differ in the last bit for some v; a corner whose sum lies within a few ulp of R^2 can then
    be classified differently.  sense() finds every such candidate and counts the disagreements."""
    R = 7
    rng = np.random.default_rng(4)
    # agents placed so that (cx-ax)^2 + (cy-ay)^2 is within an ulp or two of 49 for corner (10, 10): ax = 10 - sqrt(49 - 0.25)
    base = 10.0 - math.sqrt(49.0 - 0.25)
    offs = (np.arange(-200, 200) * 2.0 ** -49)
    xy = np.zeros((offs.size, 1, 2))
    xy[:, 0, 0] = base + offs
    xy[:, 0, 1] = 9.5
    s = map_ref.sense(torch.from_numpy(xy), 20, R)
    assert s.pow_checked > 0
    # brute force: every (env, corner) classified both ways
    diff = 0
    for e in range(xy.shape[0]):
        ax, ay = xy[e, 0]
        for cx in range(21):
            for cy in range(21):
                a = math.pow(cx - ax, 2.0) + math.pow(cy - ay, 2.0) < 49
                b = (cx - ax) * (cx - ax) + (cy - ay) * (cy - ay) < 49
                diff += a != b
    assert s.pow_diff == diff
    print("pow/mul disagreements near R^2: %d of %d candidates" % (s.pow_diff, s.pow_checked))
