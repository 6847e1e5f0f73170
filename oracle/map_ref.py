"""Float64 reference of one sensing call's belief-map update -- TEST INFRASTRUCTURE (oracle side).

The reference's _update_prob_map / _percent_in_agent_viewrange (env/flight_env.py:275-303) for a batch of envs, in
torch float64 on any device: the CPU for the committed fixtures, the GPU for the benchmark's 16 384 envs.  One call of
``sense`` + ``update`` is one sensing call of the kernels in csrc/flight_map.cuh: the map before the call, the agent
positions the kernel sensed from, and the cells of the targets that call found.

Exact parts.  A corner (cx, cy), cx, cy in 0..M, is in view of agent a when

    fl(fl((cx - ax)^2) + fl((cy - ay)^2)) < R^2

with both squares formed by multiplication, which is what every map kernel evaluates (the tiled form decides by an
fp32 interval first and re-evaluates this predicate exactly wherever an interval end lies within 1e-3 of an integer;
its result must equal the predicate).  A corner counts once however many agents see it (the reference's `break`).
The corner count of cell (i, j) is the number of its corners (i, j), (i+1, j), (i, j+1), (i+1, j+1) in view; the
cell is touched when that count is > 0.  Counts, touched set and touched count are exact: a kernel must match them
bit for bit.  The reference itself squares with Python's ``**`` (libm ``pow(v, 2.0)``), which differs from the
product in the last bit for ~0.08 % of arguments; a corner can only be classified differently when the sum lies
within a few ulp of R^2.  ``sense`` re-evaluates every such corner with ``math.pow`` on the CPU and returns the
number of (agent, corner) classifications on which the two forms disagree (``pow_diff``); ``square="pow"`` uses the
pow form for the result, which is what the committed fixtures were made with.

A found cell is [min(int(x), M-1), min(int(y), M-1)] of a target found by this call, int() truncating toward zero,
and a negative index never matches.  A found cell that is touched becomes exactly 1; an untouched one keeps its value.

Float64 update.  A touched, not found cell with value p becomes

    F = frac * q * p / (q * p + (1 - p)),   frac = count / 4,   q = 1 - d   (float64, as coopsearch_oracle.c)

and untouched cells keep their bits.  ``arith="reference"`` evaluates this in the reference's own operation order
(((frac * q) * p) / ((q * p) + (1 - p)), so a cell at p = 1 becomes fl(fl(frac q) / q), which need not be frac); it
reproduces the reference's float64 maps bit for bit.  ``arith="kernel"`` is what the kernels promise instead: a cell
at exactly p = 1 becomes exactly frac (for q > 0), because the map's derivative there is 1/q and any error of a
re-seeded cell would grow by that factor per call.

Error model of the kernels' fp32 evaluation (belief_f4 in flight_map.cuh, belief_cell in flight_common.cuh).  With
u = 2^-24, w = count / 4 and q = 1 - d carried as the fp32 pair qf = fl32(q), ql = fl32(q - qf), the kernel computes

    w    = 0.25 * count                   the 1024-entry table of build_cell_lut (flight_host.cu): exact
    lp   = fl(ql * p)                     mul.rn.f32x2; |ql| <= 2^-25 q, so its rounding is below u 2^-25 of q p
    qp   = fl(qf * p + lp)                fma.rn.f32x2                                                  (|e1| <= u)
    num  = fl(w * qp)                     mul.rn.f32x2: exact for w = 1/4, 1/2, 1, rounds once for 3/4  (|e2| <= u)
    om   = fl(1 - p)                      sub.rn.f32x2: exact for p >= 1/2, else |err| <= u (1 - p)    (e3)
    den  = fl(qp + om)                    add.rn.f32x2                                                  (|e4| <= u)
    r    = rcp.approx.ftz.f32(den)        1 ulp at most over the full range of inputs (PTX ISA, rcp):
                                          relative 2^-23                                                 (|e5| <= 2u)
    res  = fl(num * r + 0)                fma.rn.f32x2 with keep = 0 for a touched cell                 (|e6| <= u)

den carries qp e1 + om e3, at most u den because qp, om >= 0, so against F(qk), qk = qf + ql (the pair's value),

    res = F(qk) (1+e1)(1+e2)(1+e5)(1+e6) / ((1+e')(1+e4)),  |e'| <= u,  |res / F(qk) - 1| <= (1+u)^3 (1+2u) / (1-u)^2 - 1,

about 7u, plus 2^-48 for lp.  None of the ops flushes subnormals except rcp.approx.ftz, whose input den lies in
[min(q, 1), 1] for p in [0, 1] and never is subnormal.  A subnormal lp, qp, num or res carries an absolute error of at
most 2^-150 instead of a relative one; num and res are subnormal only when p is, so den ~ 1 and the term is
2^-150 (w + 1) / den + 2^-150 <= 2^-148 -- ``SUB`` terms below.

The pair's own error is a term of its own (``bound_q``): F depends on q through dlnF/dq = (1 - p) / (q den), so
evaluating it at qk instead of q moves it by F |qk - q| / q * (1 - p) / den to first order (|qk - q| <= 2^-48 q).
Unlike the rounding terms it has the same sign at every call; a cell that stays in view for N calls collects N of it.
With q rounded to fp32 alone, as the kernels did before, this term was |fl32(q) - q| / q, 1.5e-8 at d = 0.9 and
1.3e-8 at d = 0.05, which over the ~1700 calls a cell stays above 1e-37 at d = 0.05 is 2e-5: more than the rtol 1e-5
the maps are held to.  ``update`` also returns F(qk), against which the rounding terms alone can be measured.

d = 1 (q = 0): the kernels keep the bits of untouched cells and compute 0 * rcp(1 - p) = 0 for touched ones, and
0 * inf = NaN for a touched cell at p = 1 -- so does the reference (0 / 0).  Those NaNs are the only ones allowed.

``bound_ratio`` reports |got - want| / bound per cell and +inf wherever the comparison is not a finite, ordered one,
or where a cell that must be exact is not; a NaN counts as in bound only where the reference itself is NaN.
"""
import math

import torch

F64 = torch.float64
U = 2.0 ** -24                       # fp32 unit roundoff
RCP_APPROX = 2.0 ** -23              # rcp.approx.ftz.f32: 1 ulp at most over the full range (PTX ISA, "rcp")
REL = (1 + U) ** 3 * (1 + RCP_APPROX) / (1 - U) ** 2 - 1 + 2.0 ** -47    # + lp's rounding and float64 slack
SUB = 2.0 ** -150                    # half the spacing of fp32 subnormals
POW_WINDOW = 8                       # corners whose sum lies within this many ulp of R^2 are re-checked with math.pow


class Sensing:
    """Exact parts of one sensing call: corners [E, M+1, M+1] bool (in view of any agent), counts [E, M, M] int32,
    touched [E, M, M] bool, n_touched [E] int64, found [E, M, M] bool (cells of targets found by this call), and
    pow_diff / pow_checked: how many (agent, corner) classifications differ between pow and multiplication squares,
    and how many were close enough to R^2 to be checked."""

    def __init__(self, corners, found, pow_diff, pow_checked):
        self.corners = corners
        c = corners.to(torch.int32)
        self.counts = c[:, :-1, :-1] + c[:, 1:, :-1] + c[:, :-1, 1:] + c[:, 1:, 1:]
        self.touched = self.counts > 0
        self.n_touched = self.touched.flatten(1).sum(1)
        self.found = found
        self.pow_diff = pow_diff
        self.pow_checked = pow_checked

    @classmethod
    def from_counts(cls, counts, found):
        """A Sensing with given corner counts and found cells (no geometry): for checks of the update alone"""
        s = cls.__new__(cls)
        s.corners, s.counts, s.found = None, counts.to(torch.int32), found
        s.touched = s.counts > 0
        s.n_touched = s.touched.flatten(1).sum(1)
        s.pow_diff = s.pow_checked = 0
        return s


def corner_sums(xy, M):
    """fl(fl((cx-ax)^2) + fl((cy-ay)^2)) by multiplication: [E, n, M+1, M+1] float64 (xy: [E, n, 2] float64)"""
    c = torch.arange(M + 1, dtype=F64, device=xy.device)
    dx = c.view(1, 1, -1) - xy[:, :, 0:1]
    dy = c.view(1, 1, -1) - xy[:, :, 1:2]
    return (dx * dx).unsqueeze(3) + (dy * dy).unsqueeze(2)


def _pow_recheck(xy, M, R2, s):
    """(agent, corner) entries within POW_WINDOW ulp of R^2, classified again with libm pow(v, 2.0):
    returns (indices [k, 4], pow classification [k] bool, mul classification [k] bool)"""
    near = ((s - R2).abs() <= POW_WINDOW * math.ulp(R2)).nonzero()
    if near.numel() == 0:
        return near, None, None
    e, a, cx, cy = near.cpu().unbind(1)
    pts = xy[e.to(xy.device), a.to(xy.device)].cpu().tolist()
    pw = [math.pow(float(i) - p[0], 2.0) + math.pow(float(j) - p[1], 2.0) < R2
          for i, j, p in zip(cx.tolist(), cy.tolist(), pts)]
    pw = torch.tensor(pw, dtype=torch.bool)
    mul = (s[near.unbind(1)] < R2).cpu()
    return near, pw, mul


def found_cells(tgt, newf, M):
    """[E, M, M] bool: cells of the targets whose bit is set in newf [E] (targets found by this call).  tgt: [E, m, 2]
    float64.  Cell = [min(int(x), M-1), min(int(y), M-1)] with int() truncating toward zero; negative never matches."""
    E, m = tgt.shape[0], tgt.shape[1]
    dev = tgt.device
    bits = (newf.to(torch.int64).view(E, 1) >> torch.arange(m, device=dev).view(1, m)) & 1
    ci = torch.trunc(torch.clamp(tgt[:, :, 0], max=float(M))).clamp(max=M - 1).to(torch.int64)
    cj = torch.trunc(torch.clamp(tgt[:, :, 1], max=float(M))).clamp(max=M - 1).to(torch.int64)
    ok = (bits != 0) & (ci >= 0) & (cj >= 0)
    out = torch.zeros(E, M * M, dtype=torch.bool, device=dev)
    ee = torch.arange(E, device=dev).view(E, 1).expand(E, m)
    out[ee[ok], (ci * M + cj)[ok]] = True
    return out.view(E, M, M)


def sense(xy, M, R, tgt=None, newf=None, square="mul", chunk=4096):
    """Exact parts of one sensing call for every env.  xy: [E, n, 2] float64 positions the kernel sensed from;
    tgt [E, m, 2] float64 and newf [E] (bit j: target j found by this call) give the found cells (none if omitted).
    square: "mul" (the kernels) or "pow" (the reference's **)."""
    E, M, R2 = xy.shape[0], int(M), float(R) * float(R)
    corners, diff, checked = [], 0, 0
    for e0 in range(0, E, chunk):
        x = xy[e0:e0 + chunk]
        s = corner_sums(x, M)
        inside = s < R2
        near, pw, mul = _pow_recheck(x, M, R2, s)
        if pw is not None:
            checked += int(pw.numel())
            diff += int((pw != mul).sum())
            if square == "pow":
                inside[near.to(x.device).unbind(1)] = pw.to(x.device)
        corners.append(inside.any(1))
    corners = torch.cat(corners)
    if tgt is None:
        found = torch.zeros(E, M, M, dtype=torch.bool, device=xy.device)
    else:
        found = found_cells(tgt, newf, M)
    return Sensing(corners, found, diff, checked)


def q_pair(d):
    """(qf, ql): q = 1 - d (float64) as the kernels carry it, fp32 high part and fp32 remainder"""
    q = 1.0 - float(d)
    qf = float(torch.tensor(q, dtype=torch.float32))
    return qf, float(torch.tensor(q - qf, dtype=torch.float32))


def _F(frac, q, p):
    return frac * q * p / (q * p + (1 - p))


def update(p, s, d, arith="kernel", qk=None):
    """The map after the call, for the map p [E, M, M] before it (fp32 as the kernel exported it, or float64) and the
    Sensing s.  Returns a dict of [E, M, M] float64 tensors (``exact`` bool):
      want     the float64 update (q = 1 - d), found cells 1, untouched cells p, p = 1 -> frac (arith "kernel")
      want_qf  the same with q = qf + ql, the value the kernel's arithmetic approximates
      bound    the kernel's fp32 rounding terms (relative REL of want_qf + the subnormal absolute terms)
      bound_q  the term of the pair's error |F(qf + ql) - F(q)| (first order, 1 % slack); 0 where exact
      exact    cells whose value is exact: untouched, found and touched, and (arith "kernel", q > 0) p = 1"""
    p = p.to(F64)
    q = 1.0 - float(d)
    if qk is None:                   # the q the kernel's arithmetic evaluates with; default the fp32 pair's value
        qf, ql = q_pair(d)
        qk = qf + ql
    frac = s.counts.to(F64) / 4
    F = _F(frac, q, p)
    Fq = _F(frac, qk, p)
    den = qk * p + (1 - p)
    bound = REL * Fq.abs() + 2 * SUB * (frac + 1) / den + SUB
    if q > 0:
        bound_q = 1.01 * F.abs() * (abs(qk - q) / q) * (1 - p) / den
    else:
        bound_q = torch.zeros_like(p)
    ones = p == 1
    exact = ~s.touched | s.found
    if arith == "kernel" and q > 0:
        F = torch.where(ones, frac, F)
        Fq = torch.where(ones, frac, Fq)
        exact = exact | ones
    F = torch.where(s.found, torch.ones_like(F), F)
    Fq = torch.where(s.found, torch.ones_like(Fq), Fq)
    want = torch.where(s.touched, F, p)
    want_qf = torch.where(s.touched, Fq, p)
    zero = torch.zeros_like(p)
    return dict(want=want, want_qf=want_qf, bound=torch.where(exact, zero, bound),
                bound_q=torch.where(exact, zero, bound_q), exact=exact)


def bound_ratio(got, want, bound, exact=None):
    """|got - want| / bound per cell (float64), +inf wherever that is not a finite, ordered comparison, and for an
    exact cell 0 if got has want's value (NaN where want is NaN) else +inf.  got may be fp32."""
    got = got.to(F64)
    nan_ok = torch.isnan(want) & torch.isnan(got)
    err = (got - want).abs()
    r = torch.where(torch.isfinite(err) & torch.isfinite(bound), err / bound, torch.full_like(err, float("inf")))
    r = torch.nan_to_num(r, nan=float("inf"))
    r = torch.where((err == 0) & torch.isfinite(err), torch.zeros_like(r), r)     # exact agreement, bound 0 included
    if exact is not None:
        r = torch.where(exact & ~nan_ok & (err != 0), torch.full_like(r, float("inf")), r)
    return torch.where(nan_ok, torch.zeros_like(r), r)


def check_call(got, p_before, xy, M, R, d, tgt=None, newf=None, touched_delta=None, worst=None):
    """One sensing call judged against the reference: got / p_before [E, M, M] fp32 maps after / before the call as the
    kernel exported them, xy [E, n, 2] the positions it sensed from, tgt / newf its found targets.  Raises
    AssertionError on any violation; returns the Sensing and updates ``worst`` (dict) with the largest ratios:
    "total" against bound + bound_q, "rounding" against bound alone on F(qf), and the pow/mul disagreement count."""
    s = sense(xy, M, R, tgt, newf)
    u = update(p_before, s, d)
    r_tot = bound_ratio(got, u["want"], u["bound"] + u["bound_q"], u["exact"])
    r_rnd = bound_ratio(got, u["want_qf"], u["bound"], u["exact"])
    bad = ~(r_tot <= 1)
    if bool(bad.any()):
        e, i, j = [int(v) for v in bad.nonzero()[0]]
        raise AssertionError("map cell (%d, %d) of env %d: got %r, want %r (before %r, corners %d, found %d), bound %r + %r; "
                             "%d cells out of bound" % (i, j, e, float(got[e, i, j]), float(u["want"][e, i, j]),
                                                        float(p_before[e, i, j]), int(s.counts[e, i, j]), int(s.found[e, i, j]),
                                                        float(u["bound"][e, i, j]), float(u["bound_q"][e, i, j]), int(bad.sum())))
    if touched_delta is not None:
        want_t = int(s.n_touched.sum())
        assert touched_delta == want_t, "map_cells_touched grew by %d, reference %d" % (touched_delta, want_t)
    if worst is not None:
        worst["total"] = max(worst.get("total", 0.0), float(r_tot.max()) if r_tot.numel() else 0.0)
        worst["rounding"] = max(worst.get("rounding", 0.0), float(r_rnd[~u["exact"]].max()) if bool((~u["exact"]).any()) else 0.0)
        worst["pow_diff"] = worst.get("pow_diff", 0) + s.pow_diff
        worst["pow_checked"] = worst.get("pow_checked", 0) + s.pow_checked
        worst["calls"] = worst.get("calls", 0) + 1
    return s
