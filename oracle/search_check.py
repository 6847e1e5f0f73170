"""Exact checks of the search_env step reward -- TEST INFRASTRUCTURE.

The kernel sums the reward's terms (-1, 1/freq of every agent, 10 * targets found) in float64 in its own order (per-thread
partial sums, a warp butterfly, then the warps) and rounds the result once to float32.  Any float64 summation order of
k terms lies within (k-1) * 2^-53 * sum|terms| of the exact sum X, so with B = (n+1) * 2^-53 * sum|terms| the float32
reward r must satisfy fl32(X - B) <= r <= fl32(X + B).  That interval is one or two float32 values wide: a wrong freq
(1/149 vs 1/150 moves the reward by 4.5e-5, ~50 ulps at 10) or a target counted twice cannot pass it."""
import math

import numpy as np

_LONG = np.finfo(np.longdouble).nmant >= 63          # x87 extended: the row sums below are exact to far below B


def exact_sums(terms):
    """[..., k] float64 terms -> the exact sums as long double (fsum when long double is plain double)."""
    t = np.asarray(terms, np.float64)
    if _LONG:
        return t.astype(np.longdouble).sum(-1)
    flat = t.reshape(-1, t.shape[-1])
    return np.array([math.fsum(row) for row in flat], np.float64).reshape(t.shape[:-1])


def reward_interval(terms):
    """(lo, hi, X, B): the float32 interval [fl32(X - B), fl32(X + B)] the kernel's reward of each row must lie in."""
    t = np.asarray(terms, np.float64)
    X = exact_sums(t)
    B = (t.shape[-1] - 1) * 2.0 ** -53 * np.abs(t).sum(-1)
    lo = (X - B).astype(np.float32)
    hi = (X + B).astype(np.float32)
    return lo, hi, X, B


def reward_ok(r, terms):
    """Boolean per row: r inside the interval."""
    lo, hi, _, _ = reward_interval(terms)
    r = np.asarray(r, np.float32)
    return (lo <= r) & (r <= hi)


def reward_error_ratio(r, terms):
    """max |r - X| / (B + ulp(r)/2) over the rows (<= 1 for every accepted reward)."""
    _, _, X, B = reward_interval(terms)
    r = np.asarray(r, np.float32)
    half_ulp = np.spacing(np.abs(r)).astype(np.float64) / 2
    if r.size == 0:
        return 0.0
    return float(np.max(np.abs(r.astype(np.longdouble if _LONG else np.float64) - X) / (B + half_ulp)))


def kernel_order_reward(terms, threads=128):
    """The kernel's float64 summation order (csrc/search.cu, search_kernel<STEP>) of rows (-1, 1/f_0..1/f_{n-1}, 10*new),
    rounded to float32: agent a is added to thread a % threads in order, each warp reduces with an xor butterfly, thread 0
    adds the warp sums in order, then -1 and the find bonus."""
    t = np.asarray(terms, np.float64)
    rows, n = t.shape[0], t.shape[1] - 2
    part = np.zeros((rows, threads))
    for a in range(n):
        part[:, a % threads] += t[:, 1 + a]
    part = part.reshape(rows, threads // 32, 32)
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        part = part + part[:, :, lane ^ o]
    fsum = np.zeros(rows)
    for w in range(threads // 32):
        fsum = fsum + part[:, w, 0]
    return ((t[:, 0] + fsum) + t[:, n + 1]).astype(np.float32)


def band_cells(M):
    """Cells of the target_mode 1 edge band: x or y <= M//4 or >= 3M//4 (search_env.py:96-104)."""
    inner = max(0, 3 * M // 4 - M // 4 - 1)
    return M * M - inner * inner


def dense_bits(bits, M):
    """[E, M, W] int32 bit rows -> [E, M, M] uint8."""
    b = np.asarray(bits).astype(np.uint32)
    d = ((b[..., None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(b.shape[0], M, -1)[:, :, :M]
    return d.astype(np.uint8)
