"""search_env C oracle (oracle/coopsearch_oracle.c) against the Python restatement (oracle/py_envs.SearchOracle), over
several episodes with auto-reset, and the exact float32 reward criterion the GPU tests apply (oracle/search_check.py).
CPU only."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import c_oracle
from oracle import search_check as sc
from oracle.py_envs import SearchOracle, SearchSpec


def legal_actions(rng, pos, M):
    """Uniform legal moves [E, n] for positions [E, n, 2]."""
    x, y = pos[..., 0], pos[..., 1]
    av = np.stack([x > 0, y > 0, x < M - 1, y < M - 1], -1)
    u = rng.random(av.shape) * av
    return np.argmax(u, -1).astype(np.uint8)


@pytest.mark.parametrize("n,m,M,R,am,tm,steps", [(3, 4, 10, 3, 0, 0, 400), (5, 4, 12, 2, 2, 1, 600)])
def test_c_oracle_auto_reset_matches_python_oracle(n, m, M, R, am, tm, steps):
    """SearchBatch(auto_reset=True) equals SearchOracle driven with reset() at every termination, every step."""
    E, seed, base = 6, 11, 300
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R, agent_mode=am, target_mode=tm)
    b = c_oracle.SearchBatch(spec, seed, base, E, auto_reset=True)
    b.reset()
    py = [SearchOracle(spec, seed, base + e) for e in range(E)]
    for o in py:
        o.reset()
    rng = np.random.default_rng(5)
    episodes = np.zeros(E, int)
    for t in range(steps):
        act = legal_actions(rng, b.pos, M)
        r, term = b.step(act)
        obs, state, avail = b.views()
        for e, o in enumerate(py):
            where = "env %d step %d" % (e, t)
            pr, pterm, _ = o.step(act[e])
            assert r[e] == pr, where                                   # same float64 summation order
            assert bool(term[e]) == pterm, where
            assert b.target_find[e] == o.target_find, where
            assert math.fsum(b.terms[e]) == pytest.approx(pr, rel=0, abs=1e-12), where
            if pterm:
                o.reset()
                episodes[e] += 1
            assert np.array_equal(b.pos[e], np.array(o.pos)), where
            assert np.array_equal(b.freq[e], o.freq.astype(np.int32)), where
            assert b.counters[e, 0] == o.target_find and b.counters[e, 1] == o.time_step, where
            assert b.counters[e, 3] == o.episode, where
            assert np.array_equal(obs[e], o.get_obs().astype(np.float32)), where
            assert np.array_equal(state[e], o.get_state().astype(np.float32)), where
            assert np.array_equal(avail[e], np.array([o.get_avail_agent_actions(i) for i in range(n)]).astype(np.uint8)), where
    print("episodes per env", episodes.tolist())
    assert episodes.min() >= 3


def test_reward_terms_sum_to_oracle_reward():
    """The exported terms are the oracle's reward: the oracle's own float64 sum lies inside the exact interval."""
    spec = SearchSpec(n_agents=12, target_num=30, map_size=8, view_range=1, agent_mode=2, target_mode=0)
    b = c_oracle.SearchBatch(spec, 3, 0, 16, auto_reset=True)
    b.reset()
    for _ in range(300):
        r, _ = b.step(None)
        _, _, X, B = sc.reward_interval(b.terms)
        assert np.all(np.abs(r - X.astype(np.float64)) <= B)
        assert np.all(b.terms[:, 0] == -1)


def test_band_count_matches_brute_force():
    for M in range(2, 71):
        x, y = np.meshgrid(np.arange(M), np.arange(M), indexing="ij")
        lo, hi = M // 4, 3 * M // 4
        assert sc.band_cells(M) == int(((x <= lo) | (x >= hi) | (y <= lo) | (y >= hi)).sum()), M


def test_create_refuses_target_mode_1_beyond_the_band():
    """cs_search_create accepts target_num up to the band count and refuses one more, before any CUDA call."""
    import coopsearch_b200 as cs
    from coopsearch_b200 import _lib
    lib = cs.load_library()
    for M in range(2, 71):
        band = sc.band_cells(M)
        cfg = _lib.SearchCfg(struct_size=C.sizeof(_lib.SearchCfg), num_envs=1, n_agents=1, target_num=band + 1, map_size=M,
                             view_range=1, agent_mode=0, target_mode=1)
        h = C.c_void_p()
        assert lib.cs_search_create(C.byref(cfg), C.byref(h)) == -1, M
        assert (b"edge band" if band < M * M else b"fit the grid") in lib.cs_last_error(), M
        cfg.target_num = band
        rc = lib.cs_search_create(C.byref(cfg), C.byref(h))
        assert b"edge band" not in lib.cs_last_error() or rc == 0, M
        if rc == 0:
            lib.cs_search_destroy(h)


def _stacked_run(steps=400):
    """12 agents stacked on one cell of an 8x8 map (agent_mode 2, gap 0), R = 1, 30 targets, auto-reset: agents share cells,
    see the same new target together, and every episode restarts them on the stacked cell, so freq climbs past 100.  Per
    step: which rows kept their episode (their positions are the step's), terms, positions, and how many agents sighted a
    target that was new at that step."""
    n, m, M, R = 12, 30, 8, 1
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R, agent_mode=2, target_mode=0)
    E = 8
    b = c_oracle.SearchBatch(spec, 21, 0, E, auto_reset=True)
    b.reset()
    out = []
    for _ in range(steps):
        found_before = b.found.copy()
        _, term = b.step(None)
        live = term == 0
        pos = b.pos.copy()
        d = ((b.cells[:, None, :, :] - pos[:, :, None, :]) ** 2).sum(-1) <= R * R         # [E, n, m] agent sees target
        sightings = (d & (found_before[:, None, :] == 0)).sum((1, 2))
        out.append((live, b.terms.copy(), pos, sightings))
    return n, out


def test_reward_criterion_accepts_kernel_order_and_rejects_mistakes():
    n, run = _stacked_run()
    accepted = rej_stack = diff_stack = rej_off = diff_off = rej_sight = diff_sight = 0
    for live, terms, pos, sightings in run:
        # the kernel's own summation order is accepted
        assert np.all(sc.reward_ok(sc.kernel_order_reward(terms), terms))
        accepted += terms.shape[0]
        f = np.rint(1.0 / terms[:, 1:n + 1]).astype(np.int64)
        # (2) one freq off by one where 100 <= f <= 300
        for a in range(n):
            sel = (f[:, a] >= 100) & (f[:, a] <= 300)
            if sel.any():
                bad = terms[sel].copy()
                bad[:, 1 + a] = 1.0 / (f[sel, a] + 1)
                diff_off += int(sel.sum())
                rej_off += int((~sc.reward_ok(sc.kernel_order_reward(bad), terms[sel])).sum())
        terms, pos, sightings, f = terms[live], pos[live], sightings[live], f[live]
        # (1) agent 0's freq read before agents 1..n-1 moved: those that landed on its cell are not counted yet
        later = (pos[:, 1:, :] == pos[:, :1, :]).all(-1).sum(1)
        bad = terms.copy()
        bad[:, 1] = 1.0 / (f[:, 0] - later)
        d = later > 0
        diff_stack += int(d.sum())
        rej_stack += int((~sc.reward_ok(sc.kernel_order_reward(bad), terms))[d].sum())
        # (3) +10 per agent sighting instead of per target
        bad = terms.copy()
        bad[:, n + 1] = 10.0 * sightings
        d = bad[:, n + 1] != terms[:, n + 1]
        diff_sight += int(d.sum())
        rej_sight += int((~sc.reward_ok(sc.kernel_order_reward(bad), terms))[d].sum())
    print("accepted %d kernel-order rewards; rejected: stale freq %d/%d, off-by-one freq %d/%d, per-sighting bonus %d/%d"
          % (accepted, rej_stack, diff_stack, rej_off, diff_off, rej_sight, diff_sight))
    assert diff_stack > 100 and diff_off > 100 and diff_sight > 10
    assert rej_stack == diff_stack and rej_off == diff_off and rej_sight == diff_sight
