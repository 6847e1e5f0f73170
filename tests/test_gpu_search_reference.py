"""search_env kernel (csrc/search.cu) against the C oracle on the path the c5 benchmark runs: auto-reset, the in-kernel
policy, full episodes and the resets after them, and the episode statistics.

Every step's float32 reward r must lie in [fl32(X - B), fl32(X + B)], X the exact sum of the oracle's reward terms and
B = (n+1) 2^-53 sum|terms| (oracle/search_check.py); every other output is compared exactly.  Each test prints the
largest |r - X| / (B + ulp(r)/2), how many compared envs went through an auto-reset, and the statistics it compared."""
import math
import os
import types

import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import search_check as sc
from oracle.py_envs import SearchSpec

pytestmark = pytest.mark.gpu
c_oracle.set_threads(min(16, os.cpu_count() or 1))

INT_STATS = ("episodes", "targets_found_sum", "wins", "episode_len_sum", "env_steps", "illegal_moves")


def cpu(t):
    return t.detach().cpu().numpy()


def make_args(n, m, M, R, am, tm):
    return types.SimpleNamespace(env="search", map_size=M, target_num=m, target_mode=tm, target_dir="./targets/",
                                 agent_mode=am, n_agents=n, view_range=R)


class SliceCheck:
    """Rows [lo, lo + E) of a device handle against a C oracle built at the same global ids (auto_reset=True), compared
    after every step; the views, freq and bit rows every `every` steps and on the step of and after each auto-reset.
    Accumulates the statistics the oracle's episodes imply.  `orc`: an oracle already reset to the device rows' state."""

    def __init__(self, env, spec, seed, lo, E, every=50, orc=None):
        self.env, self.lo, self.E, self.M, self.n, self.every = env, lo, E, spec.map_size, spec.n_agents, every
        self.sl = slice(lo, lo + E)
        if orc is None:
            orc = c_oracle.SearchBatch(spec, seed, env.env_id_base + lo, E, auto_reset=True)
            orc.reset()
        self.orc = orc
        self.ratio = 0.0
        self.reset_seen = np.zeros(E, bool)
        self.prev_reset = np.zeros(E, bool)
        self.steps = 0
        self.st = dict.fromkeys(INT_STATS, 0)
        self.ep_X = np.zeros(E, np.longdouble)        # exact running episode reward
        self.tot_X = np.longdouble(0)
        self.tot_B = 0.0                              # sum of the per-step bounds of finished episodes
        self.ep_B = np.zeros(E)
        self.run_abs = 0.0                            # sum over steps of |running episode sum| (fp64 accumulation)
        self.ep_abs = 0.0                             # sum over episodes of |episode sum| (atomicAdd order)
        self.compare_views("after reset")

    def compare_views(self, where, envs=None):
        env, orc = self.env, self.orc
        obs, state, avail = orc.views(envs=envs)
        if envs is None:
            pick = lambda t: cpu(t[self.sl])
            rows = slice(None)
        else:
            idx = torch.as_tensor(self.lo + envs, device=env.device)
            pick = lambda t: cpu(t.index_select(0, idx))
            rows = envs
        assert np.array_equal(pick(env.get_obs()), obs), where + ": obs"
        assert np.array_equal(pick(env.get_state()), state), where + ": state"
        assert np.array_equal(pick(env.get_avail_actions()), avail), where + ": avail"
        assert np.array_equal(pick(env.freq_map), orc.freq[rows]), where + ": freq"
        assert np.array_equal(sc.dense_bits(pick(env.target_bits), self.M), orc.tmap[rows]), where + ": target_bits"
        assert np.array_equal(sc.dense_bits(pick(env.unfound_bits), self.M), orc.unfound_map()[rows]), where + ": unfound_bits"

    def step(self, t):
        """Steps the oracle once and compares with the device rows (the device has already stepped)."""
        env, orc, sl = self.env, self.orc, self.sl
        where = "rows %d.. step %d" % (self.lo, t)
        time_before = orc.counters[:, 1].copy()
        orc.step(None)
        self.steps += 1
        r = cpu(env._reward[sl])
        ok = sc.reward_ok(r, orc.terms)
        if not ok.all():
            e = int(np.nonzero(~ok)[0][0])
            lo, hi, X, B = sc.reward_interval(orc.terms[e:e + 1])
            raise AssertionError("%s env %d: reward %r outside [%r, %r] (exact %r, B %.3g)" % (where, self.lo + e, float(r[e]),
                                 float(lo[0]), float(hi[0]), float(X[0]), B[0]))
        self.ratio = max(self.ratio, sc.reward_error_ratio(r, orc.terms))
        term = cpu(env._terminated[sl])
        assert np.array_equal(term, orc.terminated), where + ": terminated"
        assert np.array_equal(cpu(env.target_find[sl]), orc.target_find), where + ": target_find"
        assert np.array_equal(cpu(env.agent_pos[sl]), orc.pos), where + ": positions"
        assert np.array_equal(cpu(env.counters[sl]), orc.counters), where + ": counters"
        assert not (orc.counters[:, 2] & 2).any(), where + ": the in-kernel policy moves legally"
        done = term.astype(bool)
        # statistics of the finished episodes, from the oracle
        _, _, X, B = sc.reward_interval(orc.terms)
        self.ep_X += X
        self.ep_B += B
        self.run_abs += float(np.abs(self.ep_X).sum())
        k = int(done.sum())
        self.st["episodes"] += k
        self.st["wins"] += k
        self.st["targets_found_sum"] += int(orc.target_find[done].sum())
        self.st["episode_len_sum"] += int((time_before[done] + 1).sum())
        self.tot_X += self.ep_X[done].sum()
        self.tot_B += float(self.ep_B[done].sum())
        self.ep_abs += float(np.abs(self.ep_X[done]).sum())
        self.ep_X[done] = 0
        self.ep_B[done] = 0
        self.reset_seen |= done
        if t % self.every == 0:
            self.compare_views(where)
        else:
            rows = np.nonzero(done | self.prev_reset)[0]
            if rows.size:
                self.compare_views(where + " (auto-reset rows)", rows)
        self.prev_reset = done

    def expected_stats(self):
        st = dict(self.st)
        st["env_steps"] = self.E * self.steps
        return st

    def reward_sum_tolerance(self):
        """Per-step bounds of the finished episodes, plus the float64 rounding of the running episode sums and of the
        atomic adds of the episode sums in any order (first-order bounds, doubled for the second-order terms)."""
        return self.tot_B + 2 * 2.0 ** -53 * (self.run_abs + self.st["episodes"] * self.ep_abs)


class DeviceStats:
    """The statistics as the device's own per-step outputs imply them, for a whole handle (on the GPU)."""

    def __init__(self, env):
        E, dev = env.num_envs, env.device
        self.env = env
        self.run = torch.zeros(E, dtype=torch.float64, device=dev)        # fp32 rewards of the running episode, summed
        self.half_ulp = torch.zeros(E, dtype=torch.float64, device=dev)
        self.len = torch.zeros(E, dtype=torch.int64, device=dev)
        self.acc = torch.zeros(6, dtype=torch.float64, device=dev)        # episodes, found, len, reward, ulps, |running|
        self.steps = 0

    def step(self):
        env = self.env
        r = env._reward
        term = env._terminated.to(torch.bool)
        self.steps += 1
        self.run += r.double()
        self.half_ulp += (torch.nextafter(r.abs(), torch.tensor(math.inf, device=r.device)) - r.abs()).double() / 2
        self.len += 1
        tf = term.double()
        self.acc += torch.stack([tf.sum(), (env.target_find.double() * tf).sum(), (self.len.double() * tf).sum(),
                                 (self.run * tf).sum(), (self.half_ulp * tf).sum(), self.run.abs().sum()])
        keep = (~term).double()
        self.run *= keep
        self.half_ulp *= keep
        self.len *= (~term).long()

    def check(self, st, what):
        eps, found, length, rsum, ulps, run_abs = cpu(self.acc).tolist()
        E = self.env.num_envs
        want = dict(episodes=eps, wins=eps, targets_found_sum=found, episode_len_sum=length, env_steps=E * self.steps,
                    illegal_moves=0)
        for k in INT_STATS:
            assert st[k] == want[k], "%s: %s %r, the device outputs say %r" % (what, k, st[k], want[k])
        tol = ulps + 4 * 2.0 ** -53 * (run_abs + eps * abs(rsum))
        assert abs(st["episode_reward_sum"] - rsum) <= tol, "%s: episode_reward_sum %r, fp32 outputs sum to %r (tol %.3g)" % (
            what, st["episode_reward_sum"], rsum, tol)
        return rsum, tol


def assert_oracle_stats(st, checks, what):
    want = dict.fromkeys(INT_STATS, 0)
    X, tol = np.longdouble(0), 0.0
    for c in checks:
        for k, v in c.expected_stats().items():
            want[k] += v
        X += c.tot_X
        tol += c.reward_sum_tolerance()
    for k in INT_STATS:
        assert st[k] == want[k], "%s: %s %r, oracle %r" % (what, k, st[k], want[k])
    err = abs(np.longdouble(st["episode_reward_sum"]) - X)
    assert err <= tol, "%s: episode_reward_sum %r, oracle %r (tol %.3g)" % (what, st["episode_reward_sum"], float(X), tol)
    return float(X), float(err), tol


C5_STEPS_K = 20             # steps per graph replay of the graph-stepped handle
C5_REPLAYS = 125            # 1 eager step + 125 x 20 replayed steps = 2501 steps


def test_c5_as_benchmarked():
    """(a) c5 as bench.py creates it -- 131072 envs, seed 42, env ids from 0, auto_reset=True, the in-kernel policy --
    against the oracle on three 256-env slices for 2501 steps, whole-handle statistics against the device's own outputs;
    (b) a second handle stepped as bench.py steps it (one eager step, then K-step CUDA graph replays) equals it bit for
    bit in every buffer after every replay, with equal integer-valued statistics."""
    import coopsearch_b200 as cs
    E, seed = 131072, 42
    spec = SearchSpec(n_agents=64, target_num=1000, map_size=64, view_range=7, agent_mode=0, target_mode=0)
    args = make_args(64, 1000, 64, 7, 0, 0)
    a = cs.VecSearchEnv(args, num_envs=E, seed=seed, env_id_base=0, auto_reset=True)
    b = cs.VecSearchEnv(args, num_envs=E, seed=seed, env_id_base=0, auto_reset=True)
    slices = [SliceCheck(a, spec, seed, lo, 256) for lo in (0, 65536, E - 256)]
    dstat = DeviceStats(a)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        b.step_random(1)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(C5_STEPS_K):
                b.step_random(1)
    names = ("agent_pos", "target_bits", "unfound_bits", "freq_map", "counters", "_obs", "_state", "_avail", "_reward",
             "_terminated", "_target_find")

    def same_buffers(t):
        torch.cuda.synchronize()
        for nm in names:
            assert torch.equal(getattr(a, nm), getattr(b, nm)), "graph-stepped handle differs in %s after step %d" % (nm, t)

    t = 0
    for rep in range(C5_REPLAYS + 1):
        if rep > 0:
            with torch.cuda.stream(side):
                graph.replay()
        for _ in range(1 if rep == 0 else C5_STEPS_K):
            t += 1
            a.step_random(1)
            dstat.step()
            for c in slices:
                c.step(t)
        same_buffers(t)
    st_a, st_b = a.stats(), b.stats()
    rsum, tol = dstat.check(st_a, "c5 eager")
    dstat.check(st_b, "c5 graph")
    for k in INT_STATS:
        assert st_a[k] == st_b[k], k
    ratio = max(c.ratio for c in slices)
    reset = int(sum(c.reset_seen.sum() for c in slices))
    print("\nc5 %d steps: max |r-X|/(B+ulp/2) = %.3f; slice envs auto-reset %d / %d; stats %s; reward sum %.6f vs fp32 "
          "outputs %.6f (tol %.3g); graph handle equal" % (t, ratio, reset, 3 * 256,
                                                           {k: st_a[k] for k in INT_STATS}, st_a["episode_reward_sum"], rsum, tol))
    assert ratio <= 1.001
    assert reset >= 0.9 * 3 * 256
    assert st_a["episodes"] > 0 and st_a["episode_reward_sum"] != 0.0


GRID = [  # n, m, M, R, agent_mode, target_mode, envs, steps
    (1, 1, 2, 1, 0, 0, 1024, 300),            # smallest map; an episode nearly every step
    (4, 55, 8, 2, 1, 1, 1024, 400),           # target_mode 1 with the edge band full
    (3, 5, 8, 16, 0, 0, 512, 300),            # R > M
    (127, 10, 31, 1, 0, 0, 512, 400),
    (128, 20, 32, 17, 2, 0, 512, 400),        # agent_mode 2, n > M: gap 0, all agents start on one cell; S = 33 > 32
    (129, 30, 33, 4, 0, 1, 512, 400),
    (64, 10, 63, 17, 0, 0, 512, 500),         # odd M: two-float state stores
    (1000, 50, 64, 7, 0, 0, 256, 400),        # observation block too large for shared memory: direct path
    (64, 8, 65, 16, 0, 0, 512, 500),          # M > 64: three words per bit row, direct observation path
    (3, 5, 97, 64, 0, 0, 128, 300),           # most envs reset every step: every view compared every step
]


@pytest.mark.parametrize("n,m,M,R,am,tm,E,T", GRID)
def test_search_grid_auto_reset_and_stats(n, m, M, R, am, tm, E, T):
    """(c) Every step of E envs against the oracle with auto-reset, then the handle's statistics against the oracle's."""
    import coopsearch_b200 as cs
    seed, base = 5, 7000
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R, agent_mode=am, target_mode=tm)
    env = cs.VecSearchEnv(make_args(n, m, M, R, am, tm), num_envs=E, seed=seed, env_id_base=base, auto_reset=True)
    chk = SliceCheck(env, spec, seed, 0, E)
    for t in range(1, T + 1):
        env.step_random(1)
        chk.step(t)
    st = env.stats()
    X, err, tol = assert_oracle_stats(st, [chk], "grid %s" % ((n, m, M, R, am, tm),))
    print("\ngrid %s: max |r-X|/(B+ulp/2) = %.3f; envs auto-reset %d / %d; stats %s; reward sum %.9g, oracle %.9g, |diff| %.3g "
          "<= %.3g" % ((n, m, M, R, am, tm), chk.ratio, int(chk.reset_seen.sum()), E, {k: st[k] for k in INT_STATS},
                       st["episode_reward_sum"], X, err, tol))
    assert chk.ratio <= 1.001
    assert chk.reset_seen.sum() >= 0.9 * E


def test_episode_counter_wraps_16_bits():
    """(d) The episode counter crosses 65535 -> 65536 (the Philox counter keeps its low 16 bits, the key the rest):
    device and oracle agree through two auto-resets, and episode 65536 is not a replay of episode 0."""
    import coopsearch_b200 as cs
    n, m, M, R, E, seed, base = 4, 3, 8, 2, 64, 9, 500
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R)
    env = cs.VecSearchEnv(make_args(n, m, M, R, 0, 0), num_envs=E, seed=seed, env_id_base=base, auto_reset=True, reset=False)
    env.counters[:, 3] = 65534                     # the next reset opens episode 65535
    env.reset()
    orc = c_oracle.SearchBatch(spec, seed, base, E, auto_reset=True)
    orc.counters[:, 3] = 65534
    orc.reset()
    chk = SliceCheck(env, spec, seed, 0, E, every=1, orc=orc)
    first = c_oracle.SearchBatch(spec, seed, base, E)
    first.reset()
    layout_65536 = np.zeros((E, M, M), np.uint8)
    got = np.zeros(E, bool)
    t = 0
    while (orc.counters[:, 3] < 65537).any():
        t += 1
        assert t <= 3000, "episodes did not end"
        env.step_random(1)
        chk.step(t)
        new = (orc.counters[:, 3] == 65536) & ~got
        layout_65536[new] = orc.tmap[new]
        got |= new
    assert got.all()
    same = [(layout_65536[e] == first.tmap[e]).all() for e in range(E)]
    print("\nepisode wrap: %d steps to episode 65537 in all %d envs; max |r-X|/(B+ulp/2) = %.3f; episode 65536 equals "
          "episode 0 in %d envs" % (t, E, chk.ratio, sum(same)))
    assert not any(same)
    assert chk.ratio <= 1.001


def test_placement_full_grid_at_512():
    """(e) M = 512 with every cell a target: exactly M^2 bits per env, as the oracle places them."""
    import coopsearch_b200 as cs
    M, E = 512, 2
    spec = SearchSpec(n_agents=1, target_num=M * M, map_size=M, view_range=1)
    env = cs.VecSearchEnv(make_args(1, M * M, M, 1, 0, 0), num_envs=E, seed=0, env_id_base=0)
    orc = c_oracle.SearchBatch(spec, 0, 0, E)
    orc.reset()
    dense = sc.dense_bits(cpu(env.target_bits), M)
    missing = [int(M * M - dense[e].sum()) for e in range(E)]
    print("\nM=512 full grid: targets missing per env %s" % missing)
    assert missing == [0] * E
    assert np.array_equal(dense, orc.tmap)
    assert np.array_equal(sc.dense_bits(cpu(env.unfound_bits), M), orc.tmap)


def test_placement_band_full_and_refused():
    """(e) target_mode 1 at M = 8: the 55 band cells are placed exactly as the oracle places them; 56 is refused."""
    import coopsearch_b200 as cs
    M, E = 8, 64
    assert sc.band_cells(M) == 55
    spec = SearchSpec(n_agents=4, target_num=55, map_size=M, view_range=2, agent_mode=1, target_mode=1)
    env = cs.VecSearchEnv(make_args(4, 55, M, 2, 1, 1), num_envs=E, seed=3, env_id_base=11)
    orc = c_oracle.SearchBatch(spec, 3, 11, E)
    orc.reset()
    dense = sc.dense_bits(cpu(env.target_bits), M)
    assert (dense.sum((1, 2)) == 55).all()
    assert np.array_equal(dense, orc.tmap)
    with pytest.raises(cs.CoopSearchError, match="edge band"):
        cs.VecSearchEnv(make_args(4, 56, M, 2, 1, 1), num_envs=E, seed=3)


def test_injected_cells_off_map_or_repeated_are_refused(tmp_path):
    """(e) reset(cells=...) and the target_mode 3 file refuse cells off the map and cells listed twice."""
    import coopsearch_b200 as cs
    M, m, E = 10, 3, 2
    env = cs.VecSearchEnv(make_args(2, m, M, 2, 0, 0), num_envs=E, seed=1)
    good = np.array([[[0, 0], [9, 9], [4, 5]], [[1, 2], [2, 1], [3, 3]]], np.int32)
    env.reset(cells=good)
    assert int(env.target_find.sum()) == 0
    for bad, msg in ((10, "off the"), (-1, "off the")):
        c = good.copy()
        c[1, 2, 1] = bad
        with pytest.raises(cs.CoopSearchError, match=msg):
            env.reset(cells=c)
        with pytest.raises(cs.CoopSearchError, match=msg):
            env.reset(cells=torch.as_tensor(c, device=env.device))
    dup = good.copy()
    dup[0, 2] = dup[0, 0]
    with pytest.raises(cs.CoopSearchError, match="more than once"):
        env.reset(cells=dup)
    f = tmp_path / "targets.txt"
    f.write_text("1 1\n2 2\n1 1\n")
    with pytest.raises(cs.CoopSearchError, match="more than once"):
        cs.VecSearchEnv(make_args(2, m, M, 2, 0, 3), targets_filename=str(f), num_envs=E)
    f.write_text("1 1\n2 2\n3 10\n")
    with pytest.raises(cs.CoopSearchError, match="off the"):
        cs.VecSearchEnv(make_args(2, m, M, 2, 0, 3), targets_filename=str(f), num_envs=E)
    f.write_text("1 1\n2 2\n3 9\n")
    ok = cs.VecSearchEnv(make_args(2, m, M, 2, 0, 3), targets_filename=str(f), num_envs=E)
    assert (sc.dense_bits(cpu(ok.target_bits), M).sum((1, 2)) == m).all()
