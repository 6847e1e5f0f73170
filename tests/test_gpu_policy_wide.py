"""The wide instantiations of both agent-network kernels (input widths 33..256: policy_kernel<S=8>, fp32, and
policy_tc_kernel<K1=256>, bf16 tensor cores) against the float64 reference of oracle/policy_ref.py, stage by stage and
on every row, each stage judged on the kernel's own input to it:
  (a) the hidden state against the reference's GRU step from the inputs the kernel read,
  (b) the action values against the reference's fc2 on the hidden state the kernel wrote,
  (c) the actions against the action rule on the kernel's own action values, exactly; for epsilon-greedy the rule
      includes the kernel's Philox draws (key (seed, 3), counter (row, t, 0, 0)).
Covers the widths around every 16- and 32-wide chunk edge up to 256, row counts around the tile and around where a
persistent CTA takes a second tile, c5's 8 388 608 rows at width 239, and the search loop
    obs, avail = env.get_obs(), env.get_avail_actions(); acts = agents.choose_actions(obs, avail=avail, ...)
    _, term, _ = env.step(acts); agents.init_hidden(mask=term)
under a captured CUDA graph with auto-reset.  The largest error / bound of each stage and precision is printed at the
end of the module."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from oracle import philox
from oracle import policy_ref as pr

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
PRECISIONS = ["fp32", "bf16"]
WORST = {}                        # (stage, precision[, "no flip"]) -> largest error / bound seen (pr.assert_within)
SMS = 148                         # CTAs of a persistent launch: one per SM for both wide instantiations


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for key, v in sorted(WORST.items()):
        print("wide policy reference: stage %s: largest |error| / bound %.3g" % (" ".join(key), v))


def make_agents(sd, E, n, obs_dim, A, last=True, reuse=True, precision="bf16", **kw):
    import coopsearch_b200 as cs
    return cs.BatchedRNNAgents(sd, num_envs=E, n_agents=n, obs_dim=obs_dim, n_actions=A, last_action=last, reuse_network=reuse,
                               device=DEV, precision=precision, **kw)


def action_rule(q, avail, epsilon, evaluate, seed, t):
    """policy_choose_action, mode 0 (agent/agent.py:66-75), on the kernel's q [R, A]: masked first maximum (action 0
    without an available action); unless evaluate, with probability epsilon (uu = (x >> 8) 2^-24 < fp32(epsilon) of
    Philox word x) the (y % n_avail)-th available action instead"""
    greedy = pr.greedy_rule(q, avail).cpu().numpy()
    if evaluate or epsilon <= 0:
        return greedy
    R, A = q.shape
    ok = np.ones((R, A), bool) if avail is None else avail.reshape(R, A).cpu().numpy() != 0
    x, y, _, _ = philox.philox4x32_np(np.arange(R, dtype=np.uint64), t, 0, 0, seed, philox.STREAM_POLICY)
    uu = (x >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
    nav = ok.sum(1)
    explore = (uu < float(np.float32(epsilon))) & (nav > 0)
    pick = (y % np.maximum(nav, 1).astype(np.uint64)).astype(np.int64)
    nth = ((np.cumsum(ok, 1) - 1) == pick[:, None]) & ok
    return np.where(explore, nth.argmax(1), greedy)


def call_checked(agents, ref, obs, avail=None, where="", epsilon=0.0, evaluate=True):
    """one choose_actions call, judged against the inputs it read"""
    h_in, last, t = agents.hidden.clone(), agents.actions.clone(), agents._t
    acts = agents.choose_actions(obs, avail=avail, epsilon=epsilon, evaluate=evaluate)
    judge(agents, ref, obs, avail, h_in, last, t, epsilon, evaluate, where)
    return acts


def judge(agents, ref, obs, avail, h_in, last, t, epsilon, evaluate, where):
    pr.check_stages(ref, obs, last if ref.last_action else None, h_in, agents.hidden, agents.q, agents.actions, avail,
                    greedy=False, where=where, worst=WORST)
    R = agents.actions.numel()
    want = action_rule(agents.q.reshape(R, -1), avail, epsilon, evaluate, agents.seed, t)
    got = agents.actions.reshape(-1).cpu().numpy()
    if not np.array_equal(got, want):
        i = int(np.flatnonzero(got != want)[0])
        raise AssertionError("%s: stage (c) row %d: action %d, the rule gives %d on the kernel's q %s"
                             % (where, i, got[i], want[i], agents.q.reshape(R, -1)[i].tolist()))


def random_start(agents, A, gen):
    """hidden states anywhere in (-1, 1) and random last actions (255 = none) instead of the zero start"""
    agents.hidden.copy_(torch.rand(agents.hidden.shape, generator=gen, device=DEV) * 2 - 1)
    la = torch.randint(0, A + 1, agents.actions.shape, generator=gen, device=DEV)
    agents.actions.copy_(torch.where(la == A, 255, la).to(torch.uint8))


def search_obs(shape, M, gen):
    """search-like observation rows: view cells in {0, 0.5, 1}, then two integer positions below M"""
    v = torch.randint(0, 3, shape, generator=gen, device=DEV).to(torch.float32) * 0.5
    v[..., -2:] = torch.randint(0, M, shape[:-1] + (2,), generator=gen, device=DEV).to(torch.float32)
    return v


def some_avail(shape, gen, p=0.6):
    """a random availability mask with at least one available action per row"""
    av = (torch.rand(shape, generator=gen, device=DEV) < p).to(torch.uint8)
    av[..., 0] |= (av.sum(-1) == 0).to(torch.uint8)
    return av


# ---- 1. widths -----------------------------------------------------------------------------------------------------

WIDTHS = [  # n_agents, obs_dim, n_actions, last_action, reuse_network -> input width
    (3, 26, 4, True, True),       # 33: the first wide width, one element in the second 32-slice / third 16-wide K-step
    (5, 27, 8, True, True),       # 40
    (8, 52, 4, True, True),       # 64
    (9, 48, 8, True, True),       # 65
    (16, 108, 4, True, True),     # 128
    (7, 114, 8, True, True),      # 129
    (3, 171, 4, True, True),      # 178: search, 3 agents
    (64, 171, 4, True, True),     # 239: search c5, 64 agents
    (76, 171, 8, True, True),     # 255
    (77, 171, 8, True, True),     # 256: the widest
    (1, 248, 8, True, False),     # 256 without agent ids
    (1, 200, 4, False, False),    # 200, obs only
]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("n,obs_dim,A,last,reuse", WIDTHS)
def test_wide_input_widths(n, obs_dim, A, last, reuse, precision):
    """~50 000 rows, "default" and "scaled" weights, two calls (the second with an availability mask and on the
    kernel's own hidden state and actions); search-like obs at obs_dim 171, uniform (-1, 1) otherwise"""
    gen = torch.Generator(device=DEV).manual_seed(6)
    in_dim = obs_dim + (A if last else 0) + (n if reuse else 0)
    E = -(-50021 // n)
    for kind in ("default", "scaled"):
        sd = pr.random_state_dict(in_dim, A, in_dim, kind)
        ref = pr.PolicyRef(sd, n, obs_dim, A, last, reuse, precision=precision, device=DEV)
        agents = make_agents(sd, E, n, obs_dim, A, last, reuse, precision=precision)
        assert ("K1=256" if precision == "bf16" else "S=8") in agents.kernel_name
        random_start(agents, A, gen)
        for call in range(2):
            obs = search_obs((E, n, obs_dim), 64, gen) if obs_dim == 171 else torch.rand(E, n, obs_dim, generator=gen, device=DEV) * 2 - 1
            avail = (torch.rand(E, n, A, generator=gen, device=DEV) < 0.6).to(torch.uint8) if call else None
            call_checked(agents, ref, obs, avail, where="%s width %d A %d call %d" % (kind, in_dim, A, call))


# ---- 2. row counts -------------------------------------------------------------------------------------------------

# tiles of 128 rows (tensor cores) and warp-iterations of 16 x 4 rows (fp32): a persistent CTA takes its second tile at
# 148 x 128 = 18 944 rows and its second iteration at 148 x 64 = 9472 rows
ROWS = [1, 127, 128, 129, SMS * 64 - 1, SMS * 64 + 1, SMS * 128 - 1, SMS * 128, SMS * 128 + 1, 2 * SMS * 128 + 129]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_wide_row_counts_and_obs_alignment(precision):
    """n_agents 1, width 239 (234 obs values + 4 + 1): exact row counts, two calls each; every other row count reads
    its obs through a view that starts 4 bytes past a 16-byte boundary (the tensor-core kernel's scalar head and tail)"""
    gen = torch.Generator(device=DEV).manual_seed(5)
    D, A = 234, 4
    for kind in ("default", "scaled"):
        sd = pr.random_state_dict(D + A + 1, A, 3, kind)
        ref = pr.PolicyRef(sd, 1, D, A, precision=precision, device=DEV)
        for i, rows in enumerate(ROWS):
            agents = make_agents(sd, rows, 1, D, A, precision=precision)
            random_start(agents, A, gen)
            for call in range(2):
                buf = torch.rand(rows * D + 1, generator=gen, device=DEV) * 2 - 1
                obs = buf[1:].view(rows, 1, D) if i % 2 else buf[:-1].view(rows, 1, D)
                avail = (torch.rand(rows, 1, A, generator=gen, device=DEV) < 0.7).to(torch.uint8) if call else None
                call_checked(agents, ref, obs, avail, where="%s rows %d call %d" % (kind, rows, call))


# ---- 3. the c5 shape -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", PRECISIONS)
def test_c5_shape(precision):
    """131 072 envs x 64 agents = 8 388 608 rows at width 239 (hidden state 2.1 GB, obs 5.7 GB), one call from a random
    start; the reference runs on the device in row slices"""
    E, n, D, A = 131072, 64, 171, 4
    gen = torch.Generator(device=DEV).manual_seed(7)
    sd = pr.random_state_dict(D + A + n, A, 8, "default")
    ref = pr.PolicyRef(sd, n, D, A, precision=precision, device=DEV)
    agents = make_agents(sd, E, n, D, A, precision=precision)
    random_start(agents, A, gen)
    call_checked(agents, ref, search_obs((E, n, D), 64, gen), where="c5")
    del agents
    torch.cuda.empty_cache()


# ---- 4. the search loop under a CUDA graph -------------------------------------------------------------------------

def search_args(n, m, M, R=7):
    return types.SimpleNamespace(env="search", map_size=M, target_num=m, target_mode=0, target_dir="", agent_mode=0,
                                 n_agents=n, view_range=R)


# Under the uniform-random policy half of the c5 envs (64 agents) have reset by step 800 and all by 2500; at 3 agents /
# 15 targets / map 50 half have by step 2200.  Under random weights an agent's greedy action hardly depends on its
# observation: even 10 % greedy steps drift it 0.1 cell per step into a wall, and no env ever finishes.  So epsilon is 1:
# the epsilon-greedy path with every action a uniform available one, each checked exactly against the Philox draws.
LOOPS = [  # n_agents, target_num, map_size, envs, eager steps, epsilon, precision, least share of envs reset at least once
    (64, 1000, 64, 2048, 2500, 1.0, "bf16", 0.9),
    (64, 1000, 64, 2048, 2500, 1.0, "fp32", 0.9),
    (3, 15, 50, 4096, 4000, 1.0, "bf16", 0.5),
]
K, REPLAYS = 10, 50               # steps per captured graph, replays of it


@pytest.mark.parametrize("n,m,M,E,steps,eps,precision,share", LOOPS)
def test_search_loop_in_cuda_graph(n, m, M, E, steps, eps, precision, share):
    """The search loop with auto-reset and epsilon-greedy actions (random weights: greedy actions alone can circle
    forever), in two worlds built from the same seeds.
    Eager phase, `steps` calls with the Philox counter advancing per call as choose_actions advances it: world A
    checks stages (a)-(c) every 100 steps and on five calls after resets, that the rows of envs that reset enter the
    next call with a zero hidden state and last action 255, that no action is unavailable and no env makes an illegal
    move, and that a stated share of the envs reset; world B runs the same calls unchecked.
    Graph phase: world B captures K steps of the loop in one CUDA graph and replays it; world A runs the same steps
    eagerly.  The counter is a kernel parameter, frozen at capture, so every replay repeats the K counters of the
    capture; world A passes that same sequence.  Both worlds end equal bit for bit, and envs reset inside the phase."""
    import coopsearch_b200 as cs
    args = search_args(n, m, M)

    def world():
        env = cs.VecSearchEnv(args, num_envs=E, device=DEV, seed=11, auto_reset=True)
        obs_dim = env.get_env_info()["obs_shape"]
        sd = pr.random_state_dict(obs_dim + 4 + n, 4, 12, "default")
        return env, make_agents(sd, E, n, obs_dim, 4, precision=precision, seed=13), sd, obs_dim

    def body(env, agents):
        obs, avail = env.get_obs(), env.get_avail_actions()
        acts = agents.choose_actions(obs, avail=avail, epsilon=eps, evaluate=False)
        _, term, _ = env.step(acts)
        agents.init_hidden(mask=term)
        return term

    env, agents, sd, obs_dim = world()
    genv, gagents, _, _ = world()
    ref = pr.PolicyRef(sd, n, obs_dim, 4, precision=precision, device=DEV)
    ever = torch.zeros(E, dtype=torch.bool, device=DEV)
    prev = torch.zeros(E, dtype=torch.bool, device=DEV)
    after_reset_checks = 0
    for s in range(steps):
        obs, avail = env.get_obs(), env.get_avail_actions()
        check = s % 100 == 0 or (after_reset_checks < 5 and bool(prev.any()))
        if check:
            obs_in, av_in, h_in, last, t = obs.clone(), avail.clone(), agents.hidden.clone(), agents.actions.clone(), agents._t
            if bool(prev.any()):
                after_reset_checks += 1
                assert bool((h_in[prev] == 0).all()) and bool((last[prev] == 255).all()), "step %d: a reset env kept its agent state" % s
        acts = agents.choose_actions(obs, avail=avail, epsilon=eps, evaluate=False)
        if check:
            judge(agents, ref, obs_in, av_in, h_in, last, t, eps, False, "%da step %d" % (n, s))
            assert bool((av_in.reshape(-1, 4).gather(1, acts.reshape(-1, 1).long()) != 0).all()), "step %d: an unavailable action" % s
        _, term, _ = env.step(acts)
        agents.init_hidden(mask=term)
        prev = term.bool().clone()
        ever |= prev
        assert not bool(env.illegal.any()), "step %d: an illegal move" % s
        body(genv, gagents)
    got_share = ever.double().mean().item()
    print("search loop %da %dt M%d %s: %.3f of %d envs reset at least once in %d steps" % (n, m, M, precision, got_share, E, steps))
    assert after_reset_checks >= 5, "fewer than five calls after a reset were checked"
    assert got_share >= share, "only %.3f of the envs reset at least once" % got_share

    t0 = agents._t
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        gagents._t = t0
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):                   # records, runs nothing
            for _ in range(K):
                body(genv, gagents)
        for _ in range(REPLAYS):
            graph.replay()
        torch.cuda.synchronize(DEV)
    resets = 0
    for r in range(REPLAYS):
        agents._t = t0
        for _ in range(K):
            resets += int(body(env, agents).sum())
    torch.cuda.synchronize(DEV)
    assert resets > 0, "no env reset during the graph phase"
    assert not bool(env.illegal.any()) and env.stats()["illegal_moves"] == 0 and genv.stats()["illegal_moves"] == 0
    pairs = (("hidden", agents.hidden, gagents.hidden), ("q", agents.q, gagents.q), ("actions", agents.actions, gagents.actions),
             ("obs", env.get_obs(), genv.get_obs()), ("positions", env.agent_pos, genv.agent_pos),
             ("counters", env.counters, genv.counters), ("state", env.get_state(), genv.get_state()))
    for name, a, b in pairs:
        assert torch.equal(a, b), "graph replays differ from the eager run in %s (%d resets in the phase)" % (name, resets)


# ---- 5. sampling ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("alg,eps", [("q", 0.3), ("reinforce", 0.2)])
def test_wide_sampling_with_masks(alg, eps, precision):
    """width 239, 1024 envs x 64 agents: epsilon-greedy (exact rule, Philox draws included) and softmax sampling with
    masks: every chosen action is available; the same seed and call count give the same draws, the next call new ones"""
    E, n, D, A = 1024, 64, 171, 4
    gen = torch.Generator(device=DEV).manual_seed(15)
    sd = pr.random_state_dict(D + A + n, A, 16, "scaled")
    ref = pr.PolicyRef(sd, n, D, A, precision=precision, device=DEV)
    obs, avail = search_obs((E, n, D), 64, gen), some_avail((E, n, A), gen)
    runs = []
    for _ in range(2):
        agents = make_agents(sd, E, n, D, A, precision=precision, seed=77, alg=alg)
        out = []
        for call in range(2):
            agents.init_hidden()
            if alg == "q":
                acts = call_checked(agents, ref, obs, avail, where="eps call %d" % call, epsilon=eps, evaluate=False)
            else:
                acts = agents.choose_actions(obs, avail=avail, epsilon=eps, evaluate=False)
            assert bool((avail.reshape(-1, A).gather(1, acts.reshape(-1, 1).long()) != 0).all()), "%s: an unavailable action" % alg
            out.append(acts.clone())
        runs.append(out)
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert (runs[0][0] != runs[0][1]).float().mean().item() > 0.05, "the second call repeated the first call's draws"


# ---- 6. widths past 256 --------------------------------------------------------------------------------------------

def test_width_257_is_refused():
    """BatchedRNNAgents raises CoopSearchError, and cs_policy_create returns an error code, naming the limit 256"""
    import coopsearch_b200 as cs
    from coopsearch_b200 import _lib
    sd = pr.random_state_dict(257, 4, 1)
    with pytest.raises(cs.CoopSearchError, match="256"):
        make_agents(sd, 4, 82, 171, 4)
    lib = _lib.load()
    host = {f: np.ascontiguousarray(sd[k].numpy(), dtype=np.float32) for k, f in
            (("fc1.weight", "fc1_w"), ("fc1.bias", "fc1_b"), ("rnn.weight_ih", "w_ih"), ("rnn.weight_hh", "w_hh"), ("rnn.bias_ih", "b_ih"),
             ("rnn.bias_hh", "b_hh"), ("fc2.0.weight", "fc2a_w"), ("fc2.0.bias", "fc2a_b"), ("fc2.2.weight", "fc2b_w"), ("fc2.2.bias", "fc2b_b"))}
    w = _lib.PolicyWeights(**{k: v.ctypes.data for k, v in host.items()})
    for obs_dim, ok in ((171, False), (170, True)):                   # widths 257 and 256
        cfg = _lib.PolicyCfg(struct_size=C.sizeof(_lib.PolicyCfg), device=0, n_agents=82, obs_dim=obs_dim, n_actions=4, hidden_dim=64,
                             last_action=1, reuse_network=1, conv_out_dim=0)
        hp = C.c_void_p()
        code = lib.cs_policy_create(C.byref(cfg), C.byref(w), C.byref(hp))
        if ok:
            assert code == 0
            lib.cs_policy_destroy(hp)
        else:
            assert code != 0 and b"256" in lib.cs_last_error()
