"""Both agent-network kernels (csrc/policy.cu: policy_kernel, fp32; csrc/policy_tc.cuh: policy_tc_kernel, bf16 tensor
cores) against the float64 reference of oracle/policy_ref.py, stage by stage and on every row, each stage judged on the
kernel's own input to it so that no error is inherited:
  (a) the hidden state the kernel wrote, against the reference's GRU step from the kernel's inputs (obs, last action,
      conv features, the hidden state it read), within the per-element bound of that kernel's arithmetic;
  (b) the action values, against the reference's fc2 on the hidden state the kernel wrote;
  (c) the actions, against the action rule applied to the kernel's own action values: exact.
Shapes: row counts around the tensor-core tile (128 rows) and around where a persistent CTA starts to own a second
tile (2 x 148 CTAs x 128 rows = 37 888), the fp32 kernel's 148 x 64-row step, every input width up to 32 and action
count up to 8, and the benchmark's 262 144 envs x 3 agents.  References of the large shapes are computed in float64 on
the device.  The largest error / bound of each stage and precision is printed at the end of the module."""
import ctypes as C
import types

import pytest
import torch

import golden_util as gu
from oracle import policy_ref as pr

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
PRECISIONS = ["fp32", "bf16"]
WORST = {}                        # (stage, precision[, "no flip"]) -> largest error / bound seen (pr.assert_within)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for key, v in sorted(WORST.items()):
        print("policy reference: stage %s: largest |error| / bound %.3g" % (" ".join(key), v))


def check_stages(*a, **k):
    pr.check_stages(*a, worst=WORST, **k)


def make_agents(sd, E, n, obs_dim, A, last=True, reuse=True, precision="bf16", **kw):
    import coopsearch_b200 as cs
    return cs.BatchedRNNAgents(sd, num_envs=E, n_agents=n, obs_dim=obs_dim, n_actions=A, last_action=last, reuse_network=reuse,
                               device=DEV, precision=precision, **kw)


def call_checked(agents, ref, obs, avail=None, where="", **kw):
    """one choose_actions call, judged against the inputs it read"""
    h_in, last = agents.hidden.clone(), agents.actions.clone()
    acts = agents.choose_actions(obs, avail=avail, **kw)
    check_stages(ref, obs, last if ref.last_action else None, h_in, agents.hidden, agents.q, acts, avail,
                 feat=agents.feat, where=where)
    return acts


def random_start(agents, A, gen):
    """hidden states anywhere in (-1, 1) and random last actions (255 = none) instead of the zero start"""
    agents.hidden.copy_(torch.rand(agents.hidden.shape, generator=gen, device=DEV) * 2 - 1)
    la = torch.randint(0, A + 1, agents.actions.shape, generator=gen, device=DEV)
    agents.actions.copy_(torch.where(la == A, 255, la).to(torch.uint8))


def weights(kind, in_dim, A, seed=1):
    if kind == "shipped":
        g = gu.load("policy_qmix_3a")
        return {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
    return pr.random_state_dict(in_dim, A, seed, kind)


# ---- 1. shape grid -------------------------------------------------------------------------------------------------

ROWS = [1, 2, 127, 128, 129, 4097, 9471, 9473, 37887, 37888, 37889, 3 * 37888 + 77]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_row_counts_around_tiles_and_persistent_loops(precision):
    """n_agents = 1, input width 8, 3 actions: exact row counts; two calls each (random start, then the kernel's own
    hidden state and actions as the next call's inputs, with an availability mask), both weight kinds"""
    gen = torch.Generator(device=DEV).manual_seed(5)
    for kind in ("default", "scaled"):
        sd = weights(kind, 8, 3)
        ref = pr.PolicyRef(sd, 1, 4, 3, precision=precision, device=DEV)
        for rows in ROWS:
            agents = make_agents(sd, rows, 1, 4, 3, precision=precision)
            random_start(agents, 3, gen)
            for call in range(2):
                obs = torch.rand(rows, 1, 4, generator=gen, device=DEV) * 2 - 1
                avail = (torch.rand(rows, 1, 3, generator=gen, device=DEV) < 0.7).to(torch.uint8) if call else None
                call_checked(agents, ref, obs, avail, where="%s rows %d call %d" % (kind, rows, call))


WIDTHS = [  # n_agents, obs_dim, n_actions, last_action, reuse_network -> input width
    (3, 4, 1, True, True),      # 8
    (10, 4, 2, True, True),     # 16
    (6, 4, 7, True, True),      # 17
    (12, 4, 8, True, True),     # 24
    (20, 4, 7, True, True),     # 31
    (20, 4, 8, True, True),     # 32: all four K chunks of fc1
    (1, 24, 8, True, False),    # 32 without agent ids
    (5, 4, 3, False, False),    # 4
    (5, 6, 3, True, False),     # 9
    (8, 4, 5, False, True),     # 12
]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("n,obs_dim,A,last,reuse", WIDTHS)
def test_input_widths_and_action_counts(n, obs_dim, A, last, reuse, precision):
    """~50 000 rows (more than one tile per CTA), both weight kinds, two calls (the second with a mask)"""
    gen = torch.Generator(device=DEV).manual_seed(6)
    in_dim = obs_dim + (A if last else 0) + (n if reuse else 0)
    E = -(-50021 // n)
    for kind in ("default", "scaled"):
        sd = weights(kind, in_dim, A, seed=in_dim)
        ref = pr.PolicyRef(sd, n, obs_dim, A, last, reuse, precision=precision, device=DEV)
        agents = make_agents(sd, E, n, obs_dim, A, last, reuse, precision=precision)
        random_start(agents, A, gen)
        for call in range(2):
            obs = torch.rand(E, n, obs_dim, generator=gen, device=DEV) * 2 - 1
            avail = (torch.rand(E, n, A, generator=gen, device=DEV) < 0.6).to(torch.uint8) if call else None
            call_checked(agents, ref, obs, avail, where="%s width %d A %d call %d" % (kind, in_dim, A, call))


@pytest.mark.parametrize("precision", PRECISIONS)
def test_benchmark_shape(precision):
    """262 144 envs x 3 agents = 786 432 rows (6144 tiles, ~21 per tensor-core CTA), all three weight kinds"""
    gen = torch.Generator(device=DEV).manual_seed(7)
    E = 262144
    for kind in ("default", "scaled", "shipped"):
        sd = weights(kind, 10, 3)
        ref = pr.PolicyRef(sd, 3, 4, 3, precision=precision, device=DEV)
        agents = make_agents(sd, E, 3, 4, 3, precision=precision)
        random_start(agents, 3, gen)
        for call in range(2):
            call_checked(agents, ref, torch.rand(E, 3, 4, generator=gen, device=DEV) * 2 - 1, where="%s call %d" % (kind, call))


# ---- 2. closed loop at the benchmark shape -------------------------------------------------------------------------

@pytest.mark.parametrize("precision", PRECISIONS)
def test_closed_loop_at_benchmark_shape(precision):
    """200 calls on the kernel's own hidden state and actions (the action tensor is the next call's last action), every
    stage checked every call; at call 100 init_hidden(mask) restarts half the envs, whose rows must then start from a
    zero hidden state and no last action while the others continue"""
    E, n = 262144, 3
    gen = torch.Generator(device=DEV).manual_seed(8)
    sd = weights("shipped", 10, 3)
    ref = pr.PolicyRef(sd, n, 4, 3, precision=precision, device=DEV)
    agents = make_agents(sd, E, n, 4, 3, precision=precision)
    for call in range(200):
        if call == 100:
            mask = torch.rand(E, generator=gen, device=DEV) < 0.5
            h0, a0 = agents.hidden.clone(), agents.actions.clone()
            agents.init_hidden(mask)
            assert bool((agents.hidden[mask] == 0).all()) and bool((agents.actions[mask] == 255).all())
            assert torch.equal(agents.hidden[~mask], h0[~mask]) and torch.equal(agents.actions[~mask], a0[~mask])
            assert bool((a0[mask] != 255).any()) and bool((h0[mask] != 0).any())
        obs = torch.rand(E, n, 4, generator=gen, device=DEV) * 2 - 1
        call_checked(agents, ref, obs, where="call %d" % call)


# ---- 3. row boundaries through the raw C ABI -----------------------------------------------------------------------

@pytest.mark.parametrize("precision", PRECISIONS)
def test_raw_abi_writes_every_row_and_nothing_past_it(precision):
    """cs_policy_act on buffers with guard regions past `rows`, filled with a byte pattern: every row < rows is written
    (and right), no guard byte changes, rows = 0 changes nothing, and q = NULL still gives the same actions"""
    from coopsearch_b200 import _lib
    sd = weights("default", 8, 3)
    ref = pr.PolicyRef(sd, 1, 4, 3, precision=precision, device=DEV)
    agents = make_agents(sd, 1, 1, 4, 3, precision=precision)
    lib, G, A = agents.lib, 333, 3
    gen = torch.Generator(device=DEV).manual_seed(9)
    stream = torch.cuda.current_stream(DEV)

    def act(rows, bufs, q=True):
        io = _lib.PolicyIO(rows=rows, evaluate=1, epsilon=0.0, seed=1, t=0, obs=bufs["obs"].data_ptr(),
                           last_action=bufs["act"].data_ptr(), avail=None, hidden=bufs["h"].data_ptr(),
                           q=bufs["q"].data_ptr() if q else None, actions=bufs["act"].data_ptr(),
                           precision=1 if precision == "bf16" else 0, mode=0, feat=None)
        _lib.check(lib.cs_policy_act(agents._h, C.byref(io), C.c_void_p(stream.cuda_stream)), "cs_policy_act")
        torch.cuda.synchronize(DEV)

    for rows in (1, 3, 127, 129, 131, 255, 9473, 9475, 37889, 38015):
        bufs = {"h": torch.empty((rows + G) * 64, device=DEV), "q": torch.empty((rows + G) * A, device=DEV),
                "act": torch.empty(rows + G, dtype=torch.uint8, device=DEV), "obs": torch.empty((rows + G) * 4, device=DEV)}
        for b in bufs.values():
            b.view(torch.uint8).fill_(0xA5)                                   # the guard pattern (also in the rows to be written)
        bufs["h"][:rows * 64] = torch.rand(rows * 64, generator=gen, device=DEV) * 2 - 1
        bufs["obs"][:rows * 4] = torch.rand(rows * 4, generator=gen, device=DEV) * 2 - 1
        la = torch.randint(0, A + 1, (rows,), generator=gen, device=DEV)
        bufs["act"][:rows] = torch.where(la == A, 255, la).to(torch.uint8)
        before = {k: v.clone() for k, v in bufs.items()}
        act(0, bufs)
        assert all(torch.equal(bufs[k], before[k]) for k in bufs), "rows = 0 wrote something"
        act(rows, bufs)
        for k, width in (("h", 64), ("q", A), ("act", 1), ("obs", 4)):
            assert torch.equal(bufs[k][rows * width:], before[k][rows * width:]), "rows %d: guard of %s changed" % (rows, k)
        assert torch.equal(bufs["obs"], before["obs"])
        check_stages(ref, before["obs"][:rows * 4], before["act"][:rows], before["h"][:rows * 64], bufs["h"][:rows * 64],
                     bufs["q"][:rows * A], bufs["act"][:rows], where="raw ABI rows %d" % rows)
        again = {k: v.clone() for k, v in before.items()}
        act(rows, again, q=False)
        assert torch.equal(again["q"], before["q"]), "q = NULL: q written"
        assert torch.equal(again["act"], bufs["act"]) and torch.equal(again["h"], bufs["h"]), "q = NULL changes the result"


# ---- 4. action rules -----------------------------------------------------------------------------------------------

def _chi2_calibration(p, draws, where):
    """Drawn actions against per-row probabilities p [R, A] (float64): never a probability-0 action, and the (row,
    action) pairs binned by p, and by action, drawn as often as their summed p says (Pearson statistic with the Bernoulli variance, a
    conservative chi-square), at a fixed seed so the outcome is deterministic"""
    from scipy.stats import chi2
    R, A = p.shape
    hit = torch.zeros_like(p)
    hit[torch.arange(R, device=p.device), draws.long()] = 1
    assert not bool((hit[p == 0] != 0).any()), "%s: drew a probability-0 action" % where
    edges = torch.tensor([0, .02, .05, .1, .15, .2, .3, .4, .5, .6, .7, .8, .9, 1.0001], dtype=torch.float64, device=p.device)
    b = torch.bucketize(p, edges) - 1
    a = torch.arange(A, device=p.device).expand(R, A)
    stat, dof = 0.0, 0
    for m in [b == i for i in range(len(edges) - 1)] + [a == i for i in range(A)]:      # by p, and by action
        m = m & (p > 0)
        o, e, v = hit[m].sum().item(), p[m].sum().item(), (p[m] * (1 - p[m])).sum().item()
        if v > 0:
            stat += (o - e) ** 2 / v
            dof += 1
    limit = chi2.ppf(1 - 1e-6, dof)
    assert stat < limit, "%s: chi-square %.1f over %d bins (limit %.1f)" % (where, stat, dof, limit)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_greedy_ties_and_rows_without_available_action(precision):
    """Equal fc2.2 rows and biases make exactly equal action values (actions 1 = 2 and 5 = 6, raised above the rest):
    the first index wins, like torch.argmax; rows with no available action take action 0"""
    A, n, E = 8, 3, 40000
    sd = weights("default", 4 + A + n, A, seed=3)
    w, b = sd["fc2.2.weight"].clone(), sd["fc2.2.bias"].clone()
    w[2], w[6] = w[1], w[5]
    b[1] = b[2] = b[1] + 1.0
    b[5] = b[6] = b[5] + 1.0
    sd["fc2.2.weight"], sd["fc2.2.bias"] = w, b
    ref = pr.PolicyRef(sd, n, 4, A, precision=precision, device=DEV)
    agents = make_agents(sd, E, n, 4, A, precision=precision)
    gen = torch.Generator(device=DEV).manual_seed(10)
    random_start(agents, A, gen)
    avail = (torch.rand(E, n, A, generator=gen, device=DEV) < 0.7).to(torch.uint8)
    avail[::7] = 0                                                            # every 7th env: nothing available
    acts = call_checked(agents, ref, torch.rand(E, n, 4, generator=gen, device=DEV) * 2 - 1, avail, where="ties")
    q = agents.q
    assert torch.equal(q[..., 1], q[..., 2]) and torch.equal(q[..., 5], q[..., 6]), "equal weights gave unequal action values"
    assert bool((acts[::7] == 0).all())
    both = (avail[..., 1] == 1) & (avail[..., 2] == 1) & (acts == 1)
    assert both.float().mean().item() > 0.05, "the tie between actions 1 and 2 was never the maximum"


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("eps", [0.1, 0.5])
def test_epsilon_greedy_frequencies(eps, precision):
    """agent.py:71-74 (not evaluate): argmax with probability 1 - eps, else a uniform available action -- so
    (1 - eps) onehot(argmax) + eps / n_avail over the row's available actions, argmax on the kernel's own q"""
    A, n, E = 5, 3, 100000
    sd = weights("default", 4 + A + n, A, seed=4)
    agents = make_agents(sd, E, n, 4, A, precision=precision, seed=21)
    gen = torch.Generator(device=DEV).manual_seed(11)
    random_start(agents, A, gen)
    avail = (torch.rand(E, n, A, generator=gen, device=DEV) < 0.6).to(torch.uint8)
    avail[..., 0] |= (avail.sum(-1) == 0).to(torch.uint8)
    acts = agents.choose_actions(torch.rand(E, n, 4, generator=gen, device=DEV) * 2 - 1, avail=avail, epsilon=eps, evaluate=False)
    ok = avail.reshape(-1, A).double()
    p = eps * ok / ok.sum(1, keepdim=True)
    best = pr.greedy_rule(agents.q.reshape(-1, A), avail)
    p[torch.arange(p.shape[0], device=DEV), best] += 1 - eps
    _chi2_calibration(p, acts.reshape(-1), "epsilon %g" % eps)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_reinforce_sampling_against_float64_mixture(precision):
    """alg=reinforce (agent.py:77-97) at 8 actions with masked actions: draws against Categorical((1 - eps) softmax(q) +
    eps / n_avail, unavailable = 0) of the kernel's own q in float64; the scaled weights spread q over tens"""
    A, n, E, eps = 8, 2, 100000, 0.2
    sd = weights("default", 4 + A + n, A, seed=5)
    sd["fc2.2.weight"], sd["fc2.2.bias"] = sd["fc2.2.weight"] * 20, sd["fc2.2.bias"] * 20
    agents = make_agents(sd, E, n, 4, A, precision=precision, seed=22, alg="reinforce")
    gen = torch.Generator(device=DEV).manual_seed(12)
    random_start(agents, A, gen)
    avail = (torch.rand(E, n, A, generator=gen, device=DEV) < 0.6).to(torch.uint8)
    avail[..., 3] = 1
    acts = agents.choose_actions(torch.rand(E, n, 4, generator=gen, device=DEV) * 2 - 1, avail=avail, epsilon=eps, evaluate=False)
    ok = avail.reshape(-1, A).double()
    p = ((1 - eps) * torch.softmax(agents.q.reshape(-1, A).double(), -1) + eps / ok.sum(1, keepdim=True)) * ok
    p = p / p.sum(1, keepdim=True)
    _chi2_calibration(p, acts.reshape(-1), "reinforce")


@pytest.mark.parametrize("alg,eps", [("q", 0.5), ("reinforce", 0.2)])
def test_draws_reproduce_by_seed_and_call_count(alg, eps):
    """The same seed and call count give the same draws; the next call draws anew"""
    A, n, E = 5, 3, 20000
    sd = weights("default", 4 + A + n, A, seed=6)
    obs = torch.rand(E, n, 4, generator=torch.Generator(device=DEV).manual_seed(13), device=DEV) * 2 - 1
    runs = []
    for _ in range(2):
        agents = make_agents(sd, E, n, 4, A, seed=77, alg=alg)
        out = []
        for _ in range(2):
            agents.init_hidden()
            out.append(agents.choose_actions(obs, epsilon=eps, evaluate=False).clone())
        runs.append(out)
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert (runs[0][0] != runs[0][1]).float().mean().item() > 0.15, "the second call repeated the first call's draws"


# ---- 5. conv front end ---------------------------------------------------------------------------------------------

def conv_weights(geo, seed):
    torch.manual_seed(seed)
    cs_ = (geo["map_size"] - geo["kernel_size_1"]) // geo["stride_1"] + 1
    c1 = torch.nn.Conv2d(1, geo["dim_1"], geo["kernel_size_1"], geo["stride_1"])
    c2 = torch.nn.Conv2d(geo["dim_1"], geo["dim_2"], geo["kernel_size_2"], geo["stride_2"], geo["padding_2"])
    lin = torch.nn.Linear(geo["dim_2"] * cs_ * cs_, geo["conv_out_dim"])
    sd = {"conv.0." + k: v for k, v in c1.state_dict().items()}
    sd.update({"conv.2." + k: v for k, v in c2.state_dict().items()})
    sd.update({"linear." + k: v for k, v in lin.state_dict().items()})
    return {k: v.detach().clone() for k, v in sd.items()}


def tiled(maps):
    """row-major [E, M, M] -> the flight env's tiled layout [E, tiles, tiles, 4, 4] (zero padded)"""
    E, M, _ = maps.shape
    T = (M + 3) // 4
    pad = torch.zeros(E, 4 * T, 4 * T, device=maps.device)
    pad[:, :M, :M] = maps
    return pad.reshape(E, T, 4, T, 4).permute(0, 1, 3, 2, 4).contiguous()


def belief_maps(E, M, gen):
    m = torch.rand(E, M, M, generator=gen, device=DEV)
    m[m < 0.1] = 0
    m[m > 0.95] = 1
    return m


GEOMETRIES = [  # map_size, dim_1, kernel_size_1, stride_1, dim_2, kernel_size_2, stride_2, padding_2, conv_out_dim
    (17, 4, 3, 1, 1, 3, 1, 1, 7),
    (30, 4, 4, 2, 2, 3, 1, 1, 16),
    (50, 4, 4, 2, 1, 3, 1, 1, 16),     # the flight agents' defaults (common/arguments.py:246-265)
    (63, 8, 5, 2, 8, 5, 1, 2, 1),      # ~107 KB of shared memory
    (63, 16, 4, 2, 2, 1, 1, 0, 7),
]
GEO_KEYS = ("map_size", "dim_1", "kernel_size_1", "stride_1", "dim_2", "kernel_size_2", "stride_2", "padding_2", "conv_out_dim")


def conv_policy(geo, precision, E, n=3, A=3, seed=0):
    sd = weights("default", geo["conv_out_dim"] + 4 + A + n, A, seed=seed)
    sd.update(conv_weights(geo, seed))
    agents = make_agents(sd, E, n, 4, A, precision=precision, conv=dict(geo))
    ref = pr.PolicyRef(sd, n, 4, A, feat_dim=geo["conv_out_dim"], precision=precision, device=DEV)
    return sd, agents, ref


def conv_checked(sd, agents, ref, geo, maps, gen, where):
    feat = agents.conv_features(prob_map_tiles=tiled(maps))
    want, ef = pr.conv_features(maps, sd, **geo)
    pr.assert_within("conv", "fp32", feat.double() - want, ef, where, WORST)
    call_checked(agents, ref, torch.rand(agents.num_envs, agents.n_agents, 4, generator=gen, device=DEV) * 2 - 1, where=where)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("g", GEOMETRIES, ids=lambda g: "M%d_d%d_k%d_s%d_d%d_k%d_p%d_out%d" % (g[0], g[1], g[2], g[3], g[4], g[5], g[7], g[8]))
def test_conv_front_end_geometries(g, precision):
    """features against float64 conv within their accumulation bound, then (a)-(c) with 3 agents, so each agent row
    gets its env's features; 4099 envs (12 297 rows), two calls on fresh maps"""
    geo = dict(zip(GEO_KEYS, g))
    E = 4099
    gen = torch.Generator(device=DEV).manual_seed(14)
    sd, agents, ref = conv_policy(geo, precision, E)
    random_start(agents, 3, gen)
    for call in range(2):
        conv_checked(sd, agents, ref, geo, belief_maps(E, geo["map_size"], gen), gen, "conv %s call %d" % (g, call))


def test_two_conv_policies_of_different_sizes_alternately():
    """a small and a large (> 48 KB of shared memory) conv front end live at once, called in turn"""
    gen = torch.Generator(device=DEV).manual_seed(15)
    pols = []
    for g, seed in ((GEOMETRIES[0], 1), (GEOMETRIES[3], 2)):
        geo = dict(zip(GEO_KEYS, g))
        pols.append((geo,) + conv_policy(geo, "bf16", 1000, seed=seed))
    for rnd in range(3):
        for geo, sd, agents, ref in pols:
            conv_checked(sd, agents, ref, geo, belief_maps(1000, geo["map_size"], gen), gen, "alternating round %d M %d" % (rnd, geo["map_size"]))


# ---- 6. the benchmark's device loop in a CUDA graph ----------------------------------------------------------------

def test_graph_of_device_loop_equals_eager():
    """get_obs -> choose_actions -> step, 10 steps captured in one CUDA graph and replayed again and again (as bench.py's
    device loop does) equal the same steps run eagerly, bit for bit: hidden, q, actions and env state after the first
    and the second replay (a value frozen at capture, such as a host-side step counter passed as a kernel parameter,
    only shows from the second replay on); two eager runs are equal"""
    import coopsearch_b200 as cs
    E, n = 262144, 3
    sd = weights("default", 10, 3)
    args = types.SimpleNamespace(env="flight_easy", map_size=50, target_num=15, target_mode=0, agent_mode=0, n_agents=n,
                                 view_range=7, time_limit=200, detect_prob=0.9, safe_dist=1, agent_velocity=1, force_dist=3)

    def world():
        env = cs.VecFlightEasyEnv(args, gu.TEMPLATE, num_envs=E, device=DEV, seed=3, auto_reset=True)
        return env, make_agents(sd, E, n, 4, 3)

    def snapshot(env, agents):
        torch.cuda.synchronize(DEV)
        return [agents.hidden.clone(), agents.q.clone(), agents.actions.clone(), env.get_state().clone()]

    eager = []                                           # [run][after 13 / 23 steps]
    for _ in range(2):
        env, agents = world()
        snaps = []
        for t in range(23):
            env.step(agents.choose_actions(env.get_obs()))
            if t in (12, 22):
                snaps.append(snapshot(env, agents))
        eager.append(snaps)
    env, agents = world()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    got = []
    with torch.cuda.stream(side):
        for _ in range(3):
            env.step(agents.choose_actions(env.get_obs()))
        torch.cuda.synchronize(DEV)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(10):
                env.step(agents.choose_actions(env.get_obs()))
        for _ in range(2):
            graph.replay()
            got.append(snapshot(env, agents))
    names = ("hidden", "q", "actions", "env state")
    for k, steps in enumerate((13, 23)):
        for name, a, b, c in zip(names, eager[0][k], eager[1][k], got[k]):
            assert torch.equal(a, b), "two eager runs differ in %s after %d steps" % (name, steps)
            assert torch.equal(a, c), "graph replay %d differs from eager in %s after %d steps" % (k + 1, name, steps)
