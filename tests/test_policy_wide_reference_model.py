"""The float64 reference of the agent network (oracle/policy_ref.py) at the wide input widths of the search agents
((2R-1)^2 + 2 = 171 obs values, a 4-action last-action one-hot and an n-agent id one-hot: 178 at 3 agents, 239 at 64)
and at the largest width the kernels take (256), checked on any box: it equals float64 torch modules built from the
same weights, an fp32 emulation of the bf16 tensor-core kernel stays inside its bf16 bounds, and four plausible
mistakes of the wide kernels' input assembly land outside the bounds."""
import pytest
import torch

from oracle import policy_ref as pr

F64 = torch.float64
WIDE = [  # n_agents, obs_dim, n_actions -> width obs_dim + n_actions + n_agents
    (3, 171, 4),      # 178: search, 3 agents, view range 7
    (64, 171, 4),     # 239: search c5, 64 agents
    (77, 171, 8),     # 256: the widest input the kernels take
]


def search_obs(R, obs_dim, M, gen):
    """search-like observation rows: view cells in {0, 0.5, 1}, then two integer positions below M"""
    v = torch.randint(0, 3, (R, obs_dim), generator=gen).to(torch.float32) * 0.5
    v[:, -2:] = torch.randint(0, M, (R, 2), generator=gen).to(torch.float32)
    return v


def last_actions(R, A, gen):
    la = torch.randint(0, A + 1, (R,), generator=gen)
    return torch.where(la == A, 255, la).to(torch.uint8)


def torch_rnn(sd):
    """the reference's RNN (network/base_net.py:22-47) in float64"""
    in_dim = sd["fc1.weight"].shape[1]
    fc1, rnn = torch.nn.Linear(in_dim, 64).double(), torch.nn.GRUCell(64, 64).double()
    fc2 = torch.nn.Sequential(torch.nn.Linear(64, 64), torch.nn.ReLU(), torch.nn.Linear(64, sd["fc2.2.weight"].shape[0])).double()
    fc1.load_state_dict({k[4:]: v.double() for k, v in sd.items() if k.startswith("fc1.")})
    rnn.load_state_dict({k[4:]: v.double() for k, v in sd.items() if k.startswith("rnn.")})
    fc2.load_state_dict({k[4:]: v.double() for k, v in sd.items() if k.startswith("fc2.")})
    return fc1, rnn, fc2


@pytest.mark.parametrize("kind", ["default", "scaled"])
@pytest.mark.parametrize("n,obs_dim,A", WIDE)
def test_reference_equals_float64_torch_rnn(n, obs_dim, A, kind):
    """PolicyRef("fp32") = fc1 -> ReLU -> GRUCell -> fc2 of float64 torch modules, within the fp32 bound (and in fact
    to float64 rounding), on 3000 rows with random last actions and hidden states"""
    in_dim = obs_dim + A + n
    sd = pr.random_state_dict(in_dim, A, seed=in_dim, kind=kind)
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision="fp32")
    assert ref.in_dim == in_dim
    gen = torch.Generator().manual_seed(in_dim)
    R = n * (3000 // n)
    obs, last = search_obs(R, obs_dim, 64, gen), last_actions(R, A, gen)
    h_in = torch.rand(R, 64, generator=gen) * 2 - 1
    x = ref.inputs(obs, last)
    la = last.long()
    onehot_a = torch.zeros(R, A, dtype=F64)
    onehot_a[la != 255, la[la != 255]] = 1
    ids = torch.eye(n, dtype=F64).repeat(R // n, 1)
    assert torch.equal(x, torch.cat([obs.double(), onehot_a, ids], 1))
    fc1, rnn, fc2 = torch_rnn(sd)
    with torch.no_grad():
        h_t = rnn(torch.relu(fc1(x)), h_in.double())
        q_t = fc2(h_t)
    h, eh = ref.hidden(x, h_in)
    q, eq = ref.q(h_t)
    assert pr.bound_ratio(h_t - h, eh).max().item() <= 1
    assert pr.bound_ratio(q_t - q, eq).max().item() <= 1
    assert (h_t - h).abs().max().item() < 1e-12 and (q_t - q).abs().max().item() < 1e-9


def emulate_bf16_kernel(ref, sd, x, h_in):
    """policy_tc_kernel in fp32 on the CPU: bf16 operands (input row, weights, x1, the GEMM copy of h, f), fp32
    accumulation, sigmoid = 0.5 tanh(0.5 x) + 0.5, fp32 hidden state -> (h', q)"""
    b = lambda t: t.to(torch.float32).to(torch.bfloat16).to(torch.float32)
    w = {k: v.to(torch.float32) for k, v in sd.items()}
    x1 = b(torch.relu(b(x) @ b(w["fc1.weight"]).T + w["fc1.bias"]))
    h = h_in.to(torch.float32)
    gi, gh = x1 @ b(w["rnn.weight_ih"]).T, b(h) @ b(w["rnn.weight_hh"]).T
    bi, bh = w["rnn.bias_ih"], w["rnn.bias_hh"]
    pre = gi[:, :128] + gh[:, :128] + (bi[:128] + bh[:128])
    r, z = 0.5 * torch.tanh(0.5 * pre[:, :64]) + 0.5, 0.5 * torch.tanh(0.5 * pre[:, 64:]) + 0.5
    nn_ = torch.tanh(gi[:, 128:] + bi[128:] + r * (gh[:, 128:] + bh[128:]))
    h_new = (1 - z) * nn_ + z * h
    f = b(torch.relu(b(h_new) @ b(w["fc2.0.weight"]).T + w["fc2.0.bias"]))
    q = f @ b(w["fc2.2.weight"]).T + w["fc2.2.bias"]
    return h_new, q


@pytest.mark.parametrize("kind", ["default", "scaled"])
@pytest.mark.parametrize("n,obs_dim,A", WIDE)
def test_fp32_emulation_of_bf16_kernel_within_bound(n, obs_dim, A, kind):
    """the bf16 rounding of a search input row is exact (values 0, 0.5, 1 and integers below 256), and an fp32
    emulation of the tensor-core kernel lies inside the bf16 bounds of stages (a) and (b)"""
    in_dim = obs_dim + A + n
    sd = pr.random_state_dict(in_dim, A, seed=in_dim + 1, kind=kind)
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision="bf16")
    gen = torch.Generator().manual_seed(in_dim + 1)
    R = n * (3000 // n)
    obs, last = search_obs(R, obs_dim, 256, gen), last_actions(R, A, gen)
    h_in = torch.rand(R, 64, generator=gen) * 2 - 1
    x = ref.inputs(obs, last)
    assert torch.equal(x, pr.PolicyRef(sd, n, obs_dim, A, precision="fp32").inputs(obs, last)), "bf16 rounded a search input"
    h_k, q_k = emulate_bf16_kernel(ref, sd, x, h_in)
    h, eh = ref.hidden(x, h_in)
    assert pr.bound_ratio(h_k.double() - h, eh).max().item() <= 1
    q, eq = ref.q(h_k)
    assert pr.bound_ratio(q_k.double() - q, eq).max().item() <= 1


# ---- the bounds discriminate: mistakes of the wide input assembly, restated on the reference -----------------------

def _x_upper_chunks_dropped(ref, obs, last, R):
    x = ref.inputs(obs, last).clone()
    x[:, 128:] = 0
    return x


def _x_id_shifted(ref, obs, last, R):
    x = ref.inputs(obs, last).clone()
    k0 = ref.obs_dim + ref.n_actions
    x[:, k0:] = torch.roll(x[:, k0:], 1, dims=1)
    return x


def _x_wrong_stride(ref, obs, last, R):
    D = ref.obs_dim
    flat = torch.cat([obs.reshape(-1), torch.zeros(D)])
    bad = torch.stack([flat[r * (D - 1):r * (D - 1) + D] for r in range(R)])
    return ref.inputs(bad, last)


def _x_blocks_swapped(ref, obs, last, R):
    x = ref.inputs(obs, last)
    D, A = ref.obs_dim, ref.n_actions
    return torch.cat([x[:, :D], x[:, D + A:], x[:, D:D + A]], 1)


MISTAKES = {
    "inputs 128..255 zeroed (upper K chunks dropped)": _x_upper_chunks_dropped,
    "agent-id one-hot shifted by one": _x_id_shifted,
    "obs read with row stride obs_dim - 1": _x_wrong_stride,
    "last-action and agent-id blocks swapped": _x_blocks_swapped,
}


@pytest.mark.parametrize("kind", ["default", "scaled"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(MISTAKES))
def test_bounds_catch_wide_input_mistakes(name, precision, kind):
    """c5's width 239 (64 agents, 171 obs values, 4 actions): on 2048 rows (32 envs) with random last actions and
    hidden states, each mistake puts a clear share of the rows outside the stage (a) bound, or changes an action of
    the exact stage (c) on the reference's own action values"""
    n, obs_dim, A = 64, 171, 4
    sd = pr.random_state_dict(obs_dim + A + n, A, seed=9, kind=kind)
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision=precision)
    gen = torch.Generator().manual_seed(2)
    R = 2048
    obs, last = search_obs(R, obs_dim, 64, gen), last_actions(R, A, gen)
    h_in = torch.rand(R, 64, generator=gen) * 2 - 1
    h, eh = ref.hidden(ref.inputs(obs, last), h_in)
    hp, _ = ref.hidden(MISTAKES[name](ref, obs, last, R), h_in)
    outside = ((hp - h).abs() > eh).any(1)
    acts = pr.greedy_rule(ref.q(h.float())[0])
    changed = pr.greedy_rule(ref.q(hp.float())[0]) != acts
    share = (outside | changed).double().mean().item()
    assert share >= 0.5, "%s: only %.1f %% of the rows caught" % (name, 100 * share)
