"""The float64 reference of the agent network (oracle/policy_ref.py) that the GPU tests judge both kernels of
csrc/policy.cu with, checked on any box: it reproduces the reference's own RNN outputs (tests/golden/policy_*.npz)
within the fp32 bound, its bf16 rounding is the host packer's rule, and its per-element bounds are tight enough that
each of a list of plausible kernel mistakes, applied to the reference itself, lands well outside them."""
import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import policy_ref as pr


def _ratio(err, bound):
    return pr.bound_ratio(err, bound).max().item()


def test_golden_rnn_outputs_within_bound():
    """policy_qmix_3a: the reference's own fp32 RNN with the shipped weights, against the float64 reference with the
    fp32 kernel's bounds.  Every stage on the golden's own inputs to that stage: hidden[t] from (obs[t], actions[t-1],
    hidden[t-1]), q[t] from hidden[t], actions[t] = argmax q[t]."""
    g = gu.load("policy_qmix_3a")
    n, obs_dim, A = [int(v) for v in g["meta"]]
    sd = {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision="fp32")
    steps = g["obs"].shape[0]
    worst = [0.0, 0.0]
    for t in range(steps):
        h_in = torch.zeros(g["hidden"][t].shape) if t == 0 else torch.from_numpy(g["hidden"][t - 1])
        last = None if t == 0 else torch.from_numpy(g["actions"][t - 1])
        h, eh = ref.hidden(ref.inputs(torch.from_numpy(g["obs"][t]), last), h_in)
        worst[0] = max(worst[0], _ratio(torch.from_numpy(g["hidden"][t]).reshape(h.shape).double() - h, eh))
        q, eq = ref.q(torch.from_numpy(g["hidden"][t]))
        worst[1] = max(worst[1], _ratio(torch.from_numpy(g["q"][t]).reshape(q.shape).double() - q, eq))
        assert np.array_equal(pr.greedy_rule(torch.from_numpy(g["q"][t])).numpy(), g["actions"][t])
    assert worst[0] <= 1 and worst[1] <= 1, worst
    # and the float64 reference is not just loose: fp32 rounding is all that separates it from the golden
    q, _ = ref.q(torch.from_numpy(g["hidden"][-1]))
    np.testing.assert_allclose(q.numpy().reshape(g["q"][-1].shape), g["q"][-1], rtol=1e-5, atol=1e-4)


def test_golden_conv_features_and_network_within_bound():
    """policy_conv_qmix_3a: the reference's RNN(conv=True) with the shipped `flight` weights on belief-map-like maps."""
    g = gu.load("policy_conv_qmix_3a")
    n, obs_dim, A, M = [int(v) for v in g["meta"]]
    sd = {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
    geo = dict(dim_1=4, kernel_size_1=4, stride_1=2, dim_2=1, kernel_size_2=3, stride_2=1, padding_2=1)
    ref = pr.PolicyRef(sd, n, obs_dim, A, feat_dim=16, precision="fp32")
    for t in range(g["obs"].shape[0]):
        feat, ef = pr.conv_features(torch.from_numpy(g["maps"][t]), sd, **geo)
        assert _ratio(torch.from_numpy(g["feat"][t]).double() - feat, ef) <= 1
        h_in = torch.zeros(g["hidden"][t].shape) if t == 0 else torch.from_numpy(g["hidden"][t - 1])
        last = None if t == 0 else torch.from_numpy(g["actions"][t - 1])
        h, eh = ref.hidden(ref.inputs(torch.from_numpy(g["obs"][t]), last, torch.from_numpy(g["feat"][t])), h_in)
        assert _ratio(torch.from_numpy(g["hidden"][t]).reshape(h.shape).double() - h, eh) <= 1, t
        q, eq = ref.q(torch.from_numpy(g["hidden"][t]))
        assert _ratio(torch.from_numpy(g["q"][t]).reshape(q.shape).double() - q, eq) <= 1, t


def test_bf16_rounding_is_the_host_packers_rule():
    """pr.bf16 (torch's fp32 -> bf16) against the rule host_bf16 packs the weights with (csrc/policy.cu): ties to even in
    both directions, subnormals, the largest finite values (which round to inf), +-0, +-inf, and 2^22 random fp32 bit
    patterns (NaNs aside: only their NaN-ness is kept)"""
    rng = np.random.default_rng(0)
    special = []
    for top in (0x3F80, 0x3F81, 0x0000, 0x0001, 0x007F, 0x7F7F, 0x8000, 0xBF81, 0xFF7F, 0x4000):
        for low in (0x0000, 0x0001, 0x7FFF, 0x8000, 0x8001, 0xFFFF):
            special.append((top << 16) | low)
    special += [0x7F800000, 0xFF800000, 0x00000001, 0x80000001, 0x007FFFFF, 0x7F7FFFFF, 0xFF7FFFFF]
    u = np.concatenate([np.array(special, np.uint32), rng.integers(0, 2 ** 32, size=1 << 22, dtype=np.uint64).astype(np.uint32)])
    f = u.view(np.float32)
    finite_or_inf = ~np.isnan(f)
    want = pr.bf16_bits_rule(u[finite_or_inf])
    got = pr.bf16(torch.from_numpy(f[finite_or_inf]).double()).to(torch.float32).numpy().view(np.uint32) >> 16
    assert np.array_equal(got.astype(np.uint16), want)
    assert np.isnan(pr.bf16(torch.from_numpy(f[~finite_or_inf]).double()).numpy()).all()
    # the ties: 1 + 2^-8 is halfway between 1 and 1 + 2^-7 -> even (1); 1 + 3 * 2^-8 -> even (1 + 2^-6)
    # and among bf16 subnormals (step 2^-133): 1.5 and 2.5 steps -> 2 steps
    t = pr.bf16(torch.tensor([1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8, -(1 + 2.0 ** -8), 1.5 * 2.0 ** -133, 2.5 * 2.0 ** -133], dtype=torch.float64))
    assert t.tolist() == [1.0, 1 + 2.0 ** -6, -1.0, 2.0 ** -132, 2.0 ** -132]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stage_check_fails_on_any_wrong_nan_or_inf_output(precision):
    """pr.check_stages (what the GPU tests judge every kernel call with) passes the reference's own outputs and fails on
    one element off, on that element with a NaN elsewhere in the same chunk (a NaN must not hide it), on outputs that
    are all NaN with action 0 (which the first-maximum rule would pick), and on an inf; so does assert_within"""
    n, obs_dim, A, E = 3, 4, 3, 500
    sd = pr.random_state_dict(obs_dim + A + n, A, seed=2)
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision=precision)
    gen = torch.Generator().manual_seed(3)
    obs = torch.rand(E * n, obs_dim, generator=gen) * 2 - 1
    last = torch.randint(0, A, (E * n,), generator=gen).to(torch.uint8)
    h_in = torch.rand(E * n, 64, generator=gen) * 2 - 1
    h_out = ref.hidden(ref.inputs(obs, last), h_in)[0].float()
    q = ref.q(h_out)[0].float()
    acts = pr.greedy_rule(q).to(torch.uint8)
    pr.check_stages(ref, obs, last, h_in, h_out, q, acts)

    def fails(h, qq, aa):
        with pytest.raises(AssertionError):
            pr.check_stages(ref, obs, last, h_in, h, qq, aa)

    off = h_out.clone()
    off[10, 5] += 0.5
    fails(off, q, acts)
    off[700, 9] = float("nan")
    fails(off, q, acts)
    fails(torch.full_like(h_out, float("nan")), torch.full_like(q, float("nan")), torch.zeros_like(acts))
    qi = q.clone()
    qi[3, 1] = float("inf")
    fails(h_out, qi, acts)
    qn = q.clone()
    qn[4, 0] = float("nan")
    fails(h_out, qn, acts)
    bound = torch.ones(4, 2, dtype=torch.float64)
    pr.assert_within("conv", precision, torch.zeros(4, 2, dtype=torch.float64), bound)
    for bad in (float("nan"), float("inf")):
        err = torch.zeros(4, 2, dtype=torch.float64)
        err[2, 1] = bad
        with pytest.raises(AssertionError):
            pr.assert_within("conv", precision, err, bound)


# ---- the bounds discriminate: kernel mistakes restated on the reference land outside them -------------------------

def _swap_rz(sd):
    sd = dict(sd)
    for k in ("rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh"):
        v = sd[k].clone()
        v[:64], v[64:128] = sd[k][64:128], sd[k][:64]
        sd[k] = v
    return sd


def _set(sd, key, fn):
    sd = dict(sd)
    v = sd[key].clone()
    fn(v)
    sd[key] = v
    return sd


def _shift_bias(v):
    v[:-1] = v[1:].clone()
    v[-1] = 0


PERTURBATIONS = {
    # name: (stage, how): stage "a" = judged on the hidden state, "b" = on the action values
    "b_hn dropped": ("a", lambda sd: _set(sd, "rnn.bias_hh", lambda v: v[128:].zero_())),
    "r and z gates swapped": ("a", _swap_rz),
    "input elements 24..31 zeroed": ("a", lambda sd: _set(sd, "fc1.weight", lambda v: v[:, 24:32].zero_())),
    "action bias shifted by one": ("b", lambda sd: _set(sd, "fc2.2.bias", _shift_bias)),
    "bf16(h) in the blend": ("a", None),
    "stale h_in": ("a", None),
    "fc2.2 action 7 zeroed": ("b", lambda sd: _set(sd, "fc2.2.weight", lambda v: v[7].zero_())),
}


@pytest.mark.parametrize("kind", ["default", "scaled"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(PERTURBATIONS))
def test_bounds_catch_kernel_mistakes(name, precision, kind):
    """n_agents 20 with last action and agent id: input width 32 (all four K chunks of the tensor-core fc1), 8 actions.
    On 4000 rows of random inputs and hidden states, each mistake must exceed the stage bound on a clear share of the
    rows it can touch (elements 24..31 are the agent ids 12..19: 40 % of the rows)."""
    n, obs_dim, A = 20, 4, 8
    sd = pr.random_state_dict(obs_dim + A + n, A, seed=7, kind=kind)
    ref = pr.PolicyRef(sd, n, obs_dim, A, precision=precision)
    gen = torch.Generator().manual_seed(1)
    R = 4000
    obs = torch.rand(R, obs_dim, generator=gen) * 2 - 1
    last = torch.randint(0, A + 1, (R,), generator=gen).to(torch.uint8)
    last[last == A] = 255
    h_prev = torch.rand(R, 64, generator=gen) * 2 - 1
    h_in, _ = ref.hidden(ref.inputs(torch.rand(R, obs_dim, generator=gen) * 2 - 1, last), h_prev)
    h_in = h_in.float()
    x = ref.inputs(obs, last)
    stage, how = PERTURBATIONS[name]
    if stage == "a":
        h, eh = ref.hidden(x, h_in)
        if name == "bf16(h) in the blend":
            hp, _ = ref.hidden(x, pr.bf16(h_in.double()).float())
        elif name == "stale h_in":
            hp, _ = ref.hidden(x, h_prev)
        else:
            bad = pr.PolicyRef(how(sd), n, obs_dim, A, precision=precision)
            hp, _ = bad.hidden(bad.inputs(obs, last), h_in)
        ratio = ((hp - h).abs() / eh).amax(1)
    else:
        h_out, _ = ref.hidden(x, h_in)
        q, eq = ref.q(h_out.float())
        bad = pr.PolicyRef(how(sd), n, obs_dim, A, precision=precision)
        qp, _ = bad.q(h_out.float())
        ratio = ((qp - q).abs() / eq).amax(1)
    share = (ratio > 1).double().mean().item()
    need = 0.3 if name == "input elements 24..31 zeroed" else 0.5
    assert share >= need, "%s: only %.1f %% of the rows outside the bound (median ratio %.2f)" % (name, 100 * share, ratio.median().item())
