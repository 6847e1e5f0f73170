"""Float64 reference of the agent network -- TEST INFRASTRUCTURE (oracle side).

The reference's RNN (network/base_net.py:5-47: input assembly of agent/agent.py:38-50, fc1 -> ReLU -> GRUCell(64) ->
Linear -> ReLU -> Linear, and the conv front end of the `flight` agents) in torch float64, on any device: the CPU for
small checks, the GPU for the benchmark's 786 432 rows.  Every value comes with a per-element bound on how far the
CUDA kernels of csrc/policy.cu may lie from it, so that a test can hold each kernel to what its arithmetic allows and
no more.

precision "bf16" restates where ``policy_tc_kernel`` (csrc/policy_tc.cuh) rounds operands to bf16 (round to nearest
even, through fp32 first, as ``__floats2bfloat162_rn`` and the host packer ``host_bf16`` do): the fc1 input row, every
weight block, x1 = ReLU(fc1), the GEMM copy of the hidden state and f = ReLU(fc2.0).  Biases, the gate arithmetic and
the GRU blend stay in float64 (the kernel keeps them in fp32; the hidden state it blends and writes back is fp32).
precision "fp32" is ``policy_kernel``: fp32 operands throughout.

Error model (all bounds are absolute, per element):
  * a dot product of K terms (a bias counts as one) accumulated in fp32 in any order: K * 2^-22 * sum |terms|.  That
    is 4 gamma_K; the tensor core's accumulation order and rounding are unspecified, so this is an assumption, and the
    GPU tests report the largest measured error / bound on the B200.
  * operand deviations carry through a dot product as sum |w| * deviation.
  * tanh.approx.f32 (the tensor-core kernel's sigmoid = 0.5 tanh(0.5 x) + 0.5 and tanh): relative error 2^-10.987, the
    maximum the PTX ISA documents for the instruction (PTX ISA 8.x, "tanh").
  * expf / tanhf of the fp32 kernel: 2 ulp (CUDA C Programming Guide, mathematical functions), with the add and the
    division of 1 / (1 + exp(-x)): 8 * 2^-24 relative.
  * a function f of an input known within x +- e: sup |f'| over that interval times e (mean value theorem).
  * every fp32 operation of the epilogues: 2^-24 relative per operation.
  * an activation the kernel rounds to bf16 for the next GEMM may land one bf16 ulp away from the reference's
    rounding where the reference value lies within its bound of a rounding tie.  The kernel's operand lies between
    the roundings of (value - bound) and (value + bound) (rounding is monotone); that spread is carried on.
"""
import torch

F64 = torch.float64
U = 2.0 ** -24                   # fp32 unit roundoff
ACC = 2.0 ** -22                 # per-term accumulation bound (4 gamma_K / K)
TANH_APPROX = 2.0 ** -10.987     # tanh.approx.f32, maximum relative error (PTX ISA)
LIBM = 8 * U                     # expf / tanhf at 2 ulp + the surrounding fp32 roundings

KEYS = ("fc1.weight", "fc1.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh", "fc2.0.weight",
        "fc2.0.bias", "fc2.2.weight", "fc2.2.bias")
GEMM_WEIGHTS = ("fc1.weight", "rnn.weight_ih", "rnn.weight_hh", "fc2.0.weight", "fc2.2.weight")


def bf16(x):
    """x -> fp32 -> bf16 (round to nearest even) -> float64"""
    return x.to(torch.float32).to(torch.bfloat16).to(F64)


def bf16_bits_rule(u):
    """The host packer's rule on fp32 bit patterns (uint32 numpy array) -> bf16 bit patterns: inf / NaN truncated,
    otherwise u += 0x7FFF + ((u >> 16) & 1), keep the top 16 bits."""
    import numpy as np
    u = np.asarray(u, dtype=np.uint64)
    special = (u & 0x7F800000) == 0x7F800000
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    return np.where(special, u >> 16, r).astype(np.uint16)


def _sup_slope(x, e, kind):
    """sup |f'| over [x - e, x + e] for f = sigmoid or tanh: the slope at the point of the interval nearest 0"""
    y = torch.minimum(torch.maximum(torch.zeros_like(x), x - e), x + e)
    if kind == "sigmoid":
        s = torch.sigmoid(y)
        return s * (1 - s)
    return 1 - torch.tanh(y) ** 2


class PolicyRef:
    """The agent network of one policy in float64 with the bounds of one kernel (precision "bf16" or "fp32")."""

    def __init__(self, state_dict, n_agents, obs_dim=4, n_actions=3, last_action=True, reuse_network=True, feat_dim=0,
                 precision="bf16", device="cpu"):
        if precision not in ("bf16", "fp32"):
            raise ValueError(precision)
        self.n_agents, self.obs_dim, self.n_actions = int(n_agents), int(obs_dim), int(n_actions)
        self.last_action, self.reuse, self.feat_dim, self.precision = bool(last_action), bool(reuse_network), int(feat_dim), precision
        self.in_dim = self.feat_dim + self.obs_dim + (self.n_actions if last_action else 0) + (self.n_agents if reuse_network else 0)
        self.device = torch.device(device)
        w = {}
        for k in KEYS:
            v = torch.as_tensor(state_dict[k]).detach().to(torch.float32).to(self.device).to(F64)
            w[k] = bf16(v) if (precision == "bf16" and k in GEMM_WEIGHTS) else v
        self.w, self.wa = w, {k: v.abs() for k, v in w.items()}
        if w["fc1.weight"].shape != (64, self.in_dim):
            raise ValueError("fc1.weight is %s, expected (64, %d)" % (tuple(w["fc1.weight"].shape), self.in_dim))

    def _op(self, x, e):
        """the kernel's GEMM operand of a value known within x +- e: (reference operand, largest deviation of the kernel's)"""
        if self.precision == "fp32":
            return x, e
        r = bf16(x)
        return r, torch.maximum(bf16(x + e) - r, r - bf16(x - e))

    def _lin(self, x, dx, key, k_terms):
        """x @ W^T + b and its bound (accumulation of k_terms + operand deviations dx)"""
        W, Wa, b = self.w[key + ".weight"], self.wa[key + ".weight"], self.w[key + ".bias"]
        y = x @ W.T + b
        e = k_terms * ACC * (x.abs() @ Wa.T + b.abs())
        if dx is not None:
            e = e + dx @ Wa.T
        return y, e

    def inputs(self, obs, last_action=None, feat=None):
        """[rows, in_dim] float64 fc1 input row as the kernel forms it: [feat of the row's env ||] obs || last-action
        one-hot (255 = none) || agent-id one-hot; rounded to bf16 in bf16 mode"""
        obs = obs.reshape(-1, self.obs_dim).to(self.device)
        R = obs.shape[0]
        parts = []
        if self.feat_dim:
            parts.append(feat.reshape(-1, self.feat_dim).to(self.device).to(F64).repeat_interleave(self.n_agents, 0))
        parts.append(obs.to(F64))
        if self.last_action:
            la = torch.full((R,), 255, dtype=torch.long, device=self.device) if last_action is None else \
                last_action.reshape(-1).to(self.device).long()
            parts.append((la[:, None] == torch.arange(self.n_actions, device=self.device)).to(F64))
        if self.reuse:
            ids = torch.arange(R, device=self.device) % self.n_agents
            parts.append((ids[:, None] == torch.arange(self.n_agents, device=self.device)).to(F64))
        x = torch.cat(parts, 1)
        return bf16(x) if self.precision == "bf16" else x

    def hidden(self, x, h_in, with_flips=False):
        """stage (a): the new hidden state of fc1 -> ReLU -> GRUCell from the input rows ``x`` (``inputs()``) and the
        fp32 hidden state ``h_in`` [rows, 64] the kernel read.  Returns (h, bound), both [rows, 64] float64, and with
        ``with_flips`` also a [rows] bool: the rows whose bound holds a bf16 flip allowance of x1."""
        w = self.w
        h = h_in.reshape(-1, 64).to(self.device).to(F64)
        hop, dh = self._op(h, torch.zeros_like(h))
        y1, e1 = self._lin(x, None, "fc1", self.in_dim + 1)
        e1 = e1 + U * y1.abs()                                                   # + bias, one fp32 add
        x1, dx1 = self._op(torch.relu(y1), e1)
        Wi, Wh, Wia, Wha = w["rnn.weight_ih"], w["rnn.weight_hh"], self.wa["rnn.weight_ih"], self.wa["rnn.weight_hh"]
        bi, bh = w["rnn.bias_ih"], w["rnn.bias_hh"]
        gi = x1 @ Wi.T
        gh = hop @ Wh.T
        si, sh = x1.abs() @ Wia.T, hop.abs() @ Wha.T                              # sum |terms| of the products
        di = dx1 @ Wia.T                                                         # deviation carried from x1
        # r | z: x1 W_i^T + h W_h^T (+ both biases), 128 products + 2 biases in one accumulator
        pre_rz = gi[:, :128] + gh[:, :128] + bi[:128] + bh[:128]
        e_rz = 130 * ACC * (si[:, :128] + sh[:, :128] + bi[:128].abs() + bh[:128].abs()) + di[:, :128] + 2 * U * pre_rz.abs()
        # n: (x1 W_in^T + b_in) + r * (h W_hn^T + b_hn)
        gin, ghn = gi[:, 128:] + bi[128:], gh[:, 128:] + bh[128:]
        e_gin = 65 * ACC * (si[:, 128:] + bi[128:].abs()) + di[:, 128:]
        e_ghn = 65 * ACC * (sh[:, 128:] + bh[128:].abs())
        pr, pz = pre_rz[:, :64], pre_rz[:, 64:]
        er, ez = e_rz[:, :64], e_rz[:, 64:]
        r, z = torch.sigmoid(pr), torch.sigmoid(pz)
        if self.precision == "bf16":
            # fmaf(0.5, tanh.approx(0.5 x), 0.5): the approximation's relative error on |tanh| <= |tanh(x/2)| + e/2
            fr = 0.5 * TANH_APPROX * torch.clamp(torch.tanh(0.5 * pr).abs() + 0.5 * er, max=1) + U
            fz = 0.5 * TANH_APPROX * torch.clamp(torch.tanh(0.5 * pz).abs() + 0.5 * ez, max=1) + U
        else:
            fr, fz = LIBM * r + U, LIBM * z + U
        er = _sup_slope(pr, er, "sigmoid") * er + fr
        ez = _sup_slope(pz, ez, "sigmoid") * ez + fz
        pn = gin + r * ghn
        en = e_gin + r * e_ghn + ghn.abs() * er + er * e_ghn + 4 * U * (gin.abs() + (r * ghn).abs())
        n = torch.tanh(pn)
        fn = (TANH_APPROX if self.precision == "bf16" else LIBM) * torch.clamp(n.abs() + en, max=1) + U
        en = _sup_slope(pn, en, "tanh") * en + fn
        h_new = (1 - z) * n + z * h
        e_h = (1 - z) * en + (n - h).abs() * ez + ez * en + 4 * U * (((1 - z) * n).abs() + (z * h).abs()) + U
        if with_flips:
            return h_new, e_h, self._flipped(dx1, e1)
        return h_new, e_h

    def q(self, h_out, with_flips=False):
        """stage (b): the action values of fc2.0 -> ReLU -> fc2.2 on the hidden state ``h_out`` the kernel wrote.
        Returns (q, bound), both [rows, n_actions] float64, and with ``with_flips`` the [rows] of ``hidden()`` for f."""
        h = h_out.reshape(-1, 64).to(self.device).to(F64)
        hop, _ = self._op(h, torch.zeros_like(h))
        y, e = self._lin(hop, None, "fc2.0", 65)
        e = e + U * y.abs()
        f, df = self._op(torch.relu(y), e)
        q, eq = self._lin(f, df, "fc2.2", 65)
        if with_flips:
            return q, eq + U * q.abs(), self._flipped(df, e)
        return q, eq + U * q.abs()

    def _flipped(self, dev, e):
        """rows where some operand's deviation ``dev`` is a bf16 flip allowance (one bf16 ulp, 2^-8 relative) rather than
        its own error bound ``e`` carried on (a ReLU zero, whose kernel value may be any bf16 in [0, e]: dev ~ e).  In
        fp32 mode every deviation is the carried bound, so no row counts."""
        if self.precision == "fp32":
            return torch.zeros(dev.shape[0], dtype=torch.bool, device=dev.device)
        return (dev > 2 * e).any(1)


def bound_ratio(err, bound):
    """|err| / bound per element, and +inf wherever that is not a finite, ordered comparison (a NaN or infinite error
    or bound), so that a kernel that writes NaN or inf fails a check instead of hiding behind a NaN-propagating max"""
    a = err.abs()
    r = torch.where(torch.isfinite(a) & torch.isfinite(bound), a / bound, torch.full_like(a, float("inf")))
    return torch.nan_to_num(r, nan=float("inf"))


def assert_within(stage, precision, err, bound, where="", worst=None, flipped=None):
    """AssertionError unless |err| <= bound everywhere (``bound_ratio``).  ``worst``: a dict that keeps the largest ratio
    per (stage, precision) and, where ``flipped`` [rows] is given, per (stage, precision, "no flip") over the rows
    whose bound holds no bf16 flip allowance (those measure the accumulation and tanh.approx terms alone)."""
    ratio = bound_ratio(err, bound)
    v = ratio.max().item() if ratio.numel() else 0.0
    if worst is not None:
        worst[(stage, precision)] = max(worst.get((stage, precision), 0.0), v)
        if flipped is not None and bool((~flipped).any()):
            key = (stage, precision, "no flip")
            worst[key] = max(worst.get(key, 0.0), ratio[~flipped].max().item())
    if not v <= 1:
        i = int(ratio.reshape(-1).argmax())
        r, c = divmod(i, ratio.shape[1])
        raise AssertionError("%s: stage (%s) row %d col %d: |error| %.4g, bound %.4g (ratio %.3g)"
                             % (where, stage, r, c, err.reshape(-1)[i].abs().item(), bound.reshape(-1)[i].item(), v))


def check_stages(ref, obs, last, h_in, h_out, q, acts, avail=None, feat=None, greedy=True, where="", worst=None):
    """Stages (a)-(c) of a kernel call on every row, each on the kernel's own input to that stage: (a) ``h_out``
    against ``ref.hidden`` of (obs, last, feat, h_in), (b) ``q`` against ``ref.q(h_out)``, (c) ``acts`` against
    ``greedy(q, avail)`` exactly.  Device-agnostic; works in chunks of whole envs so that float64 temporaries of the
    large shapes stay ~1 GB.  Raises AssertionError on the first stage that fails."""
    n = ref.n_agents
    R = h_out.numel() // 64
    step = n * max(1, (1 << 17) // n)
    for r0 in range(0, R, step):
        r1 = min(R, r0 + step)
        sl = slice(r0, r1)
        x = ref.inputs(obs.reshape(R, -1)[sl], last.reshape(-1)[sl] if last is not None else None,
                       feat.reshape(R // n, -1)[r0 // n:r1 // n] if feat is not None else None)
        h, eh, fl = ref.hidden(x, h_in.reshape(R, 64)[sl], with_flips=True)
        assert_within("a", ref.precision, h_out.reshape(R, 64)[sl].to(h.device).double() - h, eh, "%s rows %d.." % (where, r0), worst, fl)
        qk = q.reshape(R, -1)[sl].to(h.device)
        qr, eq, fl = ref.q(h_out.reshape(R, 64)[sl], with_flips=True)
        assert_within("b", ref.precision, qk.double() - qr, eq, "%s rows %d.." % (where, r0), worst, fl)
        if greedy:
            want = greedy_rule(qk, avail.reshape(R, -1)[sl] if avail is not None else None)
            got = acts.reshape(-1)[sl].to(h.device).long()
            if not torch.equal(got, want):
                i = int((got != want).nonzero()[0])
                raise AssertionError("%s: stage (c) row %d: action %d, the rule gives %d on the kernel's q %s"
                                     % (where, r0 + i, got[i], want[i], qk[i].tolist()))


def random_state_dict(in_dim, n_actions, seed, kind="default"):
    """Weights of the reference's RNN class: torch's default init ("default"), or scaled ("scaled") so that the gates
    saturate and the action values reach a few hundred, like the shipped qmix model (|q| up to ~300)."""
    torch.manual_seed(seed)
    fc1, rnn = torch.nn.Linear(in_dim, 64), torch.nn.GRUCell(64, 64)
    fc2 = torch.nn.Sequential(torch.nn.Linear(64, 64), torch.nn.ReLU(), torch.nn.Linear(64, n_actions))
    sd = {"fc1." + k: v for k, v in fc1.state_dict().items()}
    sd.update({"rnn." + k: v for k, v in rnn.state_dict().items()})
    sd.update({"fc2." + k: v for k, v in fc2.state_dict().items()})
    if kind == "scaled":
        scale = {"fc1.weight": 4, "fc1.bias": 4, "rnn.weight_ih": 4, "rnn.weight_hh": 4, "fc2.0.weight": 8, "fc2.0.bias": 8,
                 "fc2.2.weight": 60, "fc2.2.bias": 60}
        sd = {k: v * scale.get(k, 1) for k, v in sd.items()}
    return {k: v.detach().clone() for k, v in sd.items()}


def greedy_rule(q, avail=None):
    """stage (c): agent/agent.py:66-75 with evaluate: unavailable action values -inf, the first maximum (torch.argmax),
    action 0 for a row with no available action"""
    qm = q.to(F64).clone()
    if avail is not None:
        qm[avail.reshape(qm.shape).to(qm.device) == 0] = -float("inf")
    return qm.argmax(-1)


def conv_features(maps, sd, dim_1, kernel_size_1, stride_1, dim_2, kernel_size_2, stride_2, padding_2, **_):
    """network/base_net.py:10-20,31-41: maps [E, M, M] (row-major belief maps) -> conv2d -> ReLU -> conv2d -> ReLU ->
    Linear in float64, with the bound of fp32 accumulation (flight_conv_kernel: fp32 FMAs, any order).
    Returns (feat, bound), both [E, out_dim]."""
    import torch.nn.functional as Fn
    dev = maps.device
    g = lambda k: torch.as_tensor(sd[k]).detach().to(torch.float32).to(dev).to(F64)
    w1, b1, w2, b2, wl, bl = g("conv.0.weight"), g("conv.0.bias"), g("conv.2.weight"), g("conv.2.bias"), g("linear.weight"), g("linear.bias")
    m = maps.to(F64).unsqueeze(1)
    y1 = Fn.conv2d(m, w1, b1, stride=stride_1)
    e1 = (kernel_size_1 ** 2 + 1) * ACC * Fn.conv2d(m.abs(), w1.abs(), b1.abs(), stride=stride_1)
    a1 = torch.relu(y1)
    y2 = Fn.conv2d(a1, w2, b2, stride=stride_2, padding=padding_2)
    e2 = (dim_1 * kernel_size_2 ** 2 + 1) * ACC * Fn.conv2d(a1.abs(), w2.abs(), b2.abs(), stride=stride_2, padding=padding_2) + \
        Fn.conv2d(e1, w2.abs(), None, stride=stride_2, padding=padding_2)
    a2, e2 = torch.relu(y2).flatten(1), e2.flatten(1)
    feat = a2 @ wl.T + bl
    e = (a2.shape[1] + 1) * ACC * (a2 @ wl.abs().T + bl.abs()) + e2 @ wl.abs().T + U * feat.abs()
    return feat, e
