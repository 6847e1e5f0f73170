"""Batched agents: the reference's RNN agent network (network/base_net.py:5-47, with the optional conv front end of the flight agents) and the
action choice of Agents.choose_action (agent/agent.py:33-97) for every (env, agent) row of a vectorised env at once,
in one kernel launch (csrc/policy.cu, csrc/policy_tc.cuh).  The reference evaluates one (1, in) row per agent per step.

precision "bf16" (the default): the five GEMMs of a 128-row tile run on the tcgen05 tensor cores with bf16 operands,
fp32 accumulators in tensor memory and an fp32 hidden state; "fp32": the CUDA-core kernel that equals the reference's
torch modules to 1e-5.  Input widths up to 256: each kernel has one instantiation for widths <= 32 (the flight agents)
and one for 33..256 (the search agents: (2R-1)^2 + 2 obs values + 4 + n_agents, 239 at 64 agents), chosen by width.
Both are held to a float64 reference with per-element error bounds (oracle/policy_ref.py, tests/test_gpu_policy_reference.py).
alg: "q" = masked argmax / epsilon-greedy (qmix, vdn; dop's actor is the same network class with the actor's weights),
"reinforce" = softmax sampling (agent/agent.py:77-97)."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import CoopSearchError

# RNN.state_dict() key -> cs_policy_weights field
_KEYMAP = {"fc1.weight": "fc1_w", "fc1.bias": "fc1_b", "rnn.weight_ih": "w_ih", "rnn.weight_hh": "w_hh",
           "rnn.bias_ih": "b_ih", "rnn.bias_hh": "b_hh", "fc2.0.weight": "fc2a_w", "fc2.0.bias": "fc2a_b",
           "fc2.2.weight": "fc2b_w", "fc2.2.bias": "fc2b_b"}


class BatchedRNNAgents:
    """``state_dict``: the reference's ``{idx}_rnn_net_params.pkl`` contents (or any mapping with the same keys).
    ``choose_actions(obs)`` = Agents.choose_action for all envs and agents; hidden states and last actions are kept on
    the device between calls (``init_hidden()`` = policy.init_hidden + rollout.py:31)."""

    # conv front end of the `flight` agents: defaults of common/arguments.py:246-265
    CONV_DEFAULTS = dict(map_size=50, dim_1=4, kernel_size_1=4, stride_1=2, dim_2=1, kernel_size_2=3, stride_2=1, padding_2=1,
                         conv_out_dim=16)

    def __init__(self, state_dict, num_envs, n_agents, obs_dim=4, n_actions=3, last_action=True, reuse_network=True,
                 device=None, seed=0, precision=None, alg="q", conv=None):
        """conv: None = args.conv False; True or a dict of the conv arguments (map_size, dim_1, kernel_size_1, stride_1,
        dim_2, kernel_size_2, stride_2, padding_2, conv_out_dim) = the `flight` agents' network: ``state_dict`` then also
        holds conv.0.*, conv.2.*, linear.* and choose_actions() takes the env whose belief maps it reads."""
        if not torch.cuda.is_available():
            raise CoopSearchError("coopsearch_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.num_envs, self.n_agents, self.obs_dim, self.n_actions = int(num_envs), int(n_agents), int(obs_dim), int(n_actions)
        self.seed = int(seed) & 0xFFFFFFFF
        host = {}
        for key, field in _KEYMAP.items():
            if key not in state_dict:
                raise CoopSearchError("state_dict has no %r" % key)
            host[field] = np.ascontiguousarray(torch.as_tensor(state_dict[key]).detach().cpu().numpy(), dtype=np.float32)
        self.conv = None
        if conv:
            self.conv = dict(self.CONV_DEFAULTS)
            if isinstance(conv, dict):
                self.conv.update(conv)
        feat_dim = int(self.conv["conv_out_dim"]) if self.conv else 0
        in_dim = feat_dim + obs_dim + (n_actions if last_action else 0) + (n_agents if reuse_network else 0)
        if host["fc1_w"].shape != (64, in_dim):
            raise CoopSearchError("fc1.weight is %s, expected (64, %d)" % (host["fc1_w"].shape, in_dim))
        cfg = _lib.PolicyCfg(struct_size=C.sizeof(_lib.PolicyCfg), device=self.device.index, n_agents=n_agents, obs_dim=obs_dim,
                             n_actions=n_actions, hidden_dim=64, last_action=int(last_action), reuse_network=int(reuse_network),
                             conv_out_dim=feat_dim)
        w = _lib.PolicyWeights(**{k: v.ctypes.data for k, v in host.items()})
        hp = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_policy_create(C.byref(cfg), C.byref(w), C.byref(hp)), "cs_policy_create")
        self._h = hp
        self.feat = None
        if self.conv:
            ch = {}
            for key, field in (("conv.0.weight", "c1_w"), ("conv.0.bias", "c1_b"), ("conv.2.weight", "c2_w"), ("conv.2.bias", "c2_b"),
                               ("linear.weight", "lin_w"), ("linear.bias", "lin_b")):
                if key not in state_dict:
                    raise CoopSearchError("state_dict has no %r (conv front end)" % key)
                ch[field] = np.ascontiguousarray(torch.as_tensor(state_dict[key]).detach().cpu().numpy(), dtype=np.float32)
            c = self.conv
            ccfg = _lib.PolicyConvCfg(struct_size=C.sizeof(_lib.PolicyConvCfg), map_size=c["map_size"], dim_1=c["dim_1"],
                                      kernel_size_1=c["kernel_size_1"], stride_1=c["stride_1"], dim_2=c["dim_2"],
                                      kernel_size_2=c["kernel_size_2"], stride_2=c["stride_2"], padding_2=c["padding_2"], out_dim=feat_dim)
            cw = _lib.PolicyConvWeights(**{k: v.ctypes.data for k, v in ch.items()})
            with torch.cuda.device(self.device):
                _lib.check(self.lib.cs_policy_set_conv(self._h, C.byref(ccfg), C.byref(cw)), "cs_policy_set_conv")
            self.feat = torch.zeros((self.num_envs, feat_dim), dtype=torch.float32, device=self.device)
        rows = self.num_envs * self.n_agents
        self.hidden = torch.zeros((self.num_envs, self.n_agents, 64), dtype=torch.float32, device=self.device)
        self.q = torch.empty((self.num_envs, self.n_agents, self.n_actions), dtype=torch.float32, device=self.device)
        self.actions = torch.full((self.num_envs, self.n_agents), 255, dtype=torch.uint8, device=self.device)
        self._rows, self._t = rows, 0
        if precision is None:
            precision = "bf16"
        if precision not in ("bf16", "fp32"):
            raise CoopSearchError("precision must be 'bf16' (tensor cores) or 'fp32'")
        if alg not in ("q", "reinforce"):
            raise CoopSearchError("alg must be 'q' (argmax / epsilon-greedy) or 'reinforce' (softmax sampling)")
        self.precision, self.alg = precision, alg
        if precision == "bf16":
            self.kernel_name = "policy_tc_kernel<K1=%d> (tcgen05.mma, bf16 operands, TMEM accumulators)" % (32 if in_dim <= 32 else 256)
        else:
            self.kernel_name = "policy_kernel<S=%d> (fp32, CUDA cores)" % (1 if in_dim <= 32 else 8)

    def init_hidden(self, mask=None):
        """policy.init_hidden(1) + last_action = zeros (rollout.py:31-33) for all envs, or those with mask[e] != 0.
        A device mask (e.g. the terminated flags of an auto-resetting env) is applied without a host synchronisation,
        so the call can be captured in a CUDA graph."""
        if mask is None:
            self.hidden.zero_()
            self.actions.fill_(255)
        else:
            m = torch.as_tensor(mask, device=self.device).bool()
            self.hidden.masked_fill_(m.reshape(m.shape + (1,) * (self.hidden.dim() - m.dim())), 0)
            self.actions.masked_fill_(m.reshape(m.shape + (1,) * (self.actions.dim() - m.dim())), 255)

    def conv_features(self, env=None, prob_map_tiles=None):
        """The conv features of every env's belief map ([E, conv_out_dim], also kept as ``self.feat``), read once per env
        from the flight env's tiled device map -- no [E,n,M*M+4] observation is materialised."""
        if not self.conv:
            raise CoopSearchError("this policy has no conv front end")
        tiles = env.prob_map_tiles if env is not None else prob_map_tiles
        if tiles is None or tiles.dim() != 5 or tiles.shape[0] != self.num_envs:
            raise CoopSearchError("conv_features needs a VecFlightEnv (or its prob_map_tiles [E, tiles, tiles, 4, 4])")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_policy_conv_features(self._h, C.c_void_p(tiles.data_ptr()), int(tiles.shape[1]),
                                                        int(tiles.stride(0)), self.num_envs, C.c_void_p(self.feat.data_ptr()),
                                                        C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                       "cs_policy_conv_features")
        return self.feat

    def choose_actions(self, obs, avail=None, epsilon=0.0, evaluate=True, env=None):
        """obs: [E,n,obs_dim] float32 device tensor (env.get_obs(); for the `flight` variant get_obs(full=False));
        avail: [E,n,A] or None; env: the VecFlightEnv whose belief maps the conv front end reads (conv policies).
        Returns the [E,n] uint8 action tensor (also kept as the next call's last action); ``self.q`` holds the action
        values."""
        if self.conv and env is not None:
            self.conv_features(env)
        obs = obs.contiguous()
        if tuple(obs.shape) != (self.num_envs, self.n_agents, self.obs_dim) or obs.dtype != torch.float32:
            raise CoopSearchError("obs must be float32 [num_envs, n_agents, obs_dim]")
        av = None
        if avail is not None:
            av = avail.to(device=self.device, dtype=torch.uint8).contiguous()
        io = _lib.PolicyIO(rows=self._rows, evaluate=int(bool(evaluate)), epsilon=float(epsilon), seed=self.seed, t=self._t,
                           obs=obs.data_ptr(), last_action=self.actions.data_ptr(), avail=av.data_ptr() if av is not None else None,
                           hidden=self.hidden.data_ptr(), q=self.q.data_ptr(), actions=self.actions.data_ptr(),
                           precision=1 if self.precision == "bf16" else 0, mode=1 if self.alg == "reinforce" else 0,
                           feat=self.feat.data_ptr() if self.feat is not None else None)
        self._t = (self._t + 1) & 0xFFFFFFFF
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cs_policy_act(self._h, C.byref(io), C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)),
                       "cs_policy_act")
        return self.actions

    def __del__(self):
        try:
            if self._h:
                self.lib.cs_policy_destroy(self._h)
                self._h = None
        except Exception:
            pass
