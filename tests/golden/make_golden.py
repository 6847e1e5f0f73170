#!/usr/bin/env python
"""Generates tests/golden/*.npz by running the UNMODIFIED reference envs.

Needs the reference checkout (COOPSEARCH_REFERENCE, else BASELINE.json's reference_path):

    python tests/golden/make_golden.py

Inputs are seeded exactly as SURVEY.md section 8d prescribes:
  * initial targets of env e: ``np.random.seed(10_000 + e)`` then the reference's own
    ``reset()`` (MT19937 normals, env/flight_env_easy.py:107-108);
  * actions: ``np.random.default_rng(1234).integers(0, 3, size=(T, E, n))``;
  * detection uniforms: keyed Philox draw, seed 42, key (env_id, episode, t, i, j)
    (oracle/refharness.py: KeyedDraws).
The fixtures are what the oracle (tests/test_oracle_golden.py) and the CUDA path
(tests/test_gpu_*.py) are pinned against.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import refharness as rh  # noqa: E402
import contextlib as _ctx, io as _io  # noqa: E402
rh.contextlib, rh.io = _ctx, _io

OUT = os.path.dirname(os.path.abspath(__file__))
SEED = 42
TARGETS_TXT = os.path.join(rh.REFERENCE_ROOT, "flight_targets.txt")


def found_mask(env):
    return sum(1 << j for j, t in enumerate(env.target_list) if t.find)


def run_flight(cls_name, n_agents, agent_mode, E, T, env_id_base, target_mode=0, second_episode=0,
               map_steps=(), **over):
    ref = rh.import_reference()
    cls = ref[cls_name]
    envname = "flight_easy" if cls_name == "FlightSearchEnvEasy" else "flight"
    circle = rh.load_targets_reference_semantics(TARGETS_TXT)
    args = rh.make_args(envname, n_agents=n_agents, agent_mode=agent_mode, target_mode=target_mode, **over)
    m = args.target_num
    S = 4 * n_agents + 3 * m
    actions = np.random.default_rng(1234).integers(0, 3, size=(T, E, n_agents), dtype=np.uint8)
    has_map = cls_name == "FlightSearchEnv"
    g = dict(
        tgt_xy=np.zeros((E, m, 2)), init_xy=np.zeros((E, n_agents, 2)), init_yaw=np.zeros((E, n_agents)),
        init_found=np.zeros(E, np.uint32), init_win=np.zeros(E, np.uint8),
        init_obs=np.zeros((E, n_agents, 4)), init_state=np.zeros((E, S)),
        actions=actions,
        xy=np.zeros((T, E, n_agents, 2)), yaw=np.zeros((T, E, n_agents)), out=np.zeros((T, E, n_agents), np.uint8),
        found=np.zeros((T, E), np.uint32), reward=np.zeros((T, E)), terminated=np.zeros((T, E), np.uint8),
        win=np.zeros((T, E), np.uint8), target_find=np.zeros((T, E), np.int32), time_step=np.zeros((T, E), np.int32),
        obs=np.zeros((T, E, n_agents, 4)), state=np.zeros((T, E, S)),
        n_steps=np.zeros(E, np.int32), n_draws=np.zeros(E, np.int64),
    )
    if has_map:
        g["map_steps"] = np.array(map_steps, np.int32)
        g["init_map"] = np.zeros((E, args.map_size, args.map_size))
        g["maps"] = np.zeros((len(map_steps), E, args.map_size, args.map_size))
        g["final_map"] = np.zeros((E, args.map_size, args.map_size))
        if second_episode:
            g["ep2_tgt_xy"] = np.zeros((E, m, 2))
            g["ep2_actions"] = np.random.default_rng(4321).integers(0, 3, size=(second_episode, E, n_agents), dtype=np.uint8)
            g["ep2_map"] = np.zeros((E, args.map_size, args.map_size))
            g["ep2_found"] = np.zeros((second_episode, E), np.uint32)
            g["ep2_reward"] = np.zeros((second_episode, E))
    for e in range(E):
        env_id = env_id_base + e
        draws = rh.KeyedDraws(SEED, env_id, episode=0)
        np.random.seed(10_000 + env_id)
        with draws:
            draws.t = 0
            env = rh.quiet(cls, args, circle)           # ctor calls reset(init=True)
        g["tgt_xy"][e] = np.array(env.target_pos, dtype=np.float64)
        g["init_xy"][e] = np.array(env.agent_pos, dtype=np.float64)
        g["init_yaw"][e] = np.array(env.agent_yaw, dtype=np.float64)
        g["init_found"][e] = found_mask(env)
        g["init_win"][e] = int(env.win_flag)
        if has_map:
            g["init_map"][e] = env.prob_map
            g["init_obs"][e] = env.get_obs()[:, -4:]
        else:
            g["init_obs"][e] = env.get_obs()
        g["init_state"][e] = env.get_state()
        done = False
        for t in range(T):
            if not done:
                with draws:
                    draws.t = t + 1
                    r, term, win = env.step([int(a) for a in actions[t, e]])
                g["n_steps"][e] = t + 1
                done = bool(term)
            else:
                r, term = 0.0, True            # masked no-op after termination (batched API contract)
            g["xy"][t, e] = np.array(env.agent_pos, dtype=np.float64)
            g["yaw"][t, e] = np.array(env.agent_yaw, dtype=np.float64)
            g["out"][t, e] = np.array(env.out_flag)
            g["found"][t, e] = found_mask(env)
            g["reward"][t, e] = r
            g["terminated"][t, e] = int(term)
            g["win"][t, e] = int(env.win_flag)
            g["target_find"][t, e] = env.target_find
            g["time_step"][t, e] = env.time_step
            g["obs"][t, e] = env.get_obs()[:, -4:]
            g["state"][t, e] = env.get_state()
            if has_map and (t + 1) in map_steps:
                g["maps"][list(map_steps).index(t + 1), e] = env.prob_map
        if has_map:
            g["final_map"][e] = env.prob_map
            if second_episode:
                # reset() WITHOUT init: the map must survive (flight_env.py:84-86)
                draws2 = rh.KeyedDraws(SEED, env_id, episode=1)
                np.random.seed(20_000 + env_id)
                with draws2:
                    draws2.t = 0
                    env.reset()
                g["ep2_tgt_xy"][e] = np.array(env.target_pos, dtype=np.float64)
                for t in range(second_episode):
                    with draws2:
                        draws2.t = t + 1
                        r, term, win = env.step([int(a) for a in g["ep2_actions"][t, e]])
                    g["ep2_found"][t, e] = found_mask(env)
                    g["ep2_reward"][t, e] = r
                g["ep2_map"][e] = env.prob_map
        g["n_draws"][e] = draws.n_draws
    g["meta"] = np.array([n_agents, m, args.map_size, args.view_range, args.time_limit, agent_mode, target_mode,
                          env_id_base, SEED], np.int64)
    g["fmeta"] = np.array([args.agent_velocity, args.detect_prob, args.safe_dist, args.force_dist], np.float64)
    return g


def run_search(n_agents, target_num, map_size, view_range, agent_mode, target_mode, E, T, env_id_base):
    ref = rh.import_reference()
    cls = ref["SearchEnv"]
    args = rh.make_args("search", n_agents=n_agents, target_num=target_num, map_size=map_size,
                        view_range=view_range, agent_mode=agent_mode, target_mode=target_mode)
    S = 2 * view_range - 1
    rng = np.random.default_rng(1234)
    g = dict(
        cells=np.zeros((E, target_num, 2), np.int32), init_pos=np.zeros((E, n_agents, 2), np.int32),
        init_obs=np.zeros((E, n_agents, S * S + 2)), init_state=np.zeros((E, 2 * map_size ** 2), np.uint8),
        init_freq=np.zeros((E, map_size, map_size), np.int32),
        actions=np.zeros((T, E, n_agents), np.uint8), avail=np.zeros((T, E, n_agents, 4), np.uint8),
        pos=np.zeros((T, E, n_agents, 2), np.int32), reward=np.zeros((T, E)), terminated=np.zeros((T, E), np.uint8),
        target_find=np.zeros((T, E), np.int32), obs=np.zeros((T, E, n_agents, S * S + 2), np.float32),
        state=np.zeros((T, E, 2 * map_size ** 2), np.uint8), freq=np.zeros((E, map_size, map_size), np.int32),
        found=np.zeros((T, E, target_num), np.uint8), n_steps=np.zeros(E, np.int32),
    )
    for e in range(E):
        np.random.seed(10_000 + env_id_base + e)
        env = rh.quiet(cls, args)
        g["cells"][e] = np.array([t.pos for t in env.target_list])
        g["init_pos"][e] = np.array(env.agent_pos)
        g["init_obs"][e] = rh.quiet(env.get_obs)
        g["init_state"][e] = env.get_state().astype(np.uint8)
        g["init_freq"][e] = env.freq_map.astype(np.int32)
        done = False
        for t in range(T):
            av = np.array([env.get_avail_agent_actions(i) for i in range(n_agents)])
            g["avail"][t, e] = av.astype(np.uint8)
            act = np.array([rng.choice(np.nonzero(av[i])[0]) for i in range(n_agents)], np.uint8)
            g["actions"][t, e] = act
            if not done:
                r, term, _ = env.step([int(a) for a in act])
                g["n_steps"][e] = t + 1
                done = bool(term)
            else:
                r, term = 0.0, True
            g["pos"][t, e] = np.array(env.agent_pos)
            g["reward"][t, e] = r
            g["terminated"][t, e] = int(term)
            g["target_find"][t, e] = env.target_find
            g["obs"][t, e] = rh.quiet(env.get_obs)
            g["state"][t, e] = env.get_state().astype(np.uint8)
            g["found"][t, e] = np.array([int(x.find) for x in env.target_list], np.uint8)
        g["freq"][e] = env.freq_map.astype(np.int32)
    g["meta"] = np.array([n_agents, target_num, map_size, view_range, agent_mode, target_mode, env_id_base], np.int64)
    return g


def run_rollout(n_agents, agent_mode, episodes, env_id, seed0):
    """Episode batches produced by the reference's own RolloutWorker.generate_episode (common/rollout.py:22-141) with
    the reference's Agents facade and alg=random (agent/agent.py:34-36) on FlightSearchEnvEasy."""
    import types as _t
    ref = rh.import_reference()
    with rh.contextlib.redirect_stdout(rh.io.StringIO()):
        from common.rollout import RolloutWorker
        from agent.agent import Agents
    circle = rh.load_targets_reference_semantics(TARGETS_TXT)
    args = rh.make_args("flight_easy", n_agents=n_agents, agent_mode=agent_mode)
    draws = rh.KeyedDraws(SEED, env_id, episode=0)
    np.random.seed(seed0)
    with draws:
        draws.t = 0
        env = rh.quiet(ref["FlightSearchEnvEasy"], args, circle)
    info = env.get_env_info()
    for k, v in info.items():
        setattr(args, k, v)
    args.alg, args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = "random", 0, 0, 0, "step"
    args.last_action, args.reuse_network, args.cuda, args.evaluate_epoch = True, True, False, 20
    agents = rh.quiet(Agents, env, args)
    worker = rh.quiet(RolloutWorker, env, agents, args)
    captured = []
    orig_reset, orig_step = env.reset, env.step

    def reset(init=False):
        draws.t = 0
        draws.episode += 1
        out = orig_reset(init)
        captured.append(np.array(env.target_pos, dtype=np.float64))
        return out

    def step(actions):
        draws.t = env.time_step + 1
        return orig_step(actions)
    env.reset, env.step = reset, step
    g = {}
    T, S = info["episode_limit"], info["state_shape"]
    keys = ["o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated"]
    for k in keys:
        g[k] = []
    g["episode_reward"], g["win_tag"], g["targets_find"] = [], [], []
    with draws:
        for ep in range(episodes):
            np.random.seed(seed0 + 1 + ep)
            episode, rew, win, tf = worker.generate_episode(ep)
            for k in keys:
                g[k].append(episode[k][0])
            g["episode_reward"].append(rew); g["win_tag"].append(int(bool(win))); g["targets_find"].append(tf)
    out = {k: np.array(v) for k, v in g.items()}
    out["tgt_xy"] = np.array(captured)
    out["meta"] = np.array([n_agents, args.target_num, args.map_size, args.view_range, T, agent_mode, 0, env_id, SEED], np.int64)
    out["fmeta"] = np.array([args.agent_velocity, args.detect_prob, args.safe_dist, args.force_dist], np.float64)
    # float32 is what the batched writer produces; keep the fixture small
    for k in ("o", "s", "o_next", "s_next"):
        out[k] = out[k].astype(np.float32)
    for k in ("u", "avail_u", "avail_u_next", "u_onehot", "padded", "terminated"):
        out[k] = out[k].astype(np.uint8)
    return out


def run_policy(model_dir, n_agents, steps=6, rows_envs=5):
    """The reference's own agent network (network/base_net.py: RNN) with the weights it ships (model/<dir>/*_rnn_net_params.pkl),
    evaluated the way Agents.choose_action does (agent/agent.py:38-75, evaluate=True): inputs = obs || last action one-hot ||
    agent id one-hot, one (1, in) row at a time, hidden state carried per agent."""
    import glob
    import types as _t
    import torch
    rh.import_reference()
    from network.base_net import RNN
    path = sorted(glob.glob(os.path.join(rh.REFERENCE_ROOT, "model", model_dir, "*_rnn_net_params.pkl")))[0]
    sd = torch.load(path, map_location="cpu")
    n_actions, obs_dim = 3, 4
    in_dim = obs_dim + n_actions + n_agents
    args = _t.SimpleNamespace(conv=False, rnn_hidden_dim=64, n_actions=n_actions)
    net = RNN(in_dim, args)
    net.load_state_dict(sd)
    net.eval()
    rng = np.random.default_rng(11)
    E = rows_envs
    obs = rng.uniform(-1, 1, size=(steps, E, n_agents, obs_dim)).astype(np.float32)
    hidden = torch.zeros(E, n_agents, 64)
    last = np.zeros((E, n_agents, n_actions), np.float32)
    qs, hs, acts = [], [], []
    with torch.no_grad():
        for t in range(steps):
            q_t = np.zeros((E, n_agents, n_actions), np.float32)
            a_t = np.zeros((E, n_agents), np.uint8)
            for e in range(E):
                for a in range(n_agents):
                    agent_id = np.zeros(n_agents, np.float32); agent_id[a] = 1.0
                    inputs = np.hstack((obs[t, e, a], last[e, a], agent_id))                     # agent.py:44-47
                    q, h = net(torch.tensor(inputs, dtype=torch.float32).unsqueeze(0), hidden[e, a].unsqueeze(0))
                    hidden[e, a] = h[0]
                    q_t[e, a] = q[0].numpy()
                    act = int(torch.argmax(q))                                                    # agent.py:71-72
                    a_t[e, a] = act
                    last[e, a] = 0.0; last[e, a, act] = 1.0                                       # rollout.py:57-62
            qs.append(q_t); hs.append(hidden.numpy().copy()); acts.append(a_t)
    out = {"obs": obs, "q": np.array(qs), "hidden": np.array(hs), "actions": np.array(acts),
           "meta": np.array([n_agents, obs_dim, n_actions], np.int64)}
    for k, v in sd.items():
        out["w:" + k] = v.numpy().astype(np.float32)
    return out


def run_policy_conv(model_dir, n_agents, steps=4, rows_envs=4):
    """The reference's agent network WITH the conv front end (network/base_net.py:10-20,31-41, args of
    common/arguments.py:246-265) and the `flight` weights it ships, evaluated the way Agents.choose_action does on
    flight's observation rows: obs = prob_map.ravel() || (x^, y^, cos, sin) per agent (flight_env.py:223-230), then
    || last action one-hot || agent id one-hot (agent.py:44-47).  The maps mimic belief maps: 0.5 background, decayed
    patches, a few cells at 1."""
    import glob
    import types as _t
    import torch
    rh.import_reference()
    from network.base_net import RNN
    path = sorted(glob.glob(os.path.join(rh.REFERENCE_ROOT, "model", model_dir, "*_rnn_net_params.pkl")))[0]
    sd = torch.load(path, map_location="cpu")
    n_actions, obs_dim, M = 3, 4, 50
    args = _t.SimpleNamespace(conv=True, rnn_hidden_dim=64, n_actions=n_actions, map_size=M, dim_1=4, kernel_size_1=4, stride_1=2,
                              dim_2=1, kernel_size_2=3, stride_2=1, padding_2=1, conv_out_dim=16)
    in_dim = 16 + obs_dim + n_actions + n_agents                       # main.py / agent.py: conv_out_dim + obs_shape + ...
    net = RNN(in_dim, args)
    net.load_state_dict(sd)
    net.eval()
    rng = np.random.default_rng(13)
    E = rows_envs
    maps = np.full((steps, E, M, M), 0.5, np.float32)
    for t in range(steps):
        for e in range(E):
            for _ in range(3):
                i0, j0 = rng.integers(0, M - 12, size=2)
                maps[t, e, i0:i0 + 12, j0:j0 + 12] *= rng.uniform(1e-4, 1.0, size=(12, 12)).astype(np.float32)
            for _ in range(4):
                maps[t, e, rng.integers(0, M), rng.integers(0, M)] = 1.0
    sa = rng.uniform(-1, 1, size=(steps, E, n_agents, obs_dim)).astype(np.float32)
    hidden = torch.zeros(E, n_agents, 64)
    last = np.zeros((E, n_agents, n_actions), np.float32)
    qs, hs, acts, feats = [], [], [], []
    with torch.no_grad():
        for t in range(steps):
            q_t = np.zeros((E, n_agents, n_actions), np.float32)
            a_t = np.zeros((E, n_agents), np.uint8)
            f_t = np.zeros((E, 16), np.float32)
            for e in range(E):
                pm = torch.from_numpy(maps[t, e]).reshape(1, 1, M, M)
                f_t[e] = net.linear(net.conv(pm).reshape(1, -1))[0].numpy()
                for a in range(n_agents):
                    agent_id = np.zeros(n_agents, np.float32); agent_id[a] = 1.0
                    obs_row = np.concatenate((maps[t, e].ravel(), sa[t, e, a]))                   # flight_env.py:226-229
                    inputs = np.hstack((obs_row, last[e, a], agent_id))                           # agent.py:44-47
                    q, h = net(torch.tensor(inputs, dtype=torch.float32).unsqueeze(0), hidden[e, a].unsqueeze(0))
                    hidden[e, a] = h[0]
                    q_t[e, a] = q[0].numpy()
                    act = int(torch.argmax(q))
                    a_t[e, a] = act
                    last[e, a] = 0.0; last[e, a, act] = 1.0
            qs.append(q_t); hs.append(hidden.numpy().copy()); acts.append(a_t); feats.append(f_t)
    out = {"maps": maps, "obs": sa, "q": np.array(qs), "hidden": np.array(hs), "actions": np.array(acts), "feat": np.array(feats),
           "meta": np.array([n_agents, obs_dim, n_actions, M], np.int64)}
    for k, v in sd.items():
        out["w:" + k] = v.numpy().astype(np.float32)
    return out


def run_spread(n_agents, target_num, map_size, E, T, env_id_base):
    """SimpleSpreadEnv (env/simple_spread.py): reset() draws the layout from the seeded MT19937 stream, then T steps under
    uniform-random actions.  Everything is stored in float64 as the reference returns it."""
    ref = rh.import_reference()
    cls = ref["SimpleSpreadEnv"]
    args = rh.make_args("simple_spread", n_agents=n_agents, target_num=target_num, map_size=map_size)
    obs_shape = 2 + (n_agents - 1) * 2 + target_num * 4
    rng = np.random.default_rng(4321)
    g = dict(tgt=np.zeros((E, target_num, 2)), agents0=np.zeros((E, n_agents, 2)),
             init_obs=np.zeros((E, n_agents, obs_shape)), init_state=np.zeros((E, 2 * n_agents + 2 * target_num)),
             actions=np.zeros((T, E, n_agents), np.uint8), reward=np.zeros((T, E)), terminated=np.zeros((T, E), np.uint8),
             obs=np.zeros((T, E, n_agents, obs_shape)), state=np.zeros((T, E, 2 * n_agents + 2 * target_num)),
             agents=np.zeros((T, E, n_agents, 2)), occupied=np.zeros((T, E, target_num), np.uint8))
    for e in range(E):
        np.random.seed(20_000 + env_id_base + e)
        env = rh.quiet(cls, args)
        env.reset()
        g["tgt"][e] = np.array([t.pos for t in env.target_list])
        g["agents0"][e] = np.array([a.pos for a in env.agent_list])
        g["init_obs"][e] = env.get_obs()
        g["init_state"][e] = env.get_state()
        for t in range(T):
            act = rng.integers(0, 5, size=n_agents).astype(np.uint8)
            g["actions"][t, e] = act
            r, term, _ = env.step([int(a) for a in act])
            g["reward"][t, e] = r
            g["terminated"][t, e] = int(term)
            g["obs"][t, e] = env.get_obs()
            g["state"][t, e] = env.get_state()
            g["agents"][t, e] = np.array([a.pos for a in env.agent_list])
            g["occupied"][t, e] = np.array(env.occupied, np.uint8)
    g["meta"] = np.array([n_agents, target_num, map_size, env_id_base], np.int64)
    g["info"] = np.array([env.get_env_info()[k] for k in ("n_actions", "state_shape", "obs_shape", "episode_limit")], np.int64)
    return g


def compact_anchor(g):
    """A wide run reduced to what a device test needs: the inputs (targets, actions), every discrete per-step output, the
    final float64 positions / headings and a float32 observation / state checkpoint every 50 steps."""
    keep = {k: g[k] for k in ("tgt_xy", "init_xy", "init_yaw", "init_found", "actions", "found", "terminated", "win", "time_step", "out",
                              "n_steps", "meta", "fmeta")}
    keep["reward"] = g["reward"].astype(np.float32)
    keep["final_xy"], keep["final_yaw"] = g["xy"][-1], g["yaw"][-1]
    keep["chk_steps"] = np.arange(49, g["obs"].shape[0], 50, dtype=np.int32)
    keep["chk_obs"] = g["obs"][49::50].astype(np.float32)
    keep["chk_state"] = g["state"][49::50].astype(np.float32)
    keep["chk_xy"] = g["xy"][49::50]
    return keep


def thin(g, keep_every, keys=("obs", "state")):
    """obs/state are derivable from xy/yaw/found; keep every k-th step to bound fixture size."""
    for k in keys:
        g[k] = g[k][keep_every - 1::keep_every].copy()
    g["thin"] = np.array([keep_every], np.int32)
    return g


def main():
    os.makedirs(OUT, exist_ok=True)
    jobs = {
        # name: (generator, kwargs)
        "easy_1a_am0": lambda: thin(run_flight("FlightSearchEnvEasy", 1, 0, E=6, T=200, env_id_base=0), 10),
        "easy_3a_am0": lambda: thin(run_flight("FlightSearchEnvEasy", 3, 0, E=8, T=200, env_id_base=100), 10),
        "easy_3a_am1": lambda: thin(run_flight("FlightSearchEnvEasy", 3, 1, E=4, T=200, env_id_base=150), 10),
        "easy_5a_am2": lambda: thin(run_flight("FlightSearchEnvEasy", 5, 2, E=6, T=200, env_id_base=200), 10),
        "easy_5a_am3": lambda: thin(run_flight("FlightSearchEnvEasy", 5, 3, E=6, T=200, env_id_base=300), 10),
        # close-quarters: 5 agents on a 12x12 map so the repulsion/wall paths fire constantly
        "easy_5a_crowded": lambda: thin(run_flight("FlightSearchEnvEasy", 5, 1, E=4, T=200, env_id_base=400,
                                                     target_mode=1, map_size=12, view_range=3), 10),
        "easy_3a_tm1": lambda: thin(run_flight("FlightSearchEnvEasy", 3, 0, E=4, T=200, env_id_base=500,
                                                 target_mode=1), 10),
        "flight_3a_am0": lambda: thin(run_flight("FlightSearchEnv", 3, 0, E=3, T=200, env_id_base=600,
                                                   second_episode=25,
                                                   map_steps=(1, 2, 3, 5, 10, 20, 50, 100, 150, 200)), 20),
        "flight_2a_small": lambda: thin(run_flight("FlightSearchEnv", 2, 1, E=2, T=80, env_id_base=700,
                                                     target_mode=1, map_size=20, view_range=4, time_limit=80,
                                                     second_episode=10, map_steps=(1, 2, 5, 10, 40, 80)), 20),
        "policy_qmix_3a": lambda: run_policy("flight_easy_Seed22322107_qmix_3a15t(AM0TM0)", 3),
        "policy_conv_qmix_3a": lambda: run_policy_conv("flight_Seed74853802_qmix_3a15t(AM0TM0)", 3),
        "rollout_easy_3a": lambda: run_rollout(3, 0, episodes=4, env_id=950, seed0=77),
        "rollout_easy_5a_am3": lambda: run_rollout(5, 3, episodes=3, env_id=960, seed0=78),
        "search_3a_default": lambda: thin(run_search(3, 15, 50, 7, 0, 0, E=3, T=120, env_id_base=800), 10),
        "search_4a_am1_tm1": lambda: thin(run_search(4, 10, 20, 4, 1, 1, E=3, T=80, env_id_base=850), 10),
        "search_5a_am2": lambda: thin(run_search(5, 12, 24, 3, 2, 0, E=2, T=80, env_id_base=870), 10),
        "search_64a_1000t": lambda: thin(run_search(64, 1000, 64, 7, 0, 0, E=1, T=30, env_id_base=900), 10),
        # wide anchors for the device tests: hundreds of reference trajectories, compacted
        "anchor_easy_3a_384": lambda: compact_anchor(run_flight("FlightSearchEnvEasy", 3, 0, E=384, T=200, env_id_base=40_000)),
        "anchor_easy_5a_am2_192": lambda: compact_anchor(run_flight("FlightSearchEnvEasy", 5, 2, E=192, T=200, env_id_base=41_000)),
        "spread_3a3t": lambda: run_spread(3, 3, 50, E=4, T=100, env_id_base=1000),
        "spread_5a7t_small": lambda: run_spread(5, 7, 12, E=3, T=100, env_id_base=1100),
    }
    only = sys.argv[1:]
    for name, job in jobs.items():
        if only and name not in only:
            continue
        g = job()
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **g)
        print("%-22s %8.1f KB" % (name, os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main()
