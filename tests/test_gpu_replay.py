"""Device replay ring and replay statistics (SURVEY.md section 8f ranks 2 and 4) against the reference's own
common/replay_buffer.py (imported from the reference checkout or oracle/_ref) and its shipped result curves."""
import types

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import refharness as rh

pytestmark = pytest.mark.gpu


def cpu(t):
    return t.detach().cpu().numpy()


def easy_args(n_agents=3, agent_mode=0, time_limit=200):
    return types.SimpleNamespace(env="flight_easy", map_size=50, target_num=15, target_mode=0, agent_mode=agent_mode, n_agents=n_agents,
                                 view_range=7, time_limit=time_limit, detect_prob=0.9, safe_dist=1, agent_velocity=1, force_dist=3)


@pytest.mark.needs_reference
def test_replay_ring_equals_reference_replay_buffer():
    """store_episode (with wrap-around), sample_latest and row gathers of the device ring == the reference's numpy
    ReplayBuffer fed the same episode batches (common/replay_buffer.py:36-99)."""
    import coopsearch_b200 as cs
    rh.import_reference()
    with rh.contextlib.redirect_stdout(rh.io.StringIO()):
        from common.replay_buffer import ReplayBuffer
    args = easy_args(time_limit=30)
    env = cs.VecFlightEasyEnv(args, gu.TEMPLATE, num_envs=7, seed=3)
    info = env.get_env_info()
    bargs = types.SimpleNamespace(n_actions=info["n_actions"], n_agents=3, state_shape=info["state_shape"], obs_shape=info["obs_shape"],
                                  episode_limit=info["episode_limit"], conv=False, map_size=50)
    ours = cs.DeviceReplayBuffer(bargs, buffer_size=16)
    ref = rh.quiet(ReplayBuffer, bargs, 16)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for it in range(5):                                    # 35 episodes into 16 slots: wraps twice
        ep, _, _, _ = cs.generate_episodes(env, generator=gen)
        batch = {k: ep[k] for k in cs.replay.EPISODE_KEYS}
        ours.store_episode(batch)
        ref.store_episode({k: cpu(v).astype(np.float64) for k, v in batch.items()})
        assert ours.current_idx == ref.current_idx and ours.current_size == ref.current_size
        filled = ref.current_size
        for k in cs.replay.EPISODE_KEYS:
            assert np.array_equal(cpu(ours.buffers[k][:filled]).astype(np.float64), ref.buffers[k][:filled]), (it, k)
        for bs in (3, 9, 16):
            if ours.can_sample(bs):
                a, b = ours.sample_latest(bs), ref.sample_latest(bs)
                for k in cs.replay.EPISODE_KEYS:
                    assert np.array_equal(cpu(a[k]).astype(np.float64), b[k]), (it, bs, k)
    assert ours.can_sample(16) and not ours.can_sample(17)
    s = ours.sample(64, generator=gen)                     # uniform with replacement from the filled part (:63-68)
    assert s["o"].shape == (64, 30, 3, 4) and s["padded"].dtype == torch.uint8
    flat = cpu(ours.buffers["s"]).reshape(16, -1)
    for row in cpu(s["s"]).reshape(64, -1)[:8]:
        assert (flat == row).all(axis=1).any()


CHECKPOINTS = [10, 20, 40, 60, 80, 100, 150, 199]


@pytest.mark.parametrize("n_agents,agent_mode,want", [(3, 0, [0.00, 2.87, 47.93, 66.60, 70.13, 72.40, 79.53, 84.87]),
                                                      (5, 0, [0.00, 4.73, 63.33, 84.00, 86.73, 88.67, 93.13, 95.80])])
def test_collect_replay_stats_reproduces_shipped_random_policy_curves(n_agents, agent_mode, want):
    """collect_replay_stats = runner.collect_experiment_data over rollout.generate_replay with alg=random: the reference's
    result/flight_easy_Seed0_random_*a15t(AM0TM0)/average_res_529.npy (N=100 replays) within its sampling error, from
    16384 replays on the device."""
    import coopsearch_b200 as cs
    env = cs.VecFlightEasyEnv(easy_args(n_agents, agent_mode), gu.TEMPLATE, num_envs=16384, seed=529)
    out = cs.collect_replay_stats(env, agents=None, generator=torch.Generator(device="cuda").manual_seed(1))
    curve = out["average_res"]
    assert curve.shape == (200,) and out["replays"] == 16384
    err = np.abs(curve[CHECKPOINTS] - np.array(want))
    assert err.max() < 7.0, (np.round(curve[CHECKPOINTS], 2).tolist(), want)
    assert np.all(np.diff(curve) >= -1e-9) and curve[-1] <= 100.0
    assert 0 < out["average_step"] <= 200 and out["average_tgt_find"] <= 15


def test_collect_replay_stats_with_the_shipped_policy():
    """Greedy shipped qmix policy (tensor-core network): the curve dominates the random policy's and ends near 100 %."""
    import coopsearch_b200 as cs
    g = gu.load("policy_qmix_3a")
    sd = {k[2:]: g[k] for k in g if k.startswith("w:")}
    E = 4096
    env = cs.VecFlightEasyEnv(easy_args(3, 0), gu.TEMPLATE, num_envs=E, seed=60)
    agents = cs.BatchedRNNAgents(sd, num_envs=E, n_agents=3)
    out = cs.collect_replay_stats(env, agents=agents)
    curve = out["average_res"]
    assert curve[60] > 80.0 and curve[199] > 97.0, np.round(curve[CHECKPOINTS], 2).tolist()
    assert out["average_step"] < 150
