"""GPU parity of the search_env CUDA path: reference goldens + C oracle.  Everything here is
integer-valued except the 1/freq reward (north_star: 1e-5 relative; atol 1e-6 because -1 + sum(1/freq) can cancel to ~1e-17)."""
import types

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import c_oracle
from oracle.py_envs import SearchSpec

pytestmark = pytest.mark.gpu


def cpu(t):
    return t.detach().cpu().numpy()


def make_args(n, m, M, R, am, tm):
    return types.SimpleNamespace(env="search", map_size=M, target_num=m, target_mode=tm, target_dir="./targets/",
                                 agent_mode=am, n_agents=n, view_range=R)


def found_per_target(env, cells):
    """[E,m] u8 'target k found' from the unfound bit rows."""
    ub = cpu(env.unfound_bits).astype(np.uint32)
    E, m = cells.shape[:2]
    x, y = cells[..., 0], cells[..., 1]
    word = ub[np.arange(E)[:, None], x, y >> 5]
    return (((word >> (y & 31)) & 1) == 0).astype(np.uint8)


@pytest.mark.parametrize("name", gu.SEARCH_FIXTURES)
def test_search_matches_reference_golden(name):
    import coopsearch_b200 as cs
    g = gu.load(name)
    n, m, M, R, am, tm, base = [int(v) for v in g["meta"]]
    T, E = g["reward"].shape
    thin = int(g["thin"][0])
    env = cs.VecSearchEnv(make_args(n, m, M, R, am, tm), num_envs=E, env_id_base=base, reset=False)
    env.reset(cells=g["cells"])
    assert np.array_equal(cpu(env.agent_pos), g["init_pos"])
    assert np.array_equal(cpu(env.get_obs()), g["init_obs"].astype(np.float32))
    assert np.array_equal(cpu(env.get_state()), g["init_state"].astype(np.float32))
    assert np.array_equal(cpu(env.freq_map), g["init_freq"])
    for t in range(T):
        where = "%s step %d" % (name, t)
        assert np.array_equal(cpu(env.get_avail_actions()), g["avail"][t]), where
        r, term, info = env.step(g["actions"][t])
        assert info == ''
        np.testing.assert_allclose(cpu(r), g["reward"][t].astype(np.float32), rtol=1e-5, atol=1e-6, err_msg=where)
        assert np.array_equal(cpu(term), g["terminated"][t]), where
        assert np.array_equal(cpu(env.target_find), g["target_find"][t]), where
        assert np.array_equal(cpu(env.agent_pos), g["pos"][t]), where
        assert np.array_equal(found_per_target(env, g["cells"]), g["found"][t]), where
        if (t + 1) % thin == 0:
            k = (t + 1) // thin - 1
            assert np.array_equal(cpu(env.get_obs()), g["obs"][k]), where
            assert np.array_equal(cpu(env.get_state()), g["state"][k].astype(np.float32)), where
    assert not bool(env.illegal.any())
    assert np.array_equal(cpu(env.freq_map), g["freq"])


@pytest.mark.parametrize("n,m,M,R,am,tm", [(3, 15, 50, 7, 0, 0), (64, 1000, 64, 7, 0, 0), (9, 40, 33, 5, 1, 1), (6, 25, 70, 4, 2, 0)])
def test_search_matches_c_oracle(n, m, M, R, am, tm):
    """Device-side target placement + random legal policy in-kernel vs the C oracle, without auto-reset (the benchmarked
    auto-reset path, whole episodes and the statistics: test_gpu_search_reference.py)."""
    import coopsearch_b200 as cs
    E, T, seed, base = 40, 90, 13, 4000
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R, agent_mode=am, target_mode=tm)
    env = cs.VecSearchEnv(make_args(n, m, M, R, am, tm), num_envs=E, seed=seed, env_id_base=base, auto_reset=False)
    orc = c_oracle.SearchBatch(spec, seed, base, E)
    orc.reset()
    tb = cpu(env.target_bits).astype(np.uint32)
    dense = ((tb[:, :, :, None] >> np.arange(32)[None, None, None, :]) & 1).reshape(E, M, -1)[:, :, :M]
    assert np.array_equal(dense.astype(np.uint8), orc.tmap), "device target placement"
    for t in range(T):
        where = "step %d" % t
        r, term, _ = env.step_random(1)
        orr, ot = orc.step(None)
        assert np.array_equal(cpu(env.agent_pos), orc.pos), where
        np.testing.assert_allclose(cpu(r), orr.astype(np.float32), rtol=1e-5, atol=1e-6, err_msg=where)
        assert np.array_equal(cpu(term), ot), where
        assert np.array_equal(cpu(env.target_find), orc.counters[:, 0]), where
        if t % 15 == 0 or t == T - 1:
            obs, state, avail = orc.views()
            assert np.array_equal(cpu(env.get_obs()), obs), where
            assert np.array_equal(cpu(env.get_state()), state), where
            assert np.array_equal(cpu(env.get_avail_actions()), avail), where
    assert np.array_equal(cpu(env.freq_map), orc.freq)
    assert not bool(env.illegal.any())


def test_illegal_move_is_flagged_not_raised():
    import coopsearch_b200 as cs
    env = cs.VecSearchEnv(make_args(4, 5, 10, 3, 1, 0), num_envs=2, seed=1)   # bottom-left start
    pos0 = env.agent_pos.clone()
    acts = np.zeros((2, 4), np.uint8)
    acts[0, :] = 1      # 'left' for agent 0 at y = 0 is illegal (search_env.py:286,293)
    env.step(acts)
    ill = cpu(env.illegal)
    assert ill[0] and not ill[1]
    assert torch.equal(env.agent_pos[0, 0], pos0[0, 0])           # the offending agent stayed
    assert env.stats()["illegal_moves"] == 1.0


def test_search_env_info_errors_and_adapter():
    import coopsearch_b200 as cs
    env = cs.VecSearchEnv(make_args(3, 15, 50, 7, 0, 0), num_envs=1, seed=2)
    info = env.get_env_info()
    assert (info["n_actions"], info["state_shape"], info["obs_shape"], info["episode_limit"]) == (4, 5000, 171, 500)
    with pytest.raises(Exception, match="Act num mismatch agent"):
        env.step(np.zeros((1, 2), np.uint8))
    with pytest.raises(Exception, match="Agent id out of range"):
        env.get_avail_agent_actions(3)
    with pytest.raises(Exception, match="Unknown agent mode"):
        cs.VecSearchEnv(make_args(3, 15, 50, 7, 5, 0), num_envs=1)
    with pytest.raises(Exception, match="Unknown target mode"):
        cs.VecSearchEnv(make_args(3, 15, 50, 7, 0, 9), num_envs=1)
    one = cs.SingleEnvAdapter(env)
    o, s = one.get_obs(), one.get_state()
    assert o.shape == (3, 171) and s.shape == (5000,) and o.dtype == np.float64
    av = one.get_avail_agent_actions(0)
    r, term, info = one.step([int(np.nonzero(one.get_avail_agent_actions(i))[0][0]) for i in range(3)])
    assert isinstance(r, float) and isinstance(term, bool) and info == ''
    assert av.shape == (4,)


def test_search_host_step_and_shard_invariance():
    import coopsearch_b200 as cs
    args = make_args(5, 30, 40, 5, 0, 0)
    whole = cs.VecSearchEnv(args, num_envs=24, seed=9, env_id_base=100)
    lo = cs.VecSearchEnv(args, num_envs=12, seed=9, env_id_base=100)
    hi = cs.VecSearchEnv(args, num_envs=12, seed=9, env_id_base=112)
    for t in range(40):
        whole.step_random(1); lo.step_random(1); hi.step_random(1)
        assert torch.equal(whole.agent_pos, torch.cat([lo.agent_pos, hi.agent_pos]))
        assert torch.equal(whole.get_obs(), torch.cat([lo.get_obs(), hi.get_obs()]))
        assert torch.equal(whole._reward, torch.cat([lo._reward, hi._reward]))
    a = cs.VecSearchEnv(args, num_envs=8, seed=3)
    b = cs.VecSearchEnv(args, num_envs=8, seed=3)
    rng = np.random.default_rng(1)
    for t in range(20):
        av = cpu(a.get_avail_actions())
        act = np.array([[rng.choice(np.nonzero(av[e, i])[0]) for i in range(5)] for e in range(8)], np.uint8)
        r, term, _ = a.step(act)
        hr, hterm, hobs, hstate, havail = b.step_host(act)
        assert np.array_equal(cpu(r), hr) and np.array_equal(cpu(term), hterm)
        assert np.array_equal(cpu(a.get_obs()), hobs) and np.array_equal(cpu(a.get_state()), hstate)
        assert np.array_equal(cpu(a.get_avail_actions()), havail)
