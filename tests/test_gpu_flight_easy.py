"""GPU parity of the flight_easy CUDA path (through the C ABI) against
  (1) golden trajectories of the unmodified reference (tests/golden/easy_*.npz), and
  (2) the Python oracle on fresh seeded inputs,
plus the batched-API contracts (masking, auto-reset, shard invariance, host-buffer step).

Bars: found masks / rewards / terminated / win / target_find / time_step / out flags bit-exact;
fp64 positions and headings to 1e-9 (CUDA sincos vs libm differ in the last ulp); fp32 obs/state to
rtol 1e-5 + atol 1e-6 (north_star tolerance; SURVEY.md section 7 hard part 2 for the atol)."""
import types

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle.py_envs import FlightOracle, FlightSpec

pytestmark = pytest.mark.gpu


def make_args(kw):
    return types.SimpleNamespace(
        env="flight_easy" if kw["variant"] == "easy" else "flight",
        map_size=kw["map_size"], target_num=kw["target_num"], target_mode=kw["target_mode"],
        agent_mode=kw["agent_mode"], n_agents=kw["n_agents"], view_range=kw["view_range"],
        time_limit=kw["time_limit"], detect_prob=kw["detect_prob"], safe_dist=kw["safe_dist"],
        agent_velocity=kw["velocity"], force_dist=kw["force_dist"], turn_limit=np.pi / 4, wrong_alarm_prob=0.1)


TEMPLATE = gu.TEMPLATE


def cpu(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("lpe", [0, 1, 4, 32])
@pytest.mark.parametrize("name", gu.EASY_FIXTURES)
def test_matches_reference_golden(name, lpe):
    import coopsearch_b200 as cs
    g = gu.load(name)
    kw, base, seed = gu.flight_spec_kwargs(g, "easy")
    T, E = g["reward"].shape
    n = kw["n_agents"]
    env = cs.VecFlightEasyEnv(make_args(kw), None, num_envs=E, seed=seed, env_id_base=base, lanes_per_env=lpe, reset=False)
    env.reset(init=True, targets=g["tgt_xy"])
    torch.cuda.synchronize()
    assert np.array_equal(cpu(env.found_mask).astype(np.uint32), g["init_found"])
    assert np.array_equal(cpu(env.win_flag), g["init_win"])
    np.testing.assert_allclose(cpu(env.agent_xy), g["init_xy"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(cpu(env.agent_yaw), g["init_yaw"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(cpu(env.get_state()), g["init_state"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(cpu(env.get_obs()), g["init_obs"], rtol=1e-5, atol=1e-6)
    thin = int(g["thin"][0])
    for t in range(T):
        r, term, win = env.step(g["actions"][t])
        where = "%s lpe=%d step %d" % (name, lpe, t)
        assert np.array_equal(cpu(env.found_mask).astype(np.uint32), g["found"][t]), where
        assert np.array_equal(cpu(r), g["reward"][t].astype(np.float32)), where
        assert np.array_equal(cpu(term), g["terminated"][t]), where
        assert np.array_equal(cpu(win), g["win"][t]), where
        assert np.array_equal(cpu(env.target_find), g["target_find"][t]), where
        assert np.array_equal(cpu(env.time_step), g["time_step"][t]), where
        out = (cpu(env.out_mask)[:, None] >> np.arange(n)[None, :]) & 1
        assert np.array_equal(out.astype(np.uint8), g["out"][t]), where
        np.testing.assert_allclose(cpu(env.agent_xy), g["xy"][t], rtol=0, atol=1e-9, err_msg=where)
        np.testing.assert_allclose(cpu(env.agent_yaw), g["yaw"][t], rtol=0, atol=1e-12, err_msg=where)
        if (t + 1) % thin == 0:
            k = (t + 1) // thin - 1
            np.testing.assert_allclose(cpu(env.get_state()), g["state"][k], rtol=1e-5, atol=1e-6, err_msg=where)
            np.testing.assert_allclose(cpu(env.get_obs()), g["obs"][k], rtol=1e-5, atol=1e-6, err_msg=where)


def run_oracle(spec, template, seed, ids, actions, targets=None):
    """Python-oracle trajectories for env ids `ids`; actions [T, len(ids), n]."""
    T = actions.shape[0]
    n = spec.n_agents
    res = dict(found=np.zeros((T, len(ids)), np.uint32), reward=np.zeros((T, len(ids)), np.float32),
               term=np.zeros((T, len(ids)), np.uint8), win=np.zeros((T, len(ids)), np.uint8),
               xy=np.zeros((T, len(ids), n, 2)), tgt=np.zeros((len(ids), spec.target_num, 2)),
               state=np.zeros((T, len(ids), spec.state_shape)))
    for k, eid in enumerate(ids):
        o = FlightOracle(spec, template, seed, int(eid))
        o.reset(targets=None if targets is None else targets[k], init=True)
        res["tgt"][k] = np.array(o.tgt)
        done = False
        for t in range(T):
            r = 0.0
            if not done:
                r, done, _ = o.step(actions[t, k])
            res["found"][t, k] = o.found_mask()
            res["reward"][t, k] = r
            res["term"][t, k] = int(done)
            res["win"][t, k] = int(o.win)
            res["xy"][t, k] = np.array(o.pos, float)
            res["state"][t, k] = o.get_state()
    return res


@pytest.mark.parametrize("n_agents,agent_mode,target_mode,lpe", [(3, 0, 0, 0), (5, 2, 0, 8), (5, 3, 1, 1), (1, 1, 0, 2), (8, 0, 1, 16)])
def test_device_reset_and_steps_match_oracle(n_agents, agent_mode, target_mode, lpe):
    """Targets drawn on the device (keyed Box-Muller / uniform) + full episodes vs the oracle."""
    import coopsearch_b200 as cs
    E, T, seed, base = 96, 200, 7, 5000
    spec = FlightSpec(n_agents=n_agents, agent_mode=agent_mode, target_mode=target_mode)
    kw = dict(spec.__dict__)
    env = cs.VecFlightEasyEnv(make_args(kw), TEMPLATE, num_envs=E, seed=seed, env_id_base=base, lanes_per_env=lpe)
    actions = np.random.default_rng(99).integers(0, 3, size=(T, E, n_agents), dtype=np.uint8)
    want = run_oracle(spec, TEMPLATE, seed, base + np.arange(E), actions)
    np.testing.assert_allclose(cpu(env.tgt_xy), want["tgt"], rtol=0, atol=1e-9)
    for t in range(T):
        r, term, win = env.step(actions[t])
        where = "step %d" % t
        assert np.array_equal(cpu(env.found_mask).astype(np.uint32), want["found"][t]), where
        assert np.array_equal(cpu(r), want["reward"][t]), where
        assert np.array_equal(cpu(term), want["term"][t]), where
        assert np.array_equal(cpu(win), want["win"][t]), where
        np.testing.assert_allclose(cpu(env.agent_xy), want["xy"][t], rtol=0, atol=1e-8, err_msg=where)
        if t % 25 == 0:
            np.testing.assert_allclose(cpu(env.get_state()), want["state"][t], rtol=1e-5, atol=1e-6, err_msg=where)


def test_shard_invariance_and_lane_invariance():
    """Results depend on the GLOBAL env id only: one 64-env handle == two 32-env handles with
    env_id_base offsets (what 1 vs 2 GPUs do), bit for bit, and every lanes-per-env instantiation agrees."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=5, agent_mode=2)
    args = make_args(dict(spec.__dict__))
    E, T = 64, 120
    actions = torch.from_numpy(np.random.default_rng(5).integers(0, 3, size=(T, E, 5), dtype=np.uint8)).cuda()
    whole = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=3, env_id_base=1000, lanes_per_env=8)
    lo = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=32, seed=3, env_id_base=1000, lanes_per_env=1)
    hi = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=32, seed=3, env_id_base=1032, lanes_per_env=32)
    for t in range(T):
        rw, tw, ww = whole.step(actions[t])
        rl, tl, wl = lo.step(actions[t, :32])
        rh, th, wh = hi.step(actions[t, 32:])
        assert torch.equal(rw, torch.cat([rl, rh]))
        assert torch.equal(tw, torch.cat([tl, th]))
        assert torch.equal(whole._dyn, torch.cat([lo._dyn, hi._dyn]))
        assert torch.equal(whole.get_state(), torch.cat([lo.get_state(), hi.get_state()]))


@pytest.mark.parametrize("n_agents,agent_mode,target_mode,map_size,time_limit,variant",
                         [(3, 0, 0, 50, 40, "easy"), (5, 2, 1, 50, 30, "easy"), (8, 3, 1, 14, 25, "easy"), (1, 1, 0, 50, 20, "easy"),
                          (3, 0, 0, 50, 40, "probmap"), (6, 1, 1, 20, 15, "probmap")])
def test_thread_per_env_kernel_equals_lane_per_agent_kernel(n_agents, agent_mode, target_mode, map_size, time_limit, variant):
    """flight_tpe_kernel (one thread per env, the default for n_agents <= 8) and flight_kernel (one lane per agent /
    target, lanes_per_env > 0) are the same arithmetic in a different arrangement: every buffer must agree bit for
    bit, through episode ends, in-call auto-resets and device-drawn targets, under device actions and the in-kernel
    random policy."""
    compare_step_kernels(n_agents, agent_mode, target_mode, map_size, time_limit, variant, 1000, 0)


@pytest.mark.parametrize("n_agents,agent_mode,target_mode,time_limit,E",
                         [(3, 0, 0, 40, 1000), (3, 0, 0, 12, 2), (5, 2, 1, 30, 130), (8, 3, 1, 25, 4222), (1, 1, 0, 20, 258), (4, 0, 0, 15, 640),
                          (3, 0, 0, 12, 40000)])
def test_one_thread_per_env_kernel_shapes_equal_lane_per_agent_kernel(n_agents, agent_mode, target_mode, time_limit, E):
    """flight_tpe_kernel<N, 1> (lanes_per_env = 1: one thread per env, structure-of-arrays state, targets staged in shared
    memory) against flight_kernel, bit for bit: partial warps and CTAs, a single agent, eight agents, and auto-resets whose
    redrawn targets are read back from the staging area, under device actions and the in-kernel random policy."""
    compare_step_kernels(n_agents, agent_mode, target_mode, 50, time_limit, "easy", E, 1)


@pytest.mark.parametrize("variant,n_agents", [("probmap", 3), ("easy", 5), ("probmap", 6)])
def test_one_thread_per_env_forms_equal_lane_per_agent_kernel(variant, n_agents):
    """lanes_per_env = 1 (what handles of >= 32768 envs get by default): structure-of-arrays state, staged targets for
    flight_easy, the job records for the tiled map kernel for the flight variant -- against flight_kernel, bit for bit."""
    compare_step_kernels(n_agents, 0, 0, 50, 30, variant, 1001 if variant == "easy" else 600, 1)


def compare_step_kernels(n_agents, agent_mode, target_mode, map_size, time_limit, variant, E, lanes):
    import coopsearch_b200 as cs
    T = 3 * time_limit + 7
    spec = FlightSpec(n_agents=n_agents, agent_mode=agent_mode, target_mode=target_mode, map_size=map_size,
                      view_range=min(7, map_size // 3), time_limit=time_limit, variant=variant)
    args = make_args(dict(spec.__dict__))
    cls = cs.VecFlightEasyEnv if variant == "easy" else cs.VecFlightEnv
    tpe = cls(args, TEMPLATE, num_envs=E, seed=11, env_id_base=77, auto_reset=True, lanes_per_env=lanes)
    lpa = cls(args, TEMPLATE, num_envs=E, seed=11, env_id_base=77, auto_reset=True, lanes_per_env=16 if n_agents <= 16 else 32)
    assert tpe.lanes_per_env <= 8 and lpa.lanes_per_env >= 16
    actions = torch.from_numpy(np.random.default_rng(2).integers(0, 3, size=(T, E, n_agents), dtype=np.uint8)).cuda()
    for t in range(T):
        if t % 5 == 4:
            ra, ta, wa = tpe.step_random(1)
            rb, tb, wb = lpa.step_random(1)
        else:
            ra, ta, wa = tpe.step(actions[t])
            rb, tb, wb = lpa.step(actions[t])
        where = "step %d" % t
        assert torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(wa, wb), where
        assert torch.equal(tpe.target_find, lpa.target_find), where
        # positions / headings bit for bit; meta words 0..6 (word 7 is the generic map kernel's job marker, unused by the fused kernel)
        nrow = 3 * n_agents
        assert torch.equal(tpe._dyn[:, :nrow].contiguous().view(torch.int64), lpa._dyn[:, :nrow].contiguous().view(torch.int64)), where
        assert torch.equal(tpe.meta[:, :7], lpa.meta[:, :7]), where
        assert torch.equal(tpe.tgt_xy.contiguous().view(torch.int64), lpa.tgt_xy.contiguous().view(torch.int64)), where
        assert torch.equal(tpe.get_state().view(torch.int32), lpa.get_state().view(torch.int32)), where
        assert torch.equal(tpe.get_obs(full=False).view(torch.int32) if variant != "easy" else tpe.get_obs().view(torch.int32),
                           lpa.get_obs(full=False).view(torch.int32) if variant != "easy" else lpa.get_obs().view(torch.int32)), where
        if variant != "easy":
            assert torch.equal(tpe.prob_map, lpa.prob_map), where
    sa, sb = tpe.stats(), lpa.stats()
    assert sa == sb and sa["episodes"] >= 2 * E


def test_auto_reset_and_stats():
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=40)
    args = make_args(dict(spec.__dict__))
    E = 200
    env = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=11, auto_reset=True)
    total_r = np.zeros(E)
    ep_sum, eps, steps = 0.0, 0, 0
    for t in range(100):
        r, term, win = env.step_random(1)
        total_r += cpu(r)
        term = cpu(term).astype(bool)
        ep_sum += total_r[term].sum()
        eps += int(term.sum())
        total_r[term] = 0
        steps += E
        ts = cpu(env.time_step)
        assert np.all(ts[term] == 0)                 # terminated envs were reset in the same call
        assert np.all(ts <= 40)
    st = env.stats()
    assert st["env_steps"] == steps
    assert st["episodes"] == eps and eps >= 2 * E
    assert abs(st["episode_reward_sum"] - ep_sum) < 1e-6 * max(1.0, abs(ep_sum))
    assert st["episode_len_sum"] <= 40 * eps


def test_masked_noop_after_termination_and_partial_reset():
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=5)
    args = make_args(dict(spec.__dict__))
    env = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=8, seed=1)
    for _ in range(5):
        r, term, _ = env.step_random(1)
    assert cpu(term).all()
    snap = env._dyn.clone()
    state = env.get_state().clone()
    r, term, _ = env.step_random(1)
    assert cpu(term).all() and not cpu(r).any()
    assert torch.equal(env._dyn, snap) and torch.equal(env.get_state(), state)
    mask = torch.tensor([1, 0, 0, 1, 0, 0, 0, 0], dtype=torch.uint8, device="cuda")
    env.reset(mask=mask)
    ts = cpu(env.time_step)
    assert list(ts) == [0, 5, 5, 0, 5, 5, 5, 5]
    r, term, _ = env.step_random(1)
    assert list(cpu(term)) == [0, 1, 1, 0, 1, 1, 1, 1]
    assert list(cpu(env.meta[:, 4])) == [1, 0, 0, 1, 0, 0, 0, 0]      # episode counters


@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("lpe,auto_reset", [(0, True), (0, False), (16, True)])
def test_host_buffer_step_equals_device_step(lpe, auto_reset, compact):
    """cs_flight_step_host (whole slab) / cs_flight_step_host_compact (16 + 16n bytes per env, rows rebuilt on the
    host): the host results are exactly what the device buffers hold after every step, also across reset(), in-call
    auto-resets and device-resident steps in between."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=25)
    args = make_args(dict(spec.__dict__))
    E = 300
    a = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=2, auto_reset=auto_reset, lanes_per_env=lpe)
    b = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=2, auto_reset=auto_reset, lanes_per_env=lpe)
    rng = np.random.default_rng(0)
    for t in range(90):
        act = rng.integers(0, 3, size=(E, 3), dtype=np.uint8)
        if t in (40, 41):
            a.step(act); b.step(act)
            continue
        if t == 60:
            a.reset(); b.reset()
        r, term, win = a.step(act)
        hr, hterm, hwin, hobs, hstate = b.step_host(act, compact=compact)
        where = "step %d" % t
        assert np.array_equal(cpu(r), hr) and np.array_equal(cpu(term), hterm) and np.array_equal(cpu(win), hwin), where
        assert np.array_equal(cpu(a.target_find), b.host_buffers(compact)["target_find"].numpy()), where
        assert np.array_equal(cpu(a.get_obs()), hobs), where
        assert np.array_equal(cpu(a.get_state()), hstate), where


def test_compact_host_step_survives_a_mass_reset():
    """More envs reset inside one call than the compact path's side region holds (every env hits the time limit at the
    same step): the rows are refreshed in full and still equal the device rows."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=5, time_limit=6, agent_mode=2)
    args = make_args(dict(spec.__dict__))
    E = 2000
    a = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=3, auto_reset=True)
    b = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=3, auto_reset=True)
    rng = np.random.default_rng(0)
    for t in range(20):
        act = rng.integers(0, 3, size=(E, 5), dtype=np.uint8)
        r, term, win = a.step(act)
        hr, hterm, hwin, hobs, hstate = b.step_host(act)
        assert np.array_equal(cpu(r), hr) and np.array_equal(cpu(term), hterm), t
        assert np.array_equal(cpu(a.get_state()), hstate) and np.array_equal(cpu(a.get_obs()), hobs), t


@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("graph", [False, True])
def test_host_stepper_many_batches_one_call(graph, compact):
    """cs_flight_step_host_many: several env batches stepped from pinned host actions with one library call (or one
    CUDA-graph launch) equal the same batches stepped one by one on the device."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=30)
    args = make_args(dict(spec.__dict__))
    B, E = 5, 200
    ref = [cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=6, env_id_base=b * E, auto_reset=True) for b in range(B)]
    envs = [cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=6, env_id_base=b * E, auto_reset=True) for b in range(B)]
    streams = [torch.cuda.Stream() for _ in range(2)]
    torch.cuda.synchronize()
    pinned = [torch.empty((E, 3), dtype=torch.uint8).pin_memory() for _ in range(B)]
    stepper = cs.HostStepper(envs, streams, actions=pinned, graph=graph, compact=compact)
    rng = np.random.default_rng(1)
    for t in range(70):
        for b in range(B):
            pinned[b].numpy()[...] = rng.integers(0, 3, size=(E, 3), dtype=np.uint8)
        stepper.step()
        for b in range(B):
            r, term, win = ref[b].step(pinned[b].cuda())
            hb = envs[b].host_buffers(compact)
            assert np.array_equal(cpu(r), hb["reward"].numpy()) and np.array_equal(cpu(term), hb["terminated"].numpy())
            assert np.array_equal(cpu(ref[b].get_state()), hb["state"].numpy()), "batch %d step %d" % (b, t)
            assert np.array_equal(cpu(ref[b].get_obs()), hb["obs"].numpy())


@pytest.mark.parametrize("variant,graph,sizes,lpe", [("easy", False, [200, 200, 200], 0), ("easy", True, [700, 64, 4096], 1),
                                                      ("easy", True, [256, 256], 4), ("probmap", False, [96, 160], 0), ("probmap", True, [64, 64, 64], 0)])
def test_pooled_host_stepper_equals_device_steps(variant, graph, sizes, lpe):
    """cs_flight_host_pool_*: all batches stepped from ONE pinned action buffer with one H2D copy, one (grouped) step, one
    pack launch, the flat record copy and the strided copy that writes the agent rows in place -- host rows, rewards and
    flags equal the same batches stepped on the device, through auto-resets, a manual reset in between, an external action
    buffer, and (flight variant) the per-batch launch fallback."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=25, variant=variant)
    args = make_args(dict(spec.__dict__))
    cls = cs.VecFlightEasyEnv if variant == "easy" else cs.VecFlightEnv
    mk = lambda: [cls(args, TEMPLATE, num_envs=E, seed=6, env_id_base=10000 * b, auto_reset=True, lanes_per_env=lpe) for b, E in enumerate(sizes)]
    ref, envs = mk(), mk()
    streams = [torch.cuda.Stream() for _ in range(2)]
    torch.cuda.synchronize()
    stepper = cs.HostStepper(envs, streams, graph=graph, compact=True)
    assert stepper._pool is not None and stepper.actions.shape == (sum(sizes), 3)
    other = torch.empty_like(stepper.actions).pin_memory()
    first = np.concatenate([[0], np.cumsum(sizes)])
    rng = np.random.default_rng(1)
    for t in range(80):
        buf = other if t % 3 == 2 else stepper.actions
        buf.numpy()[...] = rng.integers(0, 3, size=buf.shape, dtype=np.uint8)
        if t == 40:                                    # a reset from outside: the host rows are refreshed in full
            for e, r in zip(envs, ref):
                e.reset(); r.reset()
        stepper.step(actions=other) if t % 3 == 2 else stepper.step()
        for b in range(len(sizes)):
            act = buf[first[b]:first[b + 1]]
            if t % 3 != 2:
                assert np.array_equal(envs[b].host_buffers()["actions"].numpy(), act.numpy())      # each env's segment of the pooled buffer
            r, term, win = ref[b].step(act.cuda())
            hb = envs[b].host_buffers()
            where = "batch %d step %d" % (b, t)
            assert np.array_equal(cpu(r), hb["reward"].numpy()) and np.array_equal(cpu(term), hb["terminated"].numpy()), where
            assert np.array_equal(cpu(win), hb["win"].numpy()) and np.array_equal(cpu(ref[b].target_find), hb["target_find"].numpy()), where
            assert np.array_equal(cpu(ref[b].get_state()), hb["state"].numpy()), where
            assert np.array_equal(cpu(ref[b].get_obs(full=False) if variant != "easy" else ref[b].get_obs()), hb["obs"].numpy()), where
    if variant != "easy":
        assert torch.equal(ref[0].prob_map, envs[0].prob_map)
    with pytest.raises(cs.CoopSearchError):
        envs[0].step_host(np.zeros((sizes[0], 3), np.uint8))          # a pooled env is stepped through its pool
    del stepper, envs                                                  # pool and envs go away in either order


def test_pooled_host_stepper_reset_list_tail_and_overflow():
    """The pooled step copies the first num_envs/48 reset entries with the results; 150 envs that end in one call take the
    separate tail copy, ~3900 envs that end in one call overflow the list (num_envs/16) and force a full refresh of the host rows."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=10)
    args = make_args(dict(spec.__dict__))
    E = 4096
    mk = lambda: cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=2, auto_reset=True)
    env, ref = mk(), mk()
    stepper = cs.HostStepper([env], [torch.cuda.Stream()])
    assert stepper._pool is not None
    rng = np.random.default_rng(3)
    mask = (np.arange(E) >= 150).astype(np.uint8)
    resets_seen = []
    for t in range(26):
        if t == 4:                                   # envs >= 150 start over: the first 150 end 6 calls later, on their own
            env.reset(mask=mask); ref.reset(mask=mask)
        stepper.actions.numpy()[...] = rng.integers(0, 3, size=(E, 3), dtype=np.uint8)
        stepper.step()
        r, term, win = ref.step(stepper.actions.cuda())
        hb = env.host_buffers()
        resets_seen.append(int(cpu(term).sum()))
        assert np.array_equal(cpu(r), hb["reward"].numpy()) and np.array_equal(cpu(term), hb["terminated"].numpy()), t
        assert np.array_equal(cpu(ref.get_state()), hb["state"].numpy()), t
    assert any(85 < c <= 256 for c in resets_seen) and any(c > 256 for c in resets_seen), resets_seen


@pytest.mark.parametrize("lpe,sizes", [(1, [700, 4096, 33]), (1, [700, 4096, 34, 2, 128]), (4, [700, 4096, 34, 2, 128]), (4, [256, 256, 256, 1000]), (0, [512, 512])])
def test_grouped_device_step_equals_separate_steps(lpe, sizes):
    """cs_flight_group_step: env batches of different sizes stepped in ONE launch end up bit-identical to the same
    batches stepped one by one (state, targets, outputs, statistics), through episode ends and in-call auto-resets."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3, time_limit=20)
    args = make_args(dict(spec.__dict__))
    mk = lambda: [cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=E, seed=9, env_id_base=1000 * b, auto_reset=True, lanes_per_env=lpe)
                  for b, E in enumerate(sizes)]
    ref, envs = mk(), mk()
    stepper = cs.DeviceStepper(envs)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(50):
        acts = [torch.randint(0, 3, (E, 3), dtype=torch.uint8, device="cuda", generator=gen) for E in sizes]
        stepper.step(acts)
        for a, e, r in zip(acts, envs, ref):
            rr, rt, rw = r.step(a)
            assert torch.equal(rr, e._reward) and torch.equal(rt, e._terminated) and torch.equal(rw, e._win), "step %d" % t
            assert torch.equal(r._dyn, e._dyn) and torch.equal(r.tgt_xy, e.tgt_xy), "step %d" % t
            assert torch.equal(r.get_state(), e.get_state()) and torch.equal(r.get_obs(), e.get_obs()), "step %d" % t
    assert [r.stats() for r in ref] == [e.stats() for e in envs]
    with pytest.raises(cs.CoopSearchError):
        cs.DeviceStepper([envs[0], cs.VecFlightEasyEnv(make_args(dict(FlightSpec(n_agents=5).__dict__)), TEMPLATE, num_envs=8, seed=1)])


def test_reference_error_behaviour():
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3)
    args = make_args(dict(spec.__dict__))
    env = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=4)
    with pytest.raises(Exception, match="Act num mismatch agent"):
        env.step(np.zeros((4, 2), np.uint8))
    with pytest.raises(Exception, match="Agent id out of range"):
        env.get_avail_agent_actions(3)
    with pytest.raises(IndexError):                                   # dyaw[act] with act = 3 (flight_env_easy.py:259-262)
        env.step(np.full((4, 3), 3))
    assert env.get_avail_agent_actions(2).shape == (4, 3) and bool((env.get_avail_actions() == 1).all())
    bad = make_args(dict(spec.__dict__)); bad.agent_mode = 7
    with pytest.raises(Exception, match="No such agent mode"):
        cs.VecFlightEasyEnv(bad, TEMPLATE, num_envs=4)
    bad = make_args(dict(spec.__dict__)); bad.target_mode = 5
    with pytest.raises(Exception, match="No such target mode"):
        cs.VecFlightEasyEnv(bad, TEMPLATE, num_envs=4)
    info = env.get_env_info()
    assert (info["n_actions"], info["state_shape"], info["obs_shape"], info["episode_limit"]) == (3, 57, 4, 200)


def test_single_env_adapter_types():
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=3)
    args = make_args(dict(spec.__dict__))
    env = cs.SingleEnvAdapter(cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=1, seed=4))
    env.reset()
    o, s = env.get_obs(), env.get_state()
    assert o.shape == (3, 4) and o.dtype == np.float64 and s.shape == (57,) and s.dtype == np.float64
    r, term, info = env.step([np.int64(1), torch.tensor(2), 0])
    assert isinstance(r, float) and isinstance(term, bool) and isinstance(info, bool)
    assert isinstance(env.target_find, int)
    assert np.array_equal(env.get_avail_agent_actions(0), np.ones(3))


def test_config1_rollout_protocol_single_env():
    """BASELINE.json configs[0]: flight_easy 1a15t AM0TM0, ONE env, uniform-random policy, driven through the exact
    call sequence of RolloutWorker.generate_episode (common/rollout.py:22-140): reset, then per step get_obs,
    get_state, get_avail_agent_actions per agent, step(actions), and finally target_find -- on the E=1 adapter,
    against the Python oracle fed the same actions and the same injected targets."""
    import coopsearch_b200 as cs
    spec = FlightSpec(n_agents=1, agent_mode=0, target_mode=0)
    args = make_args(dict(spec.__dict__))
    vec = cs.VecFlightEasyEnv(args, TEMPLATE, num_envs=1, seed=42, env_id_base=77)
    env = cs.SingleEnvAdapter(vec)
    info = env.get_env_info()
    assert info == {"n_actions": 3, "state_shape": 49, "obs_shape": 4, "episode_limit": 200}
    orc = FlightOracle(spec, TEMPLATE, 42, 77)
    rng = np.random.RandomState(0)
    for episode in range(3):
        env.reset()
        orc.reset(targets=cpu(vec.tgt_xy)[0], init=False, episode=episode + 1)   # ctor reset was episode 0
        terminated, step, episode_reward, win_tag = False, 0, 0.0, False
        o, s, r = [], [], []
        while not terminated and step < info["episode_limit"]:
            obs, state = env.get_obs(), env.get_state()
            np.testing.assert_allclose(obs, orc.get_obs(), rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(state, orc.get_state(), rtol=1e-5, atol=1e-6)
            actions = []
            for agent_id in range(1):
                avail = env.get_avail_agent_actions(agent_id)
                actions.append(rng.choice(np.nonzero(avail)[0]))          # agent.py:34-36 (alg=random)
            reward, terminated, info_flag = env.step(actions)
            wr, wterm, wwin = orc.step(actions)
            assert (reward, terminated, info_flag) == (float(wr), bool(wterm), bool(wwin))
            win_tag = True if terminated and info_flag else False
            o.append(obs); s.append(state); r.append([reward])
            episode_reward += reward
            step += 1
        assert env.target_find == orc.target_find
        assert step == orc.time_step and episode_reward == orc.total_reward
        assert win_tag == (orc.win and terminated)
