"""Small run of every kernel for compute-sanitizer (memcheck / racecheck)."""
import os, sys, types
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import coopsearch_b200 as cs
import golden_util as gu

def fargs(n, M=50, R=7, T=25, am=0):
    return types.SimpleNamespace(env="x", map_size=M, target_num=15, target_mode=0, agent_mode=am, n_agents=n, view_range=R,
                                 time_limit=T, detect_prob=0.9, safe_dist=1, agent_velocity=1, force_dist=3)
# (class, agents, map size, lanes_per_env: 0 = thread-per-env kernel (flight variant: fused step + map kernel),
#  16 = lane-per-agent kernel (+ generic map kernel)); CS_SAN_K=1 or 4 replaces the automatic choice (0)
san_k = int(os.environ.get("CS_SAN_K", "0"))
for cls, n, M, lpe in ((cs.VecFlightEasyEnv, 3, 50, 0), (cs.VecFlightEasyEnv, 5, 12, 0), (cs.VecFlightEasyEnv, 3, 50, 16),
                       (cs.VecFlightEnv, 3, 50, 0), (cs.VecFlightEnv, 8, 63, 0), (cs.VecFlightEnv, 5, 50, 16),
                       (cs.VecFlightEnv, 2, 51, 0), (cs.VecFlightEnv, 2, 70, 0)):
    env = cls(fargs(n, M=M, R=min(7, M // 3)), gu.TEMPLATE, num_envs=37, seed=1, auto_reset=True, count_touched=True, lanes_per_env=lpe or san_k)
    env.step_random(40)
    acts = torch.randint(0, 3, (37, n), dtype=torch.uint8, device="cuda")
    env.step(acts)
    env.step_host(acts.cpu().numpy())
    if isinstance(env, cs.VecFlightEnv):
        env.get_obs()
        env.set_obs_kernel("plain"); env.get_obs()
        env.prob_map = env.prob_map
    env.stats()
# round 2: one thread per env with staged targets (lanes_per_env=1),
# the grouped launch, the pooled host path (pack kernel, strided copy), the episode writer, the agent network on the tensor
# cores with the conv front end, simple_spread
for n in (3, 5):
    envs = [cs.VecFlightEasyEnv(fargs(n), gu.TEMPLATE, num_envs=E, seed=3, env_id_base=1000 * b, auto_reset=True, lanes_per_env=1) for b, E in enumerate((38, 130, 64))]
    for e in envs:
        e.step_random(30)
    grp = cs.DeviceStepper(envs)
    for t in range(30):
        grp.step([torch.randint(0, 3, (e.num_envs, n), dtype=torch.uint8, device="cuda") for e in envs])
    hs = cs.HostStepper(envs, [torch.cuda.Stream()])
    for t in range(30):
        hs.actions.random_(0, 3)
        hs.step()
    del hs, grp, envs
fenv = cs.VecFlightEnv(fargs(3), gu.TEMPLATE, num_envs=36, seed=4, auto_reset=True)
fh = cs.HostStepper([fenv], [torch.cuda.Stream()])
for t in range(30):
    fh.actions.random_(0, 3)
    fh.step()
eenv = cs.VecFlightEasyEnv(fargs(3), gu.TEMPLATE, num_envs=40, seed=5)
cs.generate_episodes(eenv)
torch.manual_seed(0)
sd = {"fc1.weight": torch.randn(64, 26) * 0.2, "fc1.bias": torch.zeros(64), "rnn.weight_ih": torch.randn(192, 64) * 0.1, "rnn.weight_hh": torch.randn(192, 64) * 0.1,
      "rnn.bias_ih": torch.zeros(192), "rnn.bias_hh": torch.zeros(192), "fc2.0.weight": torch.randn(64, 64) * 0.1, "fc2.0.bias": torch.zeros(64),
      "fc2.2.weight": torch.randn(3, 64) * 0.1, "fc2.2.bias": torch.zeros(3), "conv.0.weight": torch.randn(4, 1, 4, 4) * 0.3, "conv.0.bias": torch.zeros(4),
      "conv.2.weight": torch.randn(1, 4, 3, 3) * 0.3, "conv.2.bias": torch.zeros(1), "linear.weight": torch.randn(16, 576) * 0.05, "linear.bias": torch.zeros(16)}
ag = cs.BatchedRNNAgents(sd, num_envs=36, n_agents=3, conv=True)
ag.choose_actions(fenv.get_obs(full=False), env=fenv)
sp = cs.VecSimpleSpreadEnv(types.SimpleNamespace(env="simple_spread", map_size=50, target_num=3, n_agents=3), num_envs=45, seed=6, auto_reset=True)
sp.step_random(120)
sp16 = cs.VecSimpleSpreadEnv(types.SimpleNamespace(env="simple_spread", map_size=30, target_num=20, n_agents=12), num_envs=9, seed=6, auto_reset=True)
sp16.step_random(110)
sargs = types.SimpleNamespace(env="search", map_size=33, target_num=40, target_mode=1, target_dir="", agent_mode=0, n_agents=9, view_range=5)
s = cs.VecSearchEnv(sargs, num_envs=21, seed=2, auto_reset=True)
s.step_random(60)
s.stats()
torch.cuda.synchronize()
print("sanitize_run done, launches:", cs.load_library().cs_launch_count())
