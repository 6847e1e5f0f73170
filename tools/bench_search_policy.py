"""Agent network at the search env's input widths, on one GPU: prints one JSON line.

    python tools/bench_search_policy.py [--iters 20] [--compare-lib PATH --rounds 3]

- the GPU's name, power limit and maximum SM clock, read in the same run (nvidia-smi --query-gpu, read-only);
- choose_actions time from CUDA events over `iters` launches, both precisions, greedy with no mask, random-init
  weights and synthetic search observations (view cells in {0, 0.5, 1}, two integer positions):
    c5: 131072 envs x 64 agents = 8 388 608 rows at width 239 (hidden state 2.1 GB and obs 5.7 GB: far past the L2);
    3 agents: 131072 envs x 3 agents = 393 216 rows at width 178 (bench.py's search envs per GPU);
  with rows/s, FLOP/s (2 (in 64 + 2 64 192 + 64 64 + 64 A) per row: 88 448 at width 239) and bytes/s (obs, last
  action, hidden state read and written, q and action written: 1214 B per row at width 239);
- at the c5 size, the time per step of the search loop (get_obs, get_avail_actions, choose_actions with epsilon-greedy
  masked actions, step with auto-reset, init_hidden(mask=terminated)), 10 steps per CUDA graph, beside the env's
  step_random alone;
- with --compare-lib, bench.py's narrow-width `extra.policy` figures (measure_policy: widths <= 32) of that library
  and of this tree's library, run alternately in fresh processes, `rounds` times each.
Writes nothing to disk."""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H = 64


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=120)
    name, power, clock = [v.strip() for v in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def flop_per_row(in_dim, A):
    return 2 * (in_dim * H + 2 * H * 3 * H + H * H + H * A)


def bytes_per_row(obs_dim, A):
    return 4 * obs_dim + 1 + 2 * 4 * H + 4 * A + 1


def search_args(n, m=1000, M=64, R=7):
    return types.SimpleNamespace(env="search", map_size=M, target_num=m, target_mode=0, target_dir="", agent_mode=0,
                                 n_agents=n, view_range=R)


def weights(torch, in_dim, A):
    from oracle import policy_ref as pr
    return pr.random_state_dict(in_dim, A, 1, "default")


def events(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def time_choose_actions(cs, torch, dev, E, n, precision, iters, obs_dim=171, A=4):
    in_dim = obs_dim + A + n
    agents = cs.BatchedRNNAgents(weights(torch, in_dim, A), num_envs=E, n_agents=n, obs_dim=obs_dim, n_actions=A, device=dev,
                                 precision=precision)
    g = torch.Generator(device=dev).manual_seed(0)
    obs = torch.randint(0, 3, (E, n, obs_dim), generator=g, device=dev).to(torch.float32) * 0.5
    obs[..., -2:] = torch.randint(0, 64, (E, n, 2), generator=g, device=dev).to(torch.float32)
    for _ in range(3):
        agents.choose_actions(obs)
    torch.cuda.synchronize(dev)
    e0, e1 = events(torch)
    e0.record()
    for _ in range(iters):
        agents.choose_actions(obs)
    e1.record()
    torch.cuda.synchronize(dev)
    us = 1000.0 * e0.elapsed_time(e1) / iters
    rows = E * n
    out = {"shape": "%d envs x %d agents" % (E, n), "width": in_dim, "precision": precision, "kernel": agents.kernel_name,
           "rows": rows, "launches": iters, "us_per_launch": us, "rows_per_s": rows / (us * 1e-6),
           "tflops": rows * flop_per_row(in_dim, A) / (us * 1e-6) / 1e12, "flop_per_row": flop_per_row(in_dim, A),
           "hbm_gbs": rows * bytes_per_row(obs_dim, A) / (us * 1e-6) / 1e9, "bytes_per_row": bytes_per_row(obs_dim, A)}
    del agents, obs
    torch.cuda.empty_cache()
    return out


def time_search_loop(cs, torch, dev, E, n, replays, per_graph=10):
    """us per env step of the search loop in CUDA graphs of `per_graph` steps, for both precisions, and of step_random"""
    env = cs.VecSearchEnv(search_args(n), num_envs=E, device=dev, seed=1, auto_reset=True)
    obs_dim = env.get_env_info()["obs_shape"]
    out = {"shape": "search %d agents / 1000 targets / map 64, %d envs, auto-reset" % (n, E), "steps_per_graph": per_graph}
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for precision in ("bf16", "fp32"):
            agents = cs.BatchedRNNAgents(weights(torch, obs_dim + 4 + n, 4), num_envs=E, n_agents=n, obs_dim=obs_dim, n_actions=4,
                                         device=dev, precision=precision)

            def body():
                obs, avail = env.get_obs(), env.get_avail_actions()
                acts = agents.choose_actions(obs, avail=avail, epsilon=0.1, evaluate=False)
                _, term, _ = env.step(acts)
                agents.init_hidden(mask=term)

            for _ in range(3):
                body()
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for _ in range(per_graph):
                    body()
            graph.replay()
            torch.cuda.synchronize(dev)
            e0, e1 = events(torch)
            e0.record(side)
            for _ in range(replays):
                graph.replay()
            e1.record(side)
            torch.cuda.synchronize(dev)
            us = 1000.0 * e0.elapsed_time(e1) / (replays * per_graph)
            out["loop_" + precision] = {"kernel": agents.kernel_name, "us_per_step": us, "agent_steps_per_s": E * n / (us * 1e-6)}
            del graph, agents
        env.step_random(per_graph)
        torch.cuda.synchronize(dev)
        e0, e1 = events(torch)
        e0.record(side)
        for _ in range(replays):
            env.step_random(per_graph)
        e1.record(side)
        torch.cuda.synchronize(dev)
        out["step_random_us_per_step"] = 1000.0 * e0.elapsed_time(e1) / (replays * per_graph)
        torch.cuda.synchronize(dev)
        out["illegal_moves"] = env.stats()["illegal_moves"]
    del env
    torch.cuda.empty_cache()
    return out


NARROW = ("import json, sys, torch; sys.path.insert(0, %r); import bench, coopsearch_b200 as cs; "
          "print('POLICY ' + json.dumps(bench.measure_policy(cs, torch, torch.device('cuda', 0))))")


def narrow_alternating(compare_lib, rounds):
    """bench.py's measure_policy under COOPSEARCH_LIB = compare_lib and = this tree's library, alternately"""
    from coopsearch_b200 import build
    runs = []
    for r in range(rounds):
        for label, lib in (("compare", compare_lib), ("this", build.LIB_PATH)):
            env = dict(os.environ, COOPSEARCH_LIB=os.path.abspath(lib))
            p = subprocess.run([sys.executable, "-c", NARROW % ROOT], capture_output=True, text=True, env=env, timeout=1200)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("POLICY ")]
            if p.returncode != 0 or not line:
                raise RuntimeError("measure_policy with %s failed:\n%s" % (lib, p.stderr[-3000:]))
            pol = json.loads(line[0][7:])
            runs.append({"round": r, "lib": label,
                         "us_per_launch": {"%s rows %d" % (x["kernel"].split(" ")[0], x["rows"]): round(x["us_per_launch"], 2) for x in pol["runs"]},
                         "device_loop_us_per_step": round(pol["device_loop"]["us_per_step"], 2)})
    return runs


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--replays", type=int, default=5)
    ap.add_argument("--compare-lib", default=None, help="another build of libcoopsearch.so for the narrow-width comparison")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    import coopsearch_b200 as cs
    if not torch.cuda.is_available():
        raise SystemExit("bench_search_policy.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "choose_actions": []}
    for E, n in ((131072, 64), (131072, 3)):
        for precision in ("bf16", "fp32"):
            res["choose_actions"].append(time_choose_actions(cs, torch, dev, E, n, precision, a.iters))
    res["search_loop_c5"] = time_search_loop(cs, torch, dev, 131072, 64, a.replays)
    if a.compare_lib:
        res["narrow_policy_alternating"] = narrow_alternating(a.compare_lib, a.rounds)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
