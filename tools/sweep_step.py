"""Step kernel sweep: python tools/sweep_step.py [workloads...]; env CS_BENCH_LPE / CS_BENCH_STREAMS select the variant."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bench  # noqa: E402
import coopsearch_b200 as cs  # noqa: E402

dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
names = sys.argv[1:] or ["c2", "c3", "c2w"]
tag = "LPE=%s streams=%s" % (os.environ.get("CS_BENCH_LPE", "0"), os.environ.get("CS_BENCH_STREAMS", "8"))
for name in names:
    steps = {"c2": 60, "c2s": 60, "c3": 100, "c2w": 30, "c4": 100}.get(name, 50)
    r = bench.run_gpu_workload(cs, torch, name, steps, 5, dev, 0, 1, want_e2e=(name in ("c2", "c2s")), burn_in_s=0.2)
    v = r["env_steps_per_step"] / (r["ms_per_step"] * 1e-3)
    e2e = (r["env_steps_per_step"] / r["e2e_s_per_step"]) if "e2e_s_per_step" in r else float("nan")
    print("%-28s %-4s value %.3e env-steps/s  us/launch %.2f  e2e %.3e  lanes %s" % (tag, name, v, r["us_per_launch"], e2e, r["lanes_per_env"]), flush=True)
