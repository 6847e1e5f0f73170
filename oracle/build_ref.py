"""Stages the UNMODIFIED reference into oracle/_ref/ -- TEST / BASELINE INFRASTRUCTURE.

The reference (WZN1ng/Cooperative-Search) is pure Python: there is nothing to compile.  So that the CPU baseline of
bench.py (`--impl reference`, `cpu_baseline`) can time the reference's own code path on a machine the reference
checkout is not on, `__graft_entry__.build()` copies the files that path needs, byte for byte, from the reference
checkout (`source()`) into the git-ignored oracle/_ref/ (which a copy of the tree carries along).  Nothing is edited;
MANIFEST.json records the sha256 of every staged file.  Only tests/, smoke() and bench.py's CPU legs use it.
"""
import hashlib
import json
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DST = os.path.join(HERE, "_ref")
# the env-step path and its caller (common/rollout.py + the Agents facade it needs for alg=random)
FILES = [
    "env/flight_env_easy.py", "env/flight_env.py", "env/search_env.py", "env/simple_spread.py",
    "common/rollout.py", "common/arguments.py", "common/replay_buffer.py",
    "agent/agent.py",
    "policy/qmix.py", "policy/vdn.py", "policy/dop.py", "policy/reinforce.py", "policy/trandition.py",
    "network/base_net.py", "network/mixer_net.py", "network/qmix_net.py", "network/vdn_net.py", "network/offpg_net.py",
    "flight_targets.txt",
]


def source():
    """The reference checkout: the COOPSEARCH_REFERENCE environment variable, else the reference_path that BASELINE.json
    declares.  None when neither holds the reference."""
    root = os.environ.get("COOPSEARCH_REFERENCE")
    if not root:
        with open(os.path.join(HERE, "..", "BASELINE.json")) as fh:
            root = json.load(fh).get("reference_path")
    return root if root and os.path.isfile(os.path.join(root, "env", "flight_env_easy.py")) else None


def available():
    return os.path.isfile(os.path.join(REF_DST, "env", "flight_env_easy.py"))


def stage(force=False):
    """Copies the reference files into oracle/_ref/ when the reference checkout is present.  Returns the staged root or
    None."""
    src_root = source()
    if src_root is None:
        return REF_DST if available() else None
    manifest = {}
    for rel in FILES:
        src, dst = os.path.join(src_root, rel), os.path.join(REF_DST, rel)
        if not os.path.isfile(src):
            continue
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if force or not os.path.exists(dst) or open(src, "rb").read() != open(dst, "rb").read():
            shutil.copyfile(src, dst)
        manifest[rel] = hashlib.sha256(open(dst, "rb").read()).hexdigest()
    with open(os.path.join(REF_DST, "MANIFEST.json"), "w") as fh:
        json.dump({"source": "WZN1ng/Cooperative-Search (unmodified copies)", "sha256": manifest}, fh, indent=1)
    return REF_DST


if __name__ == "__main__":
    print(stage(force=True))
