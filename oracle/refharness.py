"""Harness around the UNMODIFIED reference envs -- TEST INFRASTRUCTURE.

Usable where the reference checkout is present (``COOPSEARCH_REFERENCE``, else
BASELINE.json's ``reference_path``: ``oracle/build_ref.py: source``), or where the
unmodified copies staged from it under ``oracle/_ref`` exist (git-ignored).  It is used
by ``tests/golden/make_golden.py`` to generate the committed golden fixtures, by
the ``needs_reference`` CPU tests to pin the oracle restatement against the real
thing, and by ``bench.py``'s CPU legs (the reference arm).  Nothing in the product
package imports it.

What it does:
  * injects stub ``matplotlib`` modules (the reference imports matplotlib at
    module top level: env/flight_env_easy.py:2-3, env/flight_env.py:2-3,
    env/search_env.py:4-5,49-53; matplotlib is not installed here);
  * imports the reference env classes from that tree;
  * replaces the detection draw ``np.random.rand()`` (env/flight_env_easy.py:238,
    env/flight_env.py:248) by the keyed Philox draw of oracle/philox.py, reading
    the loop indices ``i`` (agent) and ``j`` (target) from the caller's frame.
"""
import contextlib
import io
import os
import sys
import types

import numpy as np

from . import build_ref, philox

_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")     # oracle/build_ref.py: unmodified copies


REFERENCE_ROOT = build_ref.source() or _STAGED


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "env", "flight_env_easy.py"))


def _install_matplotlib_stub():
    if "matplotlib" in sys.modules:
        return

    class _Anything:
        def __init__(self, *a, **k):
            pass

        def __call__(self, *a, **k):
            return _Anything()

        def __getattr__(self, name):
            return _Anything()

        def __getitem__(self, item):
            return _Anything()

    mpl = types.ModuleType("matplotlib")
    pyplot = types.ModuleType("matplotlib.pyplot")
    patches = types.ModuleType("matplotlib.patches")
    gridspec = types.ModuleType("matplotlib.gridspec")
    def _pyplot_attr(name):
        if name.startswith("__"):            # keep inspect / importlib happy (torch walks sys.modules)
            raise AttributeError(name)
        return _Anything()
    pyplot.__getattr__ = _pyplot_attr
    patches.Circle = _Anything
    gridspec.GridSpec = _Anything
    mpl.pyplot, mpl.patches, mpl.gridspec = pyplot, patches, gridspec
    sys.modules.update({"matplotlib": mpl, "matplotlib.pyplot": pyplot,
                        "matplotlib.patches": patches, "matplotlib.gridspec": gridspec})


_ref_modules = {}


def import_reference():
    """Returns dict with the reference env classes."""
    if _ref_modules:
        return _ref_modules
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    _install_matplotlib_stub()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with contextlib.redirect_stdout(io.StringIO()):
        from env.flight_env_easy import FlightSearchEnvEasy
        from env.flight_env import FlightSearchEnv
        from env.search_env import SearchEnv
        try:
            from env.simple_spread import SimpleSpreadEnv
        except ImportError:          # an oracle/_ref staged before simple_spread was added
            SimpleSpreadEnv = None
    _ref_modules.update(FlightSearchEnvEasy=FlightSearchEnvEasy, FlightSearchEnv=FlightSearchEnv,
                        SearchEnv=SearchEnv, SimpleSpreadEnv=SimpleSpreadEnv)
    return _ref_modules


def load_targets_reference_semantics(path):
    """Same parsing rule as main.py:19-32 (skip header, whitespace split, 6 columns)."""
    cols = {"x": [], "y": [], "deter": [], "priority": [], "dx": [], "dy": []}
    with open(path, "r") as fh:
        rows = fh.readlines()[1:]
    for row in rows:
        tok = row.split()
        if not tok:
            continue
        cols["x"].append(float(tok[0])); cols["y"].append(float(tok[1]))
        cols["deter"].append(tok[2]); cols["priority"].append(int(tok[3]))
        cols["dx"].append(float(tok[4])); cols["dy"].append(float(tok[5]))
    return cols


def make_args(env="flight_easy", **over):
    """Namespace with the defaults of common/arguments.py:28-34,269-284."""
    a = types.SimpleNamespace(
        env=env, map_size=50, target_num=15, target_mode=0, target_dir="./targets/",
        agent_mode=0, n_agents=3, view_range=7,
        agent_velocity=1, time_limit=200, turn_limit=np.pi / 4, flight_height=8000,
        safe_dist=1, detect_prob=0.9, wrong_alarm_prob=0.1, force_dist=3, search_env=True,
        conv=(env == "flight"))
    for k, v in over.items():
        setattr(a, k, v)
    return a


class KeyedDraws:
    """Context that swaps ``np.random.rand`` for the keyed Philox detection draw.

    The harness sets ``.t`` before each reference call: 0 for ``reset`` (the
    ``_update_obs`` inside reset, env/flight_env_easy.py:182), k for the k-th
    ``step`` (1-based)."""

    def __init__(self, seed, env_id, episode=0):
        self.seed, self.env_id, self.episode, self.t = seed, env_id, episode, 0
        self._saved = None
        self.n_draws = 0

    def _rand(self, *shape):
        if shape:
            raise RuntimeError("keyed draw only replaces scalar np.random.rand()")
        frame = sys._getframe(1)
        if frame.f_code.co_name != "_update_obs":
            # e.g. target_mode 1 placement (env/flight_env_easy.py:124): keep the MT19937 stream
            return self._saved()
        loc = frame.f_locals
        i, j = loc["i"], loc["j"]
        self.n_draws += 1
        return philox.detect_draw(self.seed, self.env_id, self.episode, self.t, i, j) / 4294967296.0

    def __enter__(self):
        self._saved = np.random.rand
        np.random.rand = self._rand
        return self

    def __exit__(self, *exc):
        np.random.rand = self._saved
        return False


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)
