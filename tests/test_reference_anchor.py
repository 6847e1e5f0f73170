"""Wide anchor of the C oracle on the UNMODIFIED reference (needs the reference checkout or the staged oracle/_ref; skipped
elsewhere): hundreds of fresh trajectories per env type, generated here by tests/golden/make_golden.py's own harness
(MT19937 target layouts of the reference's reset injected, detection draws keyed), against the C oracle that the GPU
parity tests at configuration size are checked with.  Everything is compared with np.array_equal -- float64 positions
included -- like the committed fixtures, only on many more envs: 512 x 200 steps flight_easy 3a15t (BASELINE.json
configs[1] is 4096 of these), 256 x 200 steps 5a15t AM2 / AM3, 6 x 60 steps flight (the reference takes 16 ms per step
there), 96 x 80 steps search_env."""
import os
import sys

import numpy as np
import pytest

from oracle import c_oracle
from oracle.py_envs import FlightSpec, SearchSpec

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))

pytestmark = pytest.mark.needs_reference


def flight_kwargs(g, variant):
    n, m, M, R, T, am, tm, base, seed = [int(v) for v in g["meta"]]
    vel, d, safe, fd = [float(v) for v in g["fmeta"]]
    as_num = lambda v: int(v) if float(v).is_integer() else v
    return dict(n_agents=n, target_num=m, map_size=M, view_range=R, time_limit=T, agent_mode=am, target_mode=tm, velocity=as_num(vel),
                detect_prob=d, safe_dist=as_num(safe), force_dist=as_num(fd), variant=variant), base, seed


@pytest.mark.parametrize("cls,n,am,E,T,kw", [
    ("FlightSearchEnvEasy", 3, 0, 512, 200, {}),
    ("FlightSearchEnvEasy", 5, 2, 256, 200, {}),
    ("FlightSearchEnvEasy", 5, 3, 256, 200, {}),
    ("FlightSearchEnv", 3, 0, 6, 60, {"map_steps": (1, 5, 20, 60)}),
])
def test_c_oracle_equals_raw_reference_on_many_envs(cls, n, am, E, T, kw):
    import make_golden as mg
    g = mg.run_flight(cls, n, am, E=E, T=T, env_id_base=20_000, **kw)
    variant = "easy" if cls == "FlightSearchEnvEasy" else "probmap"
    spec_kw, base, seed = flight_kwargs(g, variant)
    spec = FlightSpec(**spec_kw)
    c_oracle.set_threads(os.cpu_count() or 1)
    b = c_oracle.FlightBatch(spec, None, seed, base, E)
    b.reset(targets=g["tgt_xy"], init=True)
    assert np.array_equal(b.found, g["init_found"]) and np.array_equal(b.xy, g["init_xy"])
    for t in range(T):
        r, term, win = b.step(g["actions"][t])
        where = (cls, n, am, t)
        assert np.array_equal(b.found, g["found"][t]), where
        assert np.array_equal(r, g["reward"][t]), where
        assert np.array_equal(term, g["terminated"][t]) and np.array_equal(win, g["win"][t]), where
        assert np.array_equal(b.time_step, g["time_step"][t]), where
        assert np.array_equal(b.xy, g["xy"][t]) and np.array_equal(b.yaw, g["yaw"][t]), where       # float64, bit for bit
        if t % 25 == 24:
            obs, state = b.obs_state()
            assert np.array_equal(obs, g["obs"][t]) and np.array_equal(state, g["state"][t]), where
        if variant == "probmap" and (t + 1) in g["map_steps"]:
            assert np.array_equal(b.map, g["maps"][list(g["map_steps"]).index(t + 1)]), where
    c_oracle.set_threads(1)
    assert int(g["terminated"][-1].sum()) > 0 or variant == "probmap"


def test_c_oracle_search_equals_raw_reference_on_many_envs():
    import make_golden as mg
    n, m, M, R, E, T = 3, 15, 50, 7, 96, 80
    g = mg.run_search(n, m, M, R, 0, 0, E=E, T=T, env_id_base=30_000)
    spec = SearchSpec(n_agents=n, target_num=m, map_size=M, view_range=R, agent_mode=0, target_mode=0)
    b = c_oracle.SearchBatch(spec, 0, 30_000, E)
    b.reset(cells=g["cells"])
    assert np.array_equal(b.pos, g["init_pos"]) and np.array_equal(b.freq, g["init_freq"])
    for t in range(T):
        _, _, avail = b.views(want_obs=False, want_state=False)
        assert np.array_equal(avail, g["avail"][t]), t
        r, term = b.step(g["actions"][t])
        assert np.array_equal(r, g["reward"][t]) and np.array_equal(term, g["terminated"][t]), t
        assert np.array_equal(b.pos, g["pos"][t]) and np.array_equal(b.found, g["found"][t]), t
        if t % 20 == 19:
            obs, state, _ = b.views()
            assert np.array_equal(obs, g["obs"][t].astype(np.float32)) and np.array_equal(state, g["state"][t].astype(np.float32)), t
    assert np.array_equal(b.freq, g["freq"])
