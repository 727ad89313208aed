"""Network oracle vs the reference on seeds that are not in the other golden fixtures: what the reference computed on
them is recorded in tests/golden/live_*.npz (`python oracle/gen_golden.py live`).  Teacher-forced, one env at a time.
intersection ids are in tests/test_intersection_oracle_live.py (free-running)."""
import numpy as np
import pytest

import net_oracle as no
from parity_utils import compare_state, load_golden

NOT_STATE = ("obs", "reward", "terminated", "truncated", "actions")


def _state(st, V):
    st = dict(st)
    st["target_lane"] = np.where(st["target_lane"] < 0, st["lane"], st["target_lane"])
    if "route" not in st:
        st["route"], st["route_len"] = np.zeros((V, no.NET_MAX_ROUTE), dtype=np.int32), np.zeros(V, dtype=np.int32)
    if "kind" in st:
        st["impact"] = np.where((st["kind"] == 3)[:, None], np.nan, st["impact"])  # objects: inert zeros
    else:
        st["kind"] = np.array([1] + [0] * (V - 1), dtype=np.int32)
    st.setdefault("count", V)
    st.setdefault("is_yielding", np.zeros(V, dtype=np.int32))
    st.setdefault("road_steps", 0)
    return st


@pytest.mark.parametrize("env_id,over,T,seeds", [
    ("roundabout-v0", {"observation": {"type": "TimeToCollision", "horizon": 10}}, 11, (31, 32)),
    ("roundabout-v1", None, 11, (33,)),
    ("merge-v0", None, 14, (34, 35)),
    ("merge-v1", None, 14, (36,)),
    ("two-way-v0", None, 10, (37, 38)),
    ("u-turn-v0", None, 10, (39, 40)),
    ("u-turn-v1", None, 10, (41,)),
])
def test_net_oracle_matches_live_reference(env_id, over, T, seeds):
    g = load_golden("live_" + env_id.replace("-", "_"))
    assert tuple(g["seeds"]) == seeds
    cfg = g["config"]
    assert cfg["_env_id"] == env_id and (over is None or cfg["observation"]["type"] == over["observation"]["type"])
    graph = no.graph_from_arrays(g)
    for seed in seeds:
        p = f"s{seed}_"
        r = {k[len(p):]: v for k, v in g.items() if k.startswith(p)}
        assert len(r["reward"]) == T
        states = [{k: r[k][t] for k in r if k not in NOT_STATE} for t in range(T + 1)]
        V = len(states[0]["x"])
        ob = no.NetOracleBatch(graph, no.cfg_from_dict(cfg, n_vehicles=V), 1)
        ob.load_state(0, _state(states[0], V))
        assert np.max(np.abs(ob.observe().reshape(r["obs"][0].shape) - r["obs"][0])) <= 1e-6
        for t in range(T):
            ob.load_state(0, _state(states[t], V))  # teacher-forced
            oo, ro, teo, tro = ob.step([int(r["actions"][t])])
            got = {k: ob.a[k][0] for k in ob.a if k not in ("speed_index", "time")}
            got["speed_index"] = ob.a["speed_index"][0]
            ctx = f"{env_id} seed {seed} t={t}"
            assert compare_state(_state(states[t + 1], V), got, ctx=ctx) < 1e-9
            assert abs(r["reward"][t] - ro[0]) < 1e-9, ctx
            assert bool(r["terminated"][t]) == bool(teo[0]) and bool(r["truncated"][t]) == bool(tro[0]), ctx
            o = r["obs"][t + 1]
            assert np.max(np.abs(o - oo[0].reshape(o.shape))) <= 1e-6, ctx
