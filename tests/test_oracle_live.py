"""Oracle vs the reference on seeds that are in no other fixture: what the reference computed on them is recorded in
tests/golden/live_*.npz (`python oracle/gen_golden.py live`).  Short on purpose; the golden fixtures cover more seeds."""
import numpy as np
import pytest

import hwy_oracle as ho
from parity_utils import compare_state, load_golden

NOT_STATE = ("obs", "reward", "terminated", "truncated", "actions", "rng_words", "config_json", "config")


def golden_states(g: dict) -> list:
    """The reference's state after reset and after every step (ref_harness.dump_state layout)."""
    keys = [k for k in g if k not in NOT_STATE]
    return [{k: g[k][t] for k in keys} for t in range(len(g["reward"]) + 1)]


@pytest.mark.parametrize("env_id,over,T,seed", [
    ("highway-fast-v0", {"vehicles_count": 50}, 12, 4242),
    ("highway-v0", {"vehicles_count": 30, "lanes_count": 5, "action": {"type": "ContinuousAction"}}, 6, 77),
])
def test_oracle_matches_live_reference(env_id, over, T, seed):
    g = load_golden("live_" + env_id.replace("-", "_"))
    assert len(g["reward"]) == T
    states = golden_states(g)
    cfg = dict(g["config"])
    assert cfg["vehicles_count"] == over["vehicles_count"]
    cfg["_others_check_collisions"] = 0 if env_id == "highway-fast-v0" else 1
    oc = ho.cfg_from_dict(cfg)
    ob = ho.OracleBatch(oc, 1, seeds=[seed])
    assert np.array_equal(ob.reset()[0], g["obs"][0])
    for t in range(T):
        ob.load_state(0, states[t])  # teacher-forced
        a = g["actions"][t]
        act = [int(a)] if oc.action_type == 0 else a[None].astype(np.float32)
        oo, ro, teo, tro = ob.step(act)
        got = {k: ob.a[k][0] for k in ob.a if k not in ("speed_index", "time")}
        got["speed_index"] = ob.a["speed_index"][0]
        assert compare_state(states[t + 1], got, ctx=f"{env_id} t={t}") < 1e-9
        assert abs(g["reward"][t] - ro[0]) < 1e-12
        assert bool(g["terminated"][t]) == bool(teo[0]) and bool(g["truncated"][t]) == bool(tro[0])
        assert np.max(np.abs(g["obs"][t + 1] - oo[0])) <= 1e-6


def test_available_actions_mask_matches_live_reference():
    """DiscreteMetaAction.get_available_actions (action.py:262-299) vs the product's tensor form (CPU tensors)"""
    import torch

    from highwayenv_b200.envs.highway_env import available_actions_mask

    g = load_golden("live_available_actions")
    table = torch.tensor([[0.0, 4.0 * l, 1.0, 0.0, -0.0, 1.0, 10000.0, 4.0] for l in range(3)], dtype=torch.float64)
    assert len(g["mask"]) == 200
    for x, y, lane, si, ref in zip(g["x"], g["y"], g["lane"], g["speed_index"], g["mask"]):
        m = available_actions_mask(torch.tensor([x], dtype=torch.float64), torch.tensor([y], dtype=torch.float64),
                                   torch.tensor([int(lane)]), torch.tensor([int(si)]), table, 3)[0].numpy()
        assert np.array_equal(m.astype(bool), ref), (lane, x, y, si)
