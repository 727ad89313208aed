"""RoadNetwork.to_config / from_config (road/road.py:370-389; lane.py:214-233, 290-309, 360-384) on the host lane table,
against what the reference's own to_config / from_config produced, recorded in tests/golden/live_network_configs.json
(`python oracle/gen_golden.py live`)."""
import json
import os

import numpy as np
import pytest

from parity_utils import GOLDEN

BUILDERS = {
    "roundabout-v0": ("highwayenv_b200.envs.roundabout_env", "make_roundabout_network"),
    "intersection-v0": ("highwayenv_b200.envs.intersection_env", "make_intersection_network"),
    "merge-v0": ("highwayenv_b200.envs.merge_env", "make_merge_network"),
    "two-way-v0": ("highwayenv_b200.envs.two_way_env", "make_two_way_network"),
    "u-turn-v0": ("highwayenv_b200.envs.u_turn_env", "make_u_turn_network"),
}


def strip(cfg):
    """drop the rendering-only line_types and turn arrays / numpy scalars into plain python"""
    out = {}
    for f, tos in cfg.items():
        out[f] = {}
        for t, lanes in tos.items():
            out[f][t] = []
            for ld in lanes:
                c = {k: (np.asarray(v).tolist() if isinstance(v, (list, tuple, np.ndarray)) else
                         (bool(v) if isinstance(v, (bool, np.bool_)) else float(v)))
                     for k, v in ld["config"].items() if k != "line_types"}
                out[f][t].append({"class_path": ld["class_path"], "config": c})
    return out


def plain(x):
    """a to_config() dict as it reads back from JSON"""
    return json.loads(json.dumps(x, default=lambda v: v.tolist()))


@pytest.mark.parametrize("env_id", sorted(BUILDERS))
def test_to_config_and_from_config_round_trip(env_id):
    import importlib

    from highwayenv_b200.road.network import NetworkTable

    mod, fn = BUILDERS[env_id]
    ours = getattr(importlib.import_module(mod), fn)()
    with open(os.path.join(GOLDEN, "live_network_configs.json")) as f:
        rec = json.load(f)[env_id]
    ref_cfg = rec["reference"]  # the reference's env.road.network.to_config() after reset(seed=0)
    # 1. our dict equals the reference's (insertion order included), rendering attributes aside
    a, b = strip(ours.to_config()), strip(ref_cfg)
    assert list(a) == list(b)
    for f in a:
        assert list(a[f]) == list(b[f]), f
        for t in a[f]:
            assert a[f][t] == b[f][t], (f, t)
    # 2. from_config(reference dict) rebuilds the device lane table bit for bit
    back = NetworkTable.from_config(ref_cfg)
    for k, v in ours.arrays.items():
        assert np.array_equal(back.arrays[k], v), k
    assert np.array_equal(back.succ, ours.succ) and back.index == ours.index
    # 3. and our own dict round-trips through the reference's from_config: the reference was given exactly this dict
    assert plain(ours.to_config()) == rec["given"]
    assert strip(rec["given_round_trip"]) == b
