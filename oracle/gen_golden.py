"""Generate golden fixtures from the UNMODIFIED Python reference (build container only).

    python oracle/gen_golden.py              # writes tests/golden/*.npz
    python oracle/gen_golden.py obs_plugins  # tests/golden/obs_plugins_*.npz
    python oracle/gen_golden.py live         # tests/golden/live_*: what the tests/test_*_live.py tests compare against

Each fixture is a seeded rollout of the reference env (ref_harness.rollout): the full
per-vehicle state after reset and after every env.step, plus obs / reward / terminated /
truncated and the action sequence.  Stepping continues past termination so all
trajectories have fixed length.  tests/test_oracle_golden.py pins the C oracle to these;
the `-m gpu` tests pin the CUDA path to them (teacher-forced and free-running on the
well-conditioned prefix, see DESIGN.md "parity protocol").
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ref_harness as rh  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (env_id, config override, seeds, n_steps, action kind)
CASES = {
    # BASELINE.json configs[0]: highway-fast-v0 defaults (V = 21)
    "highway_fast_v20": ("highway-fast-v0", None, list(range(32)), 30, "discrete5"),
    # configs[1]: highway-fast-v0, vehicles_count = 50 (V = 51)
    "highway_fast_v50": ("highway-fast-v0", {"vehicles_count": 50}, list(range(100, 132)), 30, "discrete5"),
    # highway-v0 defaults: all-pairs collisions, 15 substeps, 4 lanes
    "highway_v50": ("highway-v0", None, list(range(200, 232)), 20, "discrete5"),
    # configs[4] shape: highway-v0, vehicles_count = 100, ContinuousAction (V = 101)
    "highway_v100_continuous": (
        "highway-v0",
        {"vehicles_count": 100, "action": {"type": "ContinuousAction"}},
        list(range(300, 316)),
        12,
        "box2",
    ),
    # (f)2 plugins on the same path: DiscreteAction (action.py:165-196) and the full Kinematics feature list
    "highway_discrete_action": ("highway-v0", {"vehicles_count": 20, "action": {"type": "DiscreteAction"}},
                                list(range(800, 832)), 15, "discrete9"),
    "highway_fast_features": (
        "highway-fast-v0",
        {"observation": {"type": "Kinematics", "vehicles_count": 7, "see_behind": True,
                         "features": ["presence", "x", "y", "vx", "vy", "heading", "cos_h", "sin_h", "cos_d", "sin_d",
                                      "long_off", "lat_off", "ang_off"]}},
        list(range(810, 842)), 20, "discrete5"),
    "highway_fast_features_range": (
        "highway-fast-v0",
        {"observation": {"type": "Kinematics", "vehicles_count": 4, "absolute": True, "clip": False,
                         "features": ["x", "lat_off", "presence", "vx", "heading", "long_off"],
                         "features_range": {"x": [-100, 1500], "vx": [0, 45], "long_off": [0, 2000],
                                            "heading": [-1, 1], "vy": [-3, 3]}}},
        list(range(820, 852)), 20, "discrete5"),
    # roundabout-v0 defaults (Kinematics absolute) and BASELINE configs[3] shape (TimeToCollision)
    "roundabout_kin": ("roundabout-v0", None, list(range(400, 432)), 11, "discrete5"),
    "roundabout_ttc": ("roundabout-v0", {"observation": {"type": "TimeToCollision", "horizon": 10}},
                       list(range(500, 532)), 11, "discrete5"),
    # intersection-v0 defaults (Kinematics, 7 features) and BASELINE configs[2] shape (OccupancyGrid)
    "intersection_kin": ("intersection-v0", None, list(range(600, 632)), 13, "discrete3"),
    "intersection_grid": ("intersection-v0", {"observation": {"type": "OccupancyGrid"}},
                          list(range(700, 732)), 13, "discrete3"),
    # (f)3 connected-lane neighbour search (ConnectedLaneNeighboursMixin, abstract.py:26-37; road.py:509-529)
    "roundabout_v1_kin": ("roundabout-v1", None, list(range(900, 932)), 11, "discrete5"),
    "intersection_v2_kin": ("intersection-v2", None, list(range(910, 942)), 13, "discrete3"),
    # (f)2 MultiAgentAction / MultiAgentObservation: two controlled vehicles
    "intersection_multi_agent": ("intersection-multi-agent-v0", None, list(range(920, 952)), 13, "discrete3x2"),
    # (f)3 scenario builders on the same kernels: merge-v0 (straight + sine lanes, an Obstacle at the ramp's end)
    "merge_kin": ("merge-v0", None, list(range(930, 962)), 18, "discrete5"),
    "merge_v1_kin": ("merge-v1", None, list(range(940, 972)), 18, "discrete5"),
    # two-way-v0: oncoming traffic on ("b","a",0), IDM vehicles with enable_lane_change=False, TimeToCollision horizon 5
    "two_way_ttc": ("two-way-v0", None, list(range(960, 992)), 15, "discrete5"),
    # u-turn-v0: circular U-turn, routed traffic, ego with PURSUIT_TAU = TAU_HEADING, TimeToCollision horizon 16
    "u_turn_ttc": ("u-turn-v0", None, list(range(970, 1002)), 10, "discrete5"),
    "u_turn_v1_ttc": ("u-turn-v1", None, list(range(980, 1012)), 10, "discrete5"),
    # intersection-v1 (ContinuousIntersectionEnv): ContinuousAction with the dynamical BicycleVehicle, 8-column Kinematics;
    # and intersection-v0 with a kinematic ContinuousAction / DiscreteAction ego (plain Vehicle under RegulatedRoad)
    "intersection_v1": ("intersection-v1", None, list(range(1200, 1232)), 13, "box2"),
    "intersection_continuous": ("intersection-v0", {"action": {"type": "ContinuousAction", "longitudinal": True,
                                                               "lateral": True}},
                                list(range(1240, 1272)), 13, "box2"),
    # exit-v0: three highway sections (6 / 7 / 6 lanes) with an exit ramp, routed traffic without lane changes,
    # ExitObservation, goal reward on the exit lane
    "exit_obs": ("exit-v0", None, list(range(1100, 1132)), 18, "discrete5"),
    # the merging vehicle is moved onto the end of the ramp at speed: it runs into the Obstacle (objects.py:104-107)
    "merge_obstacle_hit": ("merge-v0", None, list(range(950, 982)), 6, "discrete5"),
}


def _ram_the_obstacle(env):
    lane = env.road.network.get_lane(("b", "c", 2))
    v = env.road.vehicles[4]
    v.position = lane.position(58.0 + 3.0 * (env.np_random.uniform()), 0.0)
    v.heading = lane.heading_at(60.0)
    v.speed, v.target_speed = 28.0, 30.0
    v.lane_index = v.target_lane_index = ("b", "c", 2)
    v.lane = lane


MUTATE = {"merge_obstacle_hit": _ram_the_obstacle}


def main() -> None:
    os.makedirs(OUT, exist_ok=True)
    only = sys.argv[1:]
    for name, (env_id, over, seeds, T, akind) in CASES.items():
        if only and name not in only:
            continue
        t0 = time.time()
        rng = np.random.default_rng(abs(hash(name)) % (2**31) if False else sum(map(ord, name)))
        per_seed = []
        for seed in seeds:
            if akind == "discrete5":
                actions = rng.integers(0, 5, size=T).astype(np.int64)
            elif akind == "discrete9":
                actions = rng.integers(0, 9, size=T).astype(np.int64)
            elif akind == "discrete3x2":
                actions = rng.integers(0, 3, size=(T, 2)).astype(np.int64)
            elif akind == "discrete3":
                actions = rng.integers(0, 3, size=T).astype(np.int64)
            else:
                actions = rng.uniform(-1, 1, size=(T, 2)).astype(np.float32)
            per_seed.append(rh.rollout(env_id, over, seed, list(actions), pad=32 if env_id.startswith("intersection") else 0,
                                       mutate=MUTATE.get(name)))
        out = {k: np.stack([p[k] for p in per_seed]) for k in per_seed[0].keys()}
        out["seeds"] = np.array(seeds, dtype=np.int64)
        env = rh.make_reference_env(env_id, over)
        import json

        cfg = dict(env.config)
        if not env_id.startswith("highway"):
            env.reset(seed=0)
            out.update(rh.dump_network(env))
        cfg["_others_check_collisions"] = 0 if env_id == "highway-fast-v0" else 1
        cfg["_env_id"] = env_id
        if env_id.startswith("merge"):
            lanes = [li for li, _ in rh.lane_list(env)]
            cfg["_merge_lane"] = lanes.index(("b", "c", 2))
            cfg["_default_side_lanes"] = len(env.road.network.all_side_lanes(env.vehicle.lane_index))
        if env_id.startswith("exit"):
            lanes = [li for li, _ in rh.lane_list(env)]
            n_l = int(cfg["lanes_count"])
            cfg["_exit_lane_a"], cfg["_exit_lane_b"] = lanes.index(("1", "2", n_l)), lanes.index(("2", "exit", 0))
            cfg["_obs_exit_lane"] = lanes.index(("1", "2", n_l))  # get_lane(("1", "2", -1)): the last lane of the road
            cfg["_default_side_lanes"] = n_l  # the controlled vehicle spawns on ("0", "1", 0)
        out["config_json"] = np.array(json.dumps(cfg))
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: {len(seeds)} seeds x {T} steps -> {path} "
              f"({os.path.getsize(path)/1e3:.0f} kB, {time.time()-t0:.1f}s)")

    # reset-only fixtures: pins the numpy-PCG64 spawn restatement on many seeds
    for name, (env_id, over) in {} if only else {
        "reset_highway_fast_v50": ("highway-fast-v0", {"vehicles_count": 50}),
        "reset_highway_v100": ("highway-v0", {"vehicles_count": 100, "action": {"type": "ContinuousAction"}}),
    }.items():
        env = rh.make_reference_env(env_id, over)
        seeds = list(range(1000, 1032))
        states, obs = [], []
        for seed in seeds:
            o, _ = env.reset(seed=seed)
            states.append(rh.dump_state(env))
            obs.append(o)
            # a second reset WITHOUT seed continues the stream (gymnasium autoreset)
            o2, _ = env.reset()
            states.append(rh.dump_state(env))
            obs.append(o2)
        out = {k: np.stack([s[k] for s in states]) for k in states[0].keys()}
        out["obs"] = np.stack(obs)
        out["seeds"] = np.array(seeds, dtype=np.int64)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: -> {path} ({os.path.getsize(path)/1e3:.0f} kB)")


# ------------------------------------------------------------------ observation plugins on every env family
# One short rollout per env id; on every visited state the reference builds each listed observation type with its own
# observation_factory (envs/common/observation.py:772-794) and observes — the plugin registry is orthogonal to the env.
GRID_RICH = {"type": "OccupancyGrid",
             "features": ["presence", "x", "y", "vx", "vy", "cos_h", "sin_h", "long_off", "lat_off", "ang_off", "heading",
                          "cos_d", "sin_d", "on_road"],
             "features_range": {"x": [-100, 100], "y": [-100, 100], "vx": [-20, 20], "vy": [-20, 20]},
             "grid_size": [[-32, 32], [-18, 18]], "grid_step": [4, 3], "align_to_vehicle_axes": True, "clip": False}
OBS_PLUGIN_CASES = {
    "obs_plugins_highway": ("highway-v0", {"vehicles_count": 30}, list(range(2000, 2004)), 8, "discrete5", [
        {"type": "TimeToCollision", "horizon": 10},
        {"type": "OccupancyGrid"},
        {"type": "OccupancyGrid", "grid_size": [[-300, 300], [-10, 10]], "grid_step": [2, 2]},  # the reference's own test
        GRID_RICH,
        {"type": "LidarObservation"},
        {"type": "LidarObservation", "cells": 36, "maximum_range": 90, "normalize": False},
    ]),
    "obs_plugins_intersection": ("intersection-v0", None, list(range(2010, 2014)), 8, "discrete3", [
        {"type": "TimeToCollision", "horizon": 5},
        {"type": "OccupancyGrid", "align_to_vehicle_axes": True, "grid_size": [[-32, 32], [-32, 32]], "grid_step": [4, 4]},
        GRID_RICH,
        {"type": "LidarObservation"},
    ]),
    "obs_plugins_roundabout": ("roundabout-v0", None, list(range(2020, 2024)), 8, "discrete5", [
        {"type": "OccupancyGrid"},
        GRID_RICH,
        {"type": "LidarObservation", "cells": 24},
        {"type": "TimeToCollision", "horizon": 7},
    ]),
    "obs_plugins_merge": ("merge-v0", None, list(range(2030, 2034)), 8, "discrete5", [
        {"type": "LidarObservation", "maximum_range": 120},
        {"type": "OccupancyGrid", "grid_size": [[-60, 60], [-12, 12]], "grid_step": [3, 2]},
        {"type": "TimeToCollision", "horizon": 6},
    ]),
}


def gen_obs_plugins(only) -> None:
    import json

    from highway_env.envs.common.observation import observation_factory

    for name, (env_id, over, seeds, T, akind, obs_cfgs) in OBS_PLUGIN_CASES.items():
        if only and name not in only:
            continue
        rng = np.random.default_rng(sum(map(ord, name)))
        pad = 32 if env_id.startswith("intersection") else 0
        states, obs = [], [[] for _ in obs_cfgs]
        for seed in seeds:
            env = rh.make_reference_env(env_id, over)
            env.reset(seed=seed)
            observers = [observation_factory(env, dict(c)) for c in obs_cfgs]
            hi = 3 if akind == "discrete3" else 5
            for t in range(T + 1):
                states.append(rh.dump_state(env, pad))
                for k, ob in enumerate(observers):
                    obs[k].append(np.asarray(ob.observe()).copy())
                if t < T:
                    env.step(int(rng.integers(0, hi)))
        keys = [k for k in states[0].keys() if all(k in s for s in states)]
        out = {k: np.stack([s[k] for s in states]) for k in keys}
        for k in range(len(obs_cfgs)):
            out[f"obs_{k}"] = np.stack(obs[k])
        env = rh.make_reference_env(env_id, over)
        env.reset(seed=0)
        out.update(rh.dump_network(env))
        cfg = dict(env.config)
        cfg["_env_id"] = env_id
        cfg["_target_speeds"] = [float(x) for x in env.vehicle.target_speeds]
        out["config_json"] = np.array(json.dumps(cfg))
        out["obs_cfgs_json"] = np.array(json.dumps(obs_cfgs))
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: {len(states)} states x {len(obs_cfgs)} observation types -> {path} ({os.path.getsize(path)/1e3:.0f} kB)")


# ------------------------------------------------------------------ fixtures of tests/test_*_live.py
# What those tests compare the oracles against, recorded from the reference on their own seeds (seeds in no fixture
# above) so that they run without it: tests/golden/live_<case>.npz and tests/golden/live_network_configs.json.
LIVE_HIGHWAY = {  # tests/test_oracle_live.py: teacher-forced, one env
    "highway-fast-v0": ({"vehicles_count": 50}, 12, 4242),
    "highway-v0": ({"vehicles_count": 30, "lanes_count": 5, "action": {"type": "ContinuousAction"}}, 6, 77),
}
LIVE_NET = {  # tests/test_net_oracle_live.py: teacher-forced, one env per seed
    "roundabout-v0": ({"observation": {"type": "TimeToCollision", "horizon": 10}}, 11, (31, 32)),
    "roundabout-v1": (None, 11, (33,)),
    "merge-v0": (None, 14, (34, 35)),
    "merge-v1": (None, 14, (36,)),
    "two-way-v0": (None, 10, (37, 38)),
    "u-turn-v0": (None, 10, (39, 40)),
    "u-turn-v1": (None, 10, (41,)),
}
LIVE_INTERSECTION = {  # tests/test_intersection_oracle_live.py: free-running, one env per seed
    ("intersection-v0", "default"): (5000, 6), ("intersection-v0", "OccupancyGrid"): (5100, 6),
    ("intersection-v2", "default"): (5200, 4), ("intersection-multi-agent-v0", "default"): (5300, 4),
}
LIVE_NETWORK_BUILDERS = {  # tests/test_network_config_live.py: RoadNetwork.to_config / from_config
    "roundabout-v0": ("highwayenv_b200.envs.roundabout_env", "make_roundabout_network"),
    "intersection-v0": ("highwayenv_b200.envs.intersection_env", "make_intersection_network"),
    "merge-v0": ("highwayenv_b200.envs.merge_env", "make_merge_network"),
    "two-way-v0": ("highwayenv_b200.envs.two_way_env", "make_two_way_network"),
    "u-turn-v0": ("highwayenv_b200.envs.u_turn_env", "make_u_turn_network"),
}


def live_name(env_id: str, obs: str = "") -> str:
    return "live_" + env_id.replace("-", "_") + ("_" + obs if obs and obs != "default" else "")


def _save(name: str, out: dict) -> None:
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name} -> {path} ({os.path.getsize(path)/1e3:.0f} kB)")


def _rng_words(env) -> np.ndarray:
    m64, st = (1 << 64) - 1, env.np_random.bit_generator.state
    return np.array([st["state"]["state"] >> 64, st["state"]["state"] & m64, st["state"]["inc"] >> 64,
                     st["state"]["inc"] & m64, (int(st["has_uint32"]) << 32) | int(st["uinteger"])], dtype=np.uint64)


def _stack_states(states: list, prefix: str = "") -> dict:
    """dump_state dicts -> {prefix + key: array stacked over steps}."""
    return {prefix + k: np.stack([s[k] for s in states]) for k in states[0]}


def _shared(out: dict, seed: int, env, cfg: dict) -> None:
    """The road network and config, stored once per file: the same for every seed of a case."""
    import json

    net = rh.dump_network(env)
    net["config_json"] = np.array(json.dumps(cfg))
    if "config_json" not in out:
        out.update(net)
    for k, v in net.items():
        assert np.array_equal(out[k], v), (seed, k)


def gen_live_highway(env_id: str) -> None:
    import json

    over, T, seed = LIVE_HIGHWAY[env_id]
    rng = np.random.default_rng(seed)  # the test's action draws, in its order
    cont = (over or {}).get("action", {}).get("type") == "ContinuousAction"
    actions = [rng.uniform(-1, 1, size=2).astype(np.float32) if cont else int(rng.integers(5)) for _ in range(T)]
    out = rh.rollout(env_id, over, seed, actions)
    out["config_json"] = np.array(json.dumps(dict(rh.make_reference_env(env_id, over).config)))
    _save(live_name(env_id), out)


def gen_live_available_actions() -> None:
    """DiscreteMetaAction.get_available_actions (action.py:262-299) on 200 scripted ego placements."""
    env = rh.make_reference_env("highway-fast-v0", {"lanes_count": 3})
    env.reset(seed=0)
    rng = np.random.default_rng(0)
    rows, masks = [], []
    for _ in range(200):
        v = env.vehicle
        lane, si = int(rng.integers(3)), int(rng.integers(3))
        x = float(rng.choice([-3.0, 0.0, 50.0, 9999.0, 10004.99, 10005.0, 10010.0]))
        y = 4.0 * lane + float(rng.uniform(-2, 2))
        v.position, v.lane_index, v.speed_index = np.array([x, y]), ("0", "1", lane), si
        v.lane = env.road.network.get_lane(v.lane_index)
        m = np.zeros(5, dtype=np.bool_)
        m[sorted(set(env.action_type.get_available_actions()))] = True
        rows.append((x, y, lane, si))
        masks.append(m)
    r = np.array(rows, dtype=np.float64)
    _save("live_available_actions", {"x": r[:, 0], "y": r[:, 1], "lane": r[:, 2].astype(np.int64),
                                     "speed_index": r[:, 3].astype(np.int64), "mask": np.stack(masks)})


def gen_live_net(env_id: str) -> None:
    """Per seed, keys prefixed s<seed>_: the state after reset and every step (the vehicle count may differ by seed)."""
    over, T, seeds = LIVE_NET[env_id]
    out = {"seeds": np.array(seeds, dtype=np.int64)}
    for seed in seeds:
        env = rh.make_reference_env(env_id, over)
        obs_ref, _ = env.reset(seed=seed)
        cfg = dict(env.config)
        cfg["_env_id"] = env_id
        if env_id.startswith("merge"):
            lanes = [li for li, _ in rh.lane_list(env)]
            cfg["_merge_lane"] = lanes.index(("b", "c", 2))
            cfg["_default_side_lanes"] = len(env.road.network.all_side_lanes(env.vehicle.lane_index))
        _shared(out, seed, env, cfg)
        p = f"s{seed}_"
        states, obs, rew, term, trunc, acts = [rh.dump_state(env)], [np.asarray(obs_ref)], [], [], [], []
        rng = np.random.default_rng(seed)  # the test's action draws
        for _ in range(T):
            a = int(rng.integers(5))
            o, r, te, tr, _ = env.step(a)
            states.append(rh.dump_state(env))
            obs.append(np.asarray(o))
            rew.append(float(r))
            term.append(bool(te))
            trunc.append(bool(tr))
            acts.append(a)
        out.update(_stack_states(states, p))
        out[p + "obs"], out[p + "reward"] = np.stack(obs), np.array(rew, dtype=np.float64)
        out[p + "terminated"], out[p + "truncated"] = np.array(term), np.array(trunc)
        out[p + "actions"] = np.array(acts, dtype=np.int64)
    _save(live_name(env_id), out)


def gen_live_intersection(env_id: str, obs_type: str) -> None:
    """The reference's side of the free-running comparison: every step until the episode ends or a non-crashed vehicle
    crawls below 1 m/s (tests/parity_utils.py well_conditioned; that step is kept, the test stops before comparing it).
    The seeds' records are concatenated along the step axis; n_steps[i] is the number of steps of seed i."""
    seed0, n = LIVE_INTERSECTION[(env_id, obs_type)]
    over = None if obs_type == "default" else {"observation": {"type": obs_type}}
    out, per_seed = {"seeds": np.arange(seed0, seed0 + n, dtype=np.int64)}, []
    for seed in range(seed0, seed0 + n):
        env = rh.make_reference_env(env_id, over)
        obs_ref, _ = env.reset(seed=seed)
        cfg = dict(env.config)
        A = int(cfg.get("controlled_vehicles", 1))
        _shared(out, seed, env, cfg)
        states, obs, rew, term, trunc, acts, words = [rh.dump_state(env, 32)], [np.asarray(obs_ref)], [], [], [], [], []
        rng = np.random.default_rng(seed)  # the test's action draws
        for _ in range(int(cfg["duration"] * cfg["policy_frequency"]) + 1):
            a = rng.integers(0, 3, size=A)
            o, r, te, tr, _ = env.step(tuple(int(x) for x in a) if A > 1 else int(a[0]))
            st = rh.dump_state(env, 32)
            states.append(st)
            obs.append(np.asarray(o, dtype=np.float64))
            rew.append(float(r))
            term.append(bool(te))
            trunc.append(bool(tr))
            acts.append(a)
            words.append(_rng_words(env))
            k = int(st["count"])
            if np.any(~st["crashed"][:k].astype(bool) & (np.abs(st["speed"][:k]) < 1.0)) or te or tr:
                break
        d = _stack_states(states)  # T + 1 states
        d["obs"] = np.stack(obs)
        d["reward"], d["terminated"], d["truncated"] = np.array(rew, dtype=np.float64), np.array(term), np.array(trunc)
        d["actions"], d["rng_words"] = np.stack(acts).astype(np.int64), np.stack(words)
        per_seed.append(d)
    out.update({k: np.concatenate([d[k] for d in per_seed]) for k in per_seed[0]})
    out["n_steps"] = np.array([len(d["reward"]) for d in per_seed], dtype=np.int64)
    _save(live_name(env_id, obs_type), out)


def _plain(x):
    """A to_config() dict as JSON: arrays and tuples -> lists, numpy scalars -> python."""
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    return x.item() if isinstance(x, np.generic) else x


def gen_live_network_config(env_id: str) -> None:
    """The reference's RoadNetwork.to_config() of the env's road, and what its RoadNetwork.from_config makes of the
    product's to_config() (the dict it was given is stored with it)."""
    import importlib
    import json

    from highway_env.road.road import RoadNetwork

    mod, fn = LIVE_NETWORK_BUILDERS[env_id]
    ours = getattr(importlib.import_module(mod), fn)().to_config()
    env = rh.make_reference_env(env_id, None)
    env.reset(seed=0)
    rec = {"reference": _plain(env.road.network.to_config()), "given": _plain(ours),
           "given_round_trip": _plain(RoadNetwork.from_config(ours).to_config())}
    path = os.path.join(OUT, "live_network_configs.json")
    allrec = {}
    if os.path.exists(path):
        with open(path) as f:
            allrec = json.load(f)
    allrec[env_id] = rec
    with open(path, "w") as f:
        json.dump({k: allrec[k] for k in sorted(allrec)}, f, indent=None, separators=(",", ":"))
        f.write("\n")
    print(f"live_network_configs[{env_id}] -> {path}")


def gen_live(only) -> None:
    """Every case in a fresh interpreter: IntersectionEnv._make_vehicles rewrites IDMVehicle class constants for the
    whole process (envs/intersection_env.py:262-265)."""
    import subprocess

    cases = ([("highway", e) for e in LIVE_HIGHWAY] + [("available_actions", "")] + [("net", e) for e in LIVE_NET]
             + [("intersection", f"{e}:{o}") for e, o in LIVE_INTERSECTION]
             + [("network_config", e) for e in LIVE_NETWORK_BUILDERS])
    for kind, arg in cases:
        if only and kind not in only:
            continue
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "live-case", kind, arg])


def gen_live_case(kind: str, arg: str) -> None:
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    rh._ensure_imports()
    if kind == "highway":
        gen_live_highway(arg)
    elif kind == "available_actions":
        gen_live_available_actions()
    elif kind == "net":
        gen_live_net(arg)
    elif kind == "intersection":
        gen_live_intersection(*arg.split(":"))
    else:
        gen_live_network_config(arg)


if __name__ == "__main__":
    if not rh.reference_available():
        raise SystemExit("reference not mounted; golden fixtures can only be generated in the build container")
    args = sys.argv[1:]
    if args and args[0] == "obs_plugins":
        rh._ensure_imports()
        gen_obs_plugins(args[1:])
    elif args and args[0] == "live":
        gen_live(args[1:])
    elif args and args[0] == "live-case":
        gen_live_case(args[1], args[2] if len(args) > 2 else "")
    else:
        main()
