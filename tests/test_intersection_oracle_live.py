"""intersection ids against the reference on seeds that are not in the other fixtures, FREE-RUNNING (no state injection
after the common seed): state, reward, flags, observation and the numpy generator words after every step.  What the
reference computed on these seeds is recorded in tests/golden/live_intersection_*.npz (`python oracle/gen_golden.py
live`, every case in its own process: IntersectionEnv._make_vehicles mutates IDMVehicle class constants process-wide,
envs/intersection_env.py:262-265)."""
import numpy as np
import pytest

import net_oracle as no
from parity_utils import load_golden
from test_net_oracle_golden import compare_inter

PER_STEP = ("reward", "terminated", "truncated", "actions", "rng_words")


@pytest.mark.parametrize("env_id,obs,seed0,n", [
    ("intersection-v0", "default", 5000, 6), ("intersection-v0", "OccupancyGrid", 5100, 6),
    ("intersection-v2", "default", 5200, 4), ("intersection-multi-agent-v0", "default", 5300, 4),
])
def test_intersection_free_running_vs_live_reference(env_id, obs, seed0, n):
    g = load_golden("live_" + env_id.replace("-", "_") + ("" if obs == "default" else "_" + obs))
    assert list(g["seeds"]) == list(range(seed0, seed0 + n))
    cfg = g["config"]
    assert obs == "default" or cfg["observation"]["type"] == obs
    A = int(cfg.get("controlled_vehicles", 1))
    net = {k: v for k, v in g.items() if k.startswith("net_")}
    per_step = set(PER_STEP)
    state_keys = [k for k in g if k not in per_step | set(net) | {"seeds", "n_steps", "obs", "config_json", "config"}]
    worst, compared, s0, p0 = 0.0, 0, 0, 0  # s0: first state of the seed; p0: its first per-step record
    for seed, T in zip(g["seeds"], g["n_steps"]):
        ob = no.IntersectionOracle(no.graph_from_arrays(net), no.cfg_from_dict(cfg), 1, net, cfg)
        ob.reset_env(0, seed=int(seed))
        st = {k: g[k][s0] for k in state_keys}
        compare_inter(st, ob.a, 0, f"{env_id} seed {seed} reset", tol=1e-8)
        obs_ref = g["obs"][s0]
        assert np.max(np.abs(ob.observe().reshape(obs_ref.shape) - obs_ref)) <= 1e-6
        for t in range(T):
            a = g["actions"][p0 + t]
            oo, ro, teo, tro = ob.step(a.reshape(1, A).astype(np.int32) if A > 1 else a.astype(np.int32))
            ctx = f"{env_id} seed {seed} t={t}"
            st = {k: g[k][s0 + t + 1] for k in state_keys}
            k = int(st["count"])
            # utils.not_zero(speed) in the steering law (controller.py:166,178) amplifies 1-ulp libm differences by > 1e6
            # per policy step once a non-crashed vehicle crawls below ~1 m/s (tests/parity_utils.py well_conditioned):
            # free-running parity is asserted up to that point, teacher-forced parity (the fixtures) on every state
            if np.any(~st["crashed"][:k].astype(bool) & (np.abs(st["speed"][:k]) < 1.0)):
                break
            compare_inter(st, ob.a, 0, ctx, tol=1e-5)
            worst = max(worst, float(np.max(np.abs(st["x"][:k] - ob.a["x"][0][:k]))),
                        float(np.max(np.abs(st["speed"][:k] - ob.a["speed"][0][:k]))))
            r, te, tr = g["reward"][p0 + t], bool(g["terminated"][p0 + t]), bool(g["truncated"][p0 + t])
            assert abs(r - ro[0]) <= 1e-6 and te == bool(teo[0]) and tr == bool(tro[0]), ctx
            o = g["obs"][s0 + t + 1]
            assert np.max(np.abs(o.reshape(-1) - oo[0].reshape(-1))) <= 1e-4, ctx
            assert [int(x) for x in ob.rng_words(0)] == [int(x) for x in g["rng_words"][p0 + t]], ctx + " numpy stream"
            compared += 1
            if te or tr:
                break
        s0, p0 = s0 + T + 1, p0 + T
    assert s0 == len(g["obs"]) and p0 == len(g["reward"])
    assert compared >= 3 * n, (compared, worst)
