#!/usr/bin/env python
"""bench.py — env-steps/s of the batched HighwayEnv hot path on B200, every BASELINE.json config in one line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--envs-per-gpu E] [--configs cfg2,cfg3] [--gather-obs] [--no-cpu-baseline] [--dump-outputs DIR]

Headline (top-level keys of the JSON line) = BASELINE.json configs[1]: highway-fast-v0, vehicles_count=50
(V = 51), 3 lanes, 5 substeps per step, Kinematics observation, DiscreteMetaAction, 4096 envs per GPU
(8192 per GPU at N = 8, so that the 8-GPU point is north_star's 65 536 envs), i.i.d. uniform random actions,
SameStep autoreset on the device.  One bench "step" = one env.step of every env of the batch.
Multi-GPU: one process per GPU (torchrun), each rank owns a contiguous env-index range; no collective on the
data path (weak scaling).  At N > 1 the line also carries a strong-scaling point (32 768 envs in total) and,
with --gather-obs, the cost of the optional NCCL all-gather of the whole-batch observation.

`configs` holds one entry per BASELINE.json config (cfg1..cfg5), each with
  value        device-timed throughput (CUDA events around every env.step on the launch stream, actions
               resident in HBM, L2 flushed between timed steps, max over ranks);
  e2e          the same metric through the public API with HOST buffers (pinned actions H2D, obs / reward /
               terminated / truncated D2H, sync every step; through env.host_stepper()'s CUDA graph when the
               env offers one);
  roofline     the dominant kernel against the measured HBM peak (algorithmic bytes of SURVEY.md §8(d)), plus
               the compute-side figures of the committed ncu capture (issue-active, fp64 pipe, thread
               instructions per vehicle-substep) because none of these kernels is bandwidth bound;
  cpu_baseline the C oracle port of the same workload on the host cores: one pinned single-threaded process
               per core, >= 3 s timed, median of 3, load average and affinity recorded; and, quoted as
               "measured elsewhere", the per-core rate of the UNMODIFIED Python reference from
               profiles/r2_python_reference.json (tools/time_reference.py, build container).

--dump-outputs DIR: after the timed steps, what the last timed env.step of every config returned to its caller
(observation, reward, terminated, truncated and the info arrays) as DIR/<config>_<name>.npy in float32 / float64, rank 0's
envs only; the inputs (reset seeds, action streams) are fixed, so two builds can be compared output for output.

--impl reference: the CPU arm of the headline config alone (the Python reference cannot travel to the GPU
box: /root/reference is absent there and gymnasium is not installed; the C port is its line-cited restatement).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (batched), highway-fast-v0 50 veh"
UNIT = "env-steps/s"
HEADLINE = "cfg2"
STRONG_TOTAL_ENVS = 32768
DUMP_LIMIT_BYTES = 64 << 20  # --dump-outputs: above this, a fixed seeded sample of the envs is written

# SURVEY.md §8(d): algorithmic bytes per env-step = 2*V*B_state + B_action + B_obs + 6
CONFIGS = {
    "cfg1": dict(
        baseline="highway-fast-v0, 1 env, vehicles_count=20, Kinematics, DiscreteMetaAction (CPU plumbing case; "
                 "batched here)",
        env_id="highway-fast-v0", config=None, envs_per_gpu=4096, actions="discrete5", vehicles=21, substeps=5,
        algo_bytes=2 * 21 * 96 + 4 + 100 + 6, kernel="highway_step_kernel<32, true>", ncu="r2_ncu_highway_step_v21.json"),
    "cfg2": dict(
        baseline="highway-fast-v0, 4096 batched envs, vehicles_count=50, Kinematics, 1xB200",
        env_id="highway-fast-v0", config={"vehicles_count": 50}, envs_per_gpu=4096, actions="discrete5",
        vehicles=51, substeps=5, algo_bytes=2 * 51 * 96 + 4 + 100 + 6, kernel="highway_step_kernel<64, true>",
        ncu="r2_ncu_highway_step_v51.json"),
    "cfg3": dict(
        baseline="intersection-v0, 8192 envs, IDM + priority-yield, OccupancyGrid observation, 1xB200",
        env_id="intersection-v0", config={"observation": {"type": "OccupancyGrid"}}, envs_per_gpu=8192,
        actions="discrete3", vehicles=32, substeps=15, algo_bytes=2 * 32 * 128 + 4 + 1936 + 6,
        kernel="network_step_kernel<16|32, regulated>", ncu="r2_ncu_network_step_intersection.json"),
    "cfg4": dict(
        baseline="roundabout-v0, 16384 envs (2 x 8192), CircularLane path, TimeToCollision observation, 2xB200",
        env_id="roundabout-v0", config={"observation": {"type": "TimeToCollision", "horizon": 10}},
        envs_per_gpu=8192, actions="discrete5", vehicles=5, substeps=15, algo_bytes=2 * 5 * 128 + 4 + 360 + 6,
        kernel="network_step_kernel<8>", ncu="r2_ncu_network_step_roundabout.json"),
    "cfg5": dict(
        baseline="highway-v0, 65536 envs sharded 8xB200 (8192 per GPU), vehicles_count=100, Kinematics, "
                 "ContinuousAction",
        env_id="highway-v0", config={"vehicles_count": 100, "action": {"type": "ContinuousAction"}},
        envs_per_gpu=8192, actions="box2", vehicles=101, substeps=15, algo_bytes=2 * 101 * 96 + 8 + 100 + 6,
        kernel="highway_step_kernel<128, true>", ncu="r2_ncu_highway_step_v101.json"),
}


def workload_name(key: str) -> str:
    c = CONFIGS[key]
    return (f"{c['env_id']} {json.dumps(c['config']) if c['config'] else 'defaults'}, V={c['vehicles']}, "
            f"{c['substeps']} substeps/step, SameStep autoreset")


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region (B200_PROFILING.md clocks line).

    The headline's timed region is tens of milliseconds, shorter than one `nvidia-smi -lms` period, so the samples come
    from NVML directly (the library nvidia-smi reads, via nvidia-ml-py) on a thread polling every `period` seconds; the
    NVML calls release the GIL.  Without NVML bindings: one nvidia-smi query loop, which needs a region of >= 0.2 s."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, uuid: str = None, period: float = 0.004):
        self.gpu_index, self.uuid, self.period = gpu_index, uuid, period
        self.sm, self.mx, self.reasons, self.power = [], [], set(), []
        self.source, self.nvml, self.handle, self.proc, self.thread = None, None, None, None, None
        self._stop = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            try:  # the CUDA ordinal is not the NVML index under CUDA_VISIBLE_DEVICES: prefer the UUID
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml, self.source = pynvml, "nvml"
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
        except Exception:
            self.nvml = None

    def _poll_once(self):
        n, h = self.nvml, self.handle
        self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
        try:
            get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = int(get(h))
            for bit, name in self.REASONS.items():
                if bits & bit:
                    self.reasons.add(name)
        except Exception:
            pass
        try:
            self.power.append(n.nvmlDeviceGetPowerUsage(h) / 1000.0)
        except Exception:
            pass

    def _poll(self):
        while not self._stop.is_set():
            try:
                self._poll_once()
            except Exception:
                pass
            self._stop.wait(self.period)

    def _read_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.sm.append(float(r[1]))
                self.mx.append(float(r[2]))
                for k, nme in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                continue

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.nvml is not None:
            try:
                self._poll_once()  # one more inside the region's closing synchronize window
            except Exception:
                pass
            self._stop.set()
            if self.thread:
                self.thread.join(timeout=1)
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML bindings and no nvidia-smi"], "samples": 0}
        out = {
            "sm_mhz": statistics.median(self.sm) if self.sm else None,
            "sm_min_mhz": min(self.sm) if self.sm else None,
            "sm_max_mhz": max(self.mx) if self.mx else None,
            "reasons": sorted(self.reasons),
            "samples": len(self.sm),
            "source": self.source,
        }
        if self.power:
            out["power_w"] = statistics.median(self.power)
        return out


# ------------------------------------------------------------------ CPU arm (C oracle port, pinned processes)
def host_cores() -> list:
    try:
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return list(range(os.cpu_count() or 1))


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _golden(name: str) -> dict:
    import numpy as np

    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"), allow_pickle=False)
    d = {k: z[k] for k in z.files}
    d["config"] = json.loads(str(d["config_json"]))
    return d


class _CpuHighway:
    """highway family on the C oracle (oracle/hwy_oracle.c), SameStep autoreset inside the C step."""

    def __init__(self, key: str, n: int, seed0: int):
        import numpy as np

        import hwy_oracle as ho
        from highwayenv_b200.config import default_config

        c = CONFIGS[key]
        cfg = default_config(c["env_id"])
        cfg.update(c["config"] or {})
        cfg["_others_check_collisions"] = 0 if c["env_id"] == "highway-fast-v0" else 1
        self.ob = ho.OracleBatch(ho.cfg_from_dict(cfg), n, seeds=range(seed0, seed0 + n), threads=1)
        self.ob.reset()
        self.rng = np.random.default_rng(1234 + seed0)
        self.n, self.box = n, c["actions"] == "box2"
        self.np = np

    def step(self):
        if self.box:
            a = self.rng.uniform(-1, 1, size=(self.n, 2)).astype(self.np.float32)
        else:
            a = self.rng.integers(0, 5, size=self.n).astype(self.np.int32)
        self.ob.step(a, autoreset=True)


class _CpuRoundabout:
    """roundabout-v0 on the C network oracle (oracle/net_oracle.c); resets through the numpy restatement of
    RoundaboutEnv._make_vehicles (highwayenv_b200.envs.roundabout_env.RoundaboutSpawner, host-only code)."""

    def __init__(self, key: str, n: int, seed0: int):
        import numpy as np

        import net_oracle as no
        from highwayenv_b200.config import default_config
        from highwayenv_b200.envs.common.action import DiscreteMetaAction
        from highwayenv_b200.envs.roundabout_env import RoundaboutSpawner, make_roundabout_network

        c = CONFIGS[key]
        cfg = default_config(c["env_id"])
        cfg.update(c["config"] or {})
        g = _golden("roundabout_ttc")
        self.ob = no.NetOracleBatch(no.graph_from_arrays(g), no.cfg_from_dict(cfg), n)
        self.sp = RoundaboutSpawner(make_roundabout_network(), cfg, DiscreteMetaAction(**cfg["action"]).target_speeds)
        self.gens = [np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed0 + i))) for i in range(n)]
        self.rng = np.random.default_rng(1234 + seed0)
        self.n, self.np = n, np
        self._respawn(np.arange(n))

    def _respawn(self, ids):
        a, sd = self.ob.a, self.sp.spawn([self.gens[i] for i in ids])
        for k in ("x", "y", "heading", "speed", "target_speed", "timer", "delta", "lane", "target_lane", "kind",
                  "route", "route_len", "speed_index"):
            a[k][ids] = sd[k]
        for k in ("crashed", "has_impact", "impact_x", "impact_y", "time"):
            a[k][ids] = 0
        a["check_collisions"][ids] = 1

    def step(self):
        act = self.rng.integers(0, 5, size=self.n).astype(self.np.int32)
        _, _, term, trunc = self.ob.step(act)
        done = self.np.nonzero(term | trunc)[0]
        if len(done):
            self._respawn(done)
            self.ob.observe()


class _CpuIntersection:
    """intersection-v0 on the C network oracle + the numpy restatement of the dynamic population
    (oracle/net_oracle.py IntersectionOracle: per-step clear / spawn, _make_vehicles with the 45 warm-up substeps)."""

    def __init__(self, key: str, n: int, seed0: int):
        import numpy as np

        import net_oracle as no
        from highwayenv_b200.config import default_config

        c = CONFIGS[key]
        cfg = default_config(c["env_id"])
        cfg.update(c["config"] or {})
        g = _golden("intersection_grid")
        self.ob = no.IntersectionOracle(no.graph_from_arrays(g), no.cfg_from_dict(cfg), n, g, cfg)
        for e in range(n):
            self.ob.reset_env(e, seed=seed0 + e)
        self.rng = np.random.default_rng(1234 + seed0)
        self.n, self.np = n, np

    def step(self):
        act = self.rng.integers(0, 3, size=self.n).astype(self.np.int32)
        _, _, term, trunc = self.ob.step(act)
        for e in self.np.nonzero(term | trunc)[0]:
            self.ob.reset_env(int(e))


_CPU_IMPL = {"cfg1": (_CpuHighway, 64), "cfg2": (_CpuHighway, 32), "cfg3": (_CpuIntersection, 4),
             "cfg4": (_CpuRoundabout, 8), "cfg5": (_CpuHighway, 8)}


def _cpu_worker(key, core, seed0, seconds, warmup, barrier, out):
    try:
        os.sched_setaffinity(0, {core})
    except Exception:
        pass
    cls, n = _CPU_IMPL[key]
    sim = cls(key, n, seed0)
    for _ in range(warmup):
        sim.step()
    barrier.wait()
    steps, t0 = 0, time.perf_counter()
    while True:
        sim.step()
        steps += 1
        dt = time.perf_counter() - t0
        if dt >= seconds:
            break
    out.put((n * steps, dt))


def cpu_arm_inprocess(key: str, seconds: float, repeats: int, warmup: int = 3) -> dict:
    """One pinned single-threaded oracle process per host core; every process times its own >= `seconds` of
    stepping after a common barrier; rate = sum of the per-process rates; median over `repeats`."""
    import multiprocessing as mp

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hwy_oracle  # noqa: F401  (builds / loads the C libraries once, before the fork)
    import net_oracle

    hwy_oracle.lib()
    net_oracle.lib()
    ctx = mp.get_context("fork")
    cores = host_cores()
    load0 = os.getloadavg()
    rates = []
    for rep in range(repeats):
        barrier, out = ctx.Barrier(len(cores)), ctx.Queue()
        n_per = _CPU_IMPL[key][1]
        procs = [ctx.Process(target=_cpu_worker, args=(key, c, 100000 * rep + i * n_per, seconds, warmup, barrier, out))
                 for i, c in enumerate(cores)]
        for p in procs:
            p.start()
        res = [out.get() for _ in procs]
        for p in procs:
            p.join()
        rates.append(sum(n / dt for n, dt in res))
    value = statistics.median(rates)
    return {
        "value": value, "unit": UNIT, "cores": len(cores), "kind": "port",
        "sample": (f"{len(cores)} pinned single-threaded processes x {_CPU_IMPL[key][1]} envs, >= {seconds:g} s timed each "
                   f"after {warmup} warm-up steps, median of {repeats} runs, {workload_name(key)}, C oracle port "
                   f"(oracle/*.c) with numpy resets, {cpu_model()}"),
        "runs": rates, "spread": (max(rates) - min(rates)) / value if value else None,
        "loadavg_before": list(load0), "loadavg_after": list(os.getloadavg()),
        "affinity_cores": len(cores), "per_core": value / len(cores),
    }


def cpu_arm(key: str, seconds: float, repeats: int) -> dict:
    """Run the CPU arm in a fresh interpreter (no CUDA context in the forking process)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-arm", key, "--cpu-seconds", str(seconds),
           "--cpu-repeats", str(repeats)]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    if out.returncode != 0:
        return {"error": out.stderr[-400:]}
    return json.loads(out.stdout.strip().splitlines()[-1])


def python_reference(key: str):
    """Per-core rate of the unmodified Python reference, measured in the build container by
    tools/time_reference.py (the reference cannot travel to the GPU box)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_python_reference.json")) as f:
            d = json.load(f)
        r = dict(d["configs"][key])
        r["measured"] = "elsewhere: " + d["host"]
        return r
    except (OSError, KeyError, ValueError):
        return None


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    seconds = max(3.0, min(20.0, 0.1 * args.steps))
    cb = cpu_arm(HEADLINE, seconds, 3)
    if "error" in cb:
        print(json.dumps({"impl": "reference", "unavailable": cb["error"][-200:]}), flush=True)
        return
    cb["python_reference"] = python_reference(HEADLINE)
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * _CPU_IMPL[HEADLINE][1] * cb["cores"] / value, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(HEADLINE), "envs": _CPU_IMPL[HEADLINE][1] * cb["cores"],
                   "autoreset": "SameStep"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm
def _ncu_summary(name: str):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


def _peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _make_actions(kind, shape_n, count, gen, dev, torch):
    if kind == "box2":
        return torch.rand((count, shape_n, 2), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    hi = 3 if kind == "discrete3" else 5
    return torch.randint(0, hi, (count, shape_n), generator=gen, device=dev, dtype=torch.int32)


def _host_arrays(x, name: str, out: dict) -> None:
    """The tensors of an env.step return value (nested in tuples / dicts) as float32 / float64 numpy arrays."""
    import numpy as np
    import torch

    if isinstance(x, (dict, tuple, list)):
        for k, v in (x.items() if isinstance(x, dict) else enumerate(x)):
            _host_arrays(v, f"{name}_{k}" if name else str(k), out)
    elif isinstance(x, torch.Tensor):
        a = x.detach().cpu().numpy()
        out[name] = a if a.dtype.kind == "f" and a.itemsize >= 4 else a.astype(np.float32 if a.dtype.kind == "b" else np.float64)


def dump_outputs(outputs: dict, path: str) -> None:
    """outputs: config -> {name: array [envs, ...]}.  Writes <path>/<config>_<name>.npy; if the whole exceeds
    DUMP_LIMIT_BYTES, every config keeps the same fraction of its envs, chosen by a fixed seed (written as
    <config>_env_index.npy)."""
    import numpy as np

    total = sum(a.nbytes for arrays in outputs.values() for a in arrays.values())
    frac = min(1.0, DUMP_LIMIT_BYTES / total) if total else 1.0
    os.makedirs(path, exist_ok=True)
    for key, arrays in outputs.items():
        n = len(next(iter(arrays.values())))
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(0).permutation(n)[:max(1, int(n * frac * 0.99))])
            arrays = {name: a[idx] for name, a in arrays.items()}
            arrays["env_index"] = idx.astype(np.float64)
        for name, a in arrays.items():
            np.save(os.path.join(path, f"{key}_{name}.npy"), a)


def measure_config(key, E, K, W, rank, world, dev, ctx, do_e2e=True, gather=False, dump=False):
    """Device-timed and end-to-end throughput of one config on this rank; returns local timings (and, with
    `dump`, the host copies of what the last timed step returned, under "outputs")."""
    import torch
    import torch.distributed as dist

    import highwayenv_b200 as hb

    c = CONFIGS[key]
    lib = ctx["lib"]
    env = hb.make(c["env_id"], num_envs=E, config=c["config"], device=dev, env_index_offset=rank * E)
    env.reset(seed=0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    actions = _make_actions(c["actions"], E, W + K, gen, dev, torch)
    stream = torch.cuda.current_stream(dev)
    flush = ctx["flush"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for t in range(W):
        env.step(actions[t])
    barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    env._kernel_events = []
    launches0 = lib.hwy_launch_count()
    sampler = None
    if rank == 0 and key == HEADLINE:
        try:
            uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
        except Exception:
            uuid = None
        sampler = ClockSampler(dev.index or 0, uuid)
    if sampler:
        sampler.start()
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(K):
        flush.fill_(k & 0xFF)  # > L2: the state is read from HBM in every timed step
        ev[k][0].record(stream)
        last = env.step(actions[W + k])
        ev[k][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    outputs = {}
    if dump:  # before the e2e and road-only passes below reuse the env's output buffers
        _host_arrays(dict(zip(("obs", "reward", "terminated", "truncated", "info"), last)), "", outputs)
    del last
    launches = int(lib.hwy_launch_count() - launches0)
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    kev, env._kernel_events = env._kernel_events, None
    kern_ms = sum(a.elapsed_time(b) for a, b in kev) / max(1, len(kev)) if kev else total_ms / K
    res = {"total_ms": total_ms, "kern_ms": kern_ms, "launches": launches, "wall_s": t_wall, "clocks": clocks,
           "obs_bytes": int(env._obs[0].numel() * 4), "act_bytes": int(actions[0].numel() * actions.element_size() // E)}
    if dump:
        res["outputs"] = outputs

    if gather and world > 1:
        from highwayenv_b200.parallel import all_gather_batch

        for _ in range(3):
            all_gather_batch(env._obs)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(20):
            out = all_gather_batch(env._obs)
        g1.record(stream)
        barrier()
        res["gather_ms"] = g0.elapsed_time(g1) / 20
        res["gather_bytes"] = int(out.numel() * 4)

    if do_e2e:
        Ke = K
        h_actions = torch.empty(tuple(actions[0].shape), dtype=actions.dtype).pin_memory()
        pool = actions[W:W + Ke].cpu()
        h_obs = torch.empty(tuple(env._obs.shape), dtype=torch.float32).pin_memory()
        h_rew = torch.empty(E, dtype=torch.float64).pin_memory()
        h_term = torch.empty(E, dtype=torch.bool).pin_memory()
        h_trunc = torch.empty(E, dtype=torch.bool).pin_memory()
        d_actions = torch.empty_like(actions[0])

        def eager_step(k):
            h_actions.copy_(pool[k])  # the policy's host-side output
            d_actions.copy_(h_actions, non_blocking=True)
            obs, rew, term, trunc, _ = env.step(d_actions)
            h_obs.copy_(obs, non_blocking=True)
            h_rew.copy_(rew, non_blocking=True)
            h_term.copy_(term, non_blocking=True)
            h_trunc.copy_(trunc, non_blocking=True)
            torch.cuda.synchronize(dev)  # the caller reads the results before acting again

        for k in range(min(3, Ke)):
            eager_step(k)
        barrier()
        t0 = time.perf_counter()
        for k in range(Ke):
            eager_step(k)
        barrier()
        res["e2e_eager_s"] = time.perf_counter() - t0
        res["e2e_s"], res["e2e_api"] = res["e2e_eager_s"], "env.step + explicit pinned copies"
        if hasattr(env, "host_stepper"):
            try:
                hs = env.host_stepper()
                pool_np = pool.numpy()
                for k in range(min(3, Ke)):
                    hs.actions[:] = pool_np[k]
                    hs.step()
                barrier()
                t0 = time.perf_counter()
                for k in range(Ke):
                    hs.actions[:] = pool_np[k]  # the policy's host-side output
                    hs.step()                   # returns after the results are in host memory
                barrier()
                s = time.perf_counter() - t0
                if s < res["e2e_s"]:
                    res["e2e_s"] = s
                    res["e2e_api"] = "env.host_stepper().step() (one CUDA graph: H2D + step kernels + D2H)"
            except Exception as exc:  # graph capture unavailable: keep the eager number, say why
                res["e2e_api"] += f" (host_stepper unavailable: {type(exc).__name__}: {exc})"[:200]
        res["h2d"] = int(h_actions.numel() * h_actions.element_size())
        res["d2h"] = int(h_obs.numel() * 4 + E * (8 + 1 + 1))
    # BASELINE.md's other timing: Road.act() + Road.step(dt) alone (no action mapping, observation, reward or reset),
    # `substeps` of them per launch = the simulation part of one env.step.  Last, on a freshly reset batch: without resets
    # the population drifts (crashed vehicles stay), so only a few launches are timed.
    if hasattr(env, "road_substeps"):
        env.reset(seed=0)
        n_road = 12
        for _ in range(2):
            env.road_substeps(c["substeps"])
        barrier()
        rv = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n_road)]
        for k in range(n_road):
            flush.fill_(k & 0xFF)
            rv[k][0].record(stream)
            env.road_substeps(c["substeps"])
            rv[k][1].record(stream)
        barrier()
        res["road_ms"] = sum(a.elapsed_time(b) for a, b in rv) / n_road
    del env
    return res


def run_gpu_arm(args) -> None:
    import torch
    import torch.distributed as dist

    from highwayenv_b200 import _native as N

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    K, W = args.steps, args.warmup
    ctx = {"lib": N.load(), "flush": torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)}  # > 126 MB L2
    peak, peak_src = _peak()
    keys = [k for k in CONFIGS if (not args.configs or k in args.configs.split(","))]
    if HEADLINE not in keys:
        keys.insert(0, HEADLINE)

    def envs_for(key):
        if args.envs_per_gpu and key == HEADLINE:
            return args.envs_per_gpu
        if key == HEADLINE and world >= 8:
            return 8192  # north_star: 65 536 envs on 8 GPUs
        return CONFIGS[key]["envs_per_gpu"]

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.cpu()]

    def reduce_sum(v):
        t = torch.tensor([v], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return int(t.item())

    entries, head, head_raw, outputs = [], None, None, {}
    for key in keys:
        E = envs_for(key)
        Kc = K if key == HEADLINE or not args.other_steps else args.other_steps
        r = measure_config(key, E, Kc, W, rank, world, dev, ctx, gather=args.gather_obs and key == HEADLINE,
                           dump=bool(args.dump_outputs) and rank == 0)
        if "outputs" in r:
            outputs[key] = r.pop("outputs")
        total_ms, e2e_s, e2e_eager, kern_ms = reduce_max([r["total_ms"], r["e2e_s"], r["e2e_eager_s"], r["kern_ms"]])
        launches = reduce_sum(r["launches"])
        n_total = E * world
        c = CONFIGS[key]
        achieved = c["algo_bytes"] * E / (kern_ms * 1e-3) / 1e9
        ncu = _ncu_summary(c["ncu"]) or {}
        traffic = (float(ncu["dram_bytes_read"]) + float(ncu["dram_bytes_write"])) if "dram_bytes_read" in ncu else None
        veh_sub = E * c["vehicles"] * c["substeps"]
        entry = {
            "id": key, "baseline_config": c["baseline"], "workload": workload_name(key),
            "envs_per_gpu": E, "envs_total": n_total, "steps": Kc,
            "value": n_total * Kc / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / Kc,
            "vehicle_substeps_per_s": veh_sub * world * Kc / (total_ms * 1e-3),
            "gpu_launches": launches,
            "e2e": {"value": n_total * Kc / e2e_s, "unit": UNIT, "h2d_bytes_per_step": r["h2d"],
                    "d2h_bytes_per_step": r["d2h"], "api": r["e2e_api"], "eager_value": n_total * Kc / e2e_eager},
            "roofline": {
                "bound": "hbm", "kernel": c["kernel"], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": c["algo_bytes"] * E, "kernel_ms": kern_ms,
                "issue_active_pct": ncu.get("issue_active_pct"), "fp64_pipe_pct": ncu.get("fp64_pipe_pct"),
                "warps_active_pct": ncu.get("warps_active_pct"),
                "thread_inst_per_vehicle_substep": ncu.get("thread_inst_per_vehicle_substep"),
                "registers_per_thread": ncu.get("registers_per_thread"),
                "ncu_source": ("profiles/" + c["ncu"]) if ncu else None,
                "note": "compute/latency bound (fp64 + libm, branchy), not HBM bound: see DESIGN.md roofline",
            },
        }
        if "road_ms" in r:
            (road_ms,) = reduce_max([r["road_ms"]])
            entry["road_only"] = {
                "what": (f"{c['substeps']} x (Road.act + Road.step) per launch through env.road_substeps "
                         f"({'hwy_highway_substeps' if c['env_id'].startswith('highway') else 'hwy_network_substeps'}), "
                         "fresh populations, no resets"),
                "ms_per_launch": road_ms, "value": n_total / (road_ms * 1e-3), "unit": "env-steps/s equivalent",
                "road_substeps_per_s": n_total * c["substeps"] / (road_ms * 1e-3)}
        if key == HEADLINE:
            head, head_raw = entry, r
        entries.append(entry)

    strong = None
    if world > 1 and not args.no_strong:
        Es = STRONG_TOTAL_ENVS // world
        r = measure_config(HEADLINE, Es, max(20, K // 2), W, rank, world, dev, ctx, do_e2e=False)
        (total_ms,) = reduce_max([r["total_ms"]])
        Ks = max(20, K // 2)
        strong = {"scaling": "strong", "envs_total": Es * world, "envs_per_gpu": Es,
                  "value": Es * world * Ks / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / Ks,
                  "note": "same total batch at every N; compare with the N=1 line run with --envs-per-gpu 32768"}
    gather = None
    if head_raw and "gather_ms" in head_raw:
        (gms,) = reduce_max([head_raw["gather_ms"]])
        gather = {"collective": "all_gather_into_tensor (NCCL) of the whole-batch observation", "ms": gms,
                  "bytes_out_per_rank": head_raw["gather_bytes"],
                  "algbw_GBps": head_raw["gather_bytes"] / (gms * 1e-3) / 1e9,
                  "step_ms_without": head["ms_per_step"]}

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(outputs, args.dump_outputs)
        if not args.no_cpu_baseline:
            for entry in entries:
                cb = cpu_arm(entry["id"], args.cpu_seconds, 3)
                cb["python_reference"] = python_reference(entry["id"])
                entry["cpu_baseline"] = cb
        E = head["envs_per_gpu"]
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"{workload_name(HEADLINE)}, {E} envs/GPU (device-side resets, reference RNG streams)",
                "envs_per_gpu": E, "envs_total": E * world, "vehicles_per_env": CONFIGS[HEADLINE]["vehicles"],
                "l2": "flushed (256 MiB write) between timed steps, outside the event pairs",
                "timing": "CUDA events per step on the launch stream, summed; max over ranks",
                "parallelism": f"env-range sharding x{world}, no collective",
                "envs_per_gpu_rule": "4096 (BASELINE configs[1]) for N < 8; 8192 at N = 8 = north_star's 65 536 envs",
            },
            "clocks": head_raw["clocks"],
            "e2e": dict(head["e2e"], note="per-step pinned host actions -> device, public API, obs / reward / "
                                          "terminated / truncated -> pinned host, sync every step"),
            "gpu_launches": head["gpu_launches"],
            "roofline": head["roofline"],
            "cpu_baseline": head.get("cpu_baseline"),
            "configs": entries,
            "strong_scaling": strong,
            "gather_obs": gather,
            "wall_s_timed_region": head_raw["wall_s"],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="timed steps of every config")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="override for the headline config")
    ap.add_argument("--other-steps", type=int, default=0, help="timed steps of the non-headline configs (default: --steps)")
    ap.add_argument("--configs", default="", help="comma list (cfg1..cfg5); default all")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--gather-obs", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=3.0)
    ap.add_argument("--cpu-repeats", type=int, default=3)
    ap.add_argument("--cpu-arm", default="", help="internal: run the CPU arm of one config and print its JSON")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step of every config returned as DIR/<config>_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.other_steps < 0:
        ap.error("--steps must be >= 1 and --other-steps >= 0")
    if args.cpu_arm:
        print(json.dumps(cpu_arm_inprocess(args.cpu_arm, args.cpu_seconds, args.cpu_repeats)), flush=True)
        return
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_gpu_arm(args)


if __name__ == "__main__":
    main()
