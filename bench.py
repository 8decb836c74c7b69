#!/usr/bin/env python
"""bench.py — drone-substeps/sec of the fused DYN step kernel (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: the reference's own Python on the host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + what the last timed step returned, as DIR/*.npy

Workload (BASELINE.json configs[1]): HoverAviary single-drone PPO-rollout shape, 65,536 parallel envs per GPU,
Physics.DYN, ActionType.RPM, KIN observation (72 floats), FP32, 240 Hz sim / 30 Hz ctrl (8 substeps per step),
uniform random float32 actions, SB3-style auto-reset on.  One "step" = one env.step() of all 65,536 envs
= one launch of the fused kernel.  The 42 MB per-step working set fits the 126 MB L2, so the bench rotates
over `--sets` independent env sets (8 x ~46 MB > L2): every step touches data last used 8 steps ago.

value   = E*N*S*K / device time of EXACTLY K steps (CUDA events, max over ranks), inputs resident in HBM.  The K steps are
          ONE CUDA graph (K <= 1024; longer runs replay a 16-step graph), enqueued behind a short device-side sleep so that
          no host launch latency falls inside the event window; the window is measured `--trials` times (each bracketed by
          barrier + synchronize) and the median trial is reported, all trials listed.
e2e     = the same metric through HoverAviary.step(numpy): pinned host actions in, what the device computed (kin, reward,
          flags: 54 B per env) out into the host observation mirror (gpd_step_mirror); the step kernel moves both over PCIe
          itself (mapped pinned memory) instead of separate copy operations
roofline= algorithmic bytes (646 B per env-step, SURVEY §8d) * E / kernel time, against MEASURED_PEAKS.json hbm_gbs
other_configs = BASELINE.json configs[2..4] (C3 / C4 / C5), device-timed the same way, max over ranks
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_BYTES_PER_ENV_STEP = {30: 646, 48: 934}      # SURVEY §8d, FP32, HoverAviary RPM KIN
# FP64 mode: the 13-value state and the reward double; actions, ring and observation stay float32
ALGO_BYTES_PER_ENV_STEP_F64 = {30: 646 + 2 * 52 + 4, 48: 934 + 2 * 52 + 4}
METRIC = "drone-substeps/sec"
ISSUE_PEAK_FFMA_LANE_OPS = 3.571e13       # profiles/r01/microbench.jsonl (measured on this pool's B200): FP32 lane-ops/s
MUFU_PEAK_OPS = 4.637e12                  # same file: MUFU.EX2 ops/s


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20000)
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--ctrl-freq", type=int, default=30)
    ap.add_argument("--sets", type=int, default=8, help="independent env sets rotated to defeat L2 residency")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--tpb", type=int, default=0)
    ap.add_argument("--streams", type=int, default=1,
                    help="async env pools: env set j always steps on stream j %% STREAMS, so independent sets overlap (default 1 = "
                         "every step ordered on one stream, the headline mode)")
    ap.add_argument("--trials", type=int, default=0, help="timed windows of K steps (0 = 5 for short windows, 1 for long ones)")
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--launch", default="auto", choices=["auto", "direct", "single", "cycles"])
    ap.add_argument("--no-extra", action="store_true", help="skip the informational measurements and other_configs")
    ap.add_argument("--no-others", action="store_true", help="skip other_configs (BASELINE configs[2..4])")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "python", "port"],
                    help="reference arm: the staged reference Python (oracle/_ref) or the C oracle port")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, reward, terminated, truncated of the env set it stepped; "
                         "rank 0) as DIR/<name>.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def workload_name(a):
    return (f"HoverAviary DYN RPM KIN {a.precision} {a.envs} envs/GPU x 1 drone, 240/{a.ctrl_freq} Hz "
            f"(S={240 // a.ctrl_freq}), U(-1,1) float32 actions, auto-reset")


def config_dict(a, world, **extra):
    """Same keys on both arms (the driver compares the dicts)."""
    S = 240 // a.ctrl_freq
    c = {"workload": workload_name(a), "envs_per_gpu": a.envs, "substeps_per_step": S,
         "parallelism": f"env-sharded x{world}, no data-path collective",
         "l2": (f"GPU arm: {a.sets} independent env sets per GPU stepped in rotation (~{a.sets * a.envs * 700 / 1e6:.0f} MB touched per "
                "cycle > 126 MB L2), so every step's inputs were last touched a whole cycle ago; CPU arm: not applicable")}
    c.update(extra)
    return c


# ----------------------------------------------------------------------------------------------
# CPU arms.  (1) the reference's own, unmodified Python under the pybullet/gymnasium stand-ins (oracle/_ref staged by
# __graft_entry__.build() from the reference tree; kind = "reference"); (2) the C oracle port on pthreads (kind = "port").
def cpu_port_run(a, seconds=None, steps=None, warmup=2, budget_s=60.0):
    """The oracle port on all host cores.  With a fixed number of `steps` the per-step sample (number of envs, at most
    the bench's own) is sized from a calibration step so that the whole run stays within `budget_s`: the metric is
    per drone-substep, and the CPU cost is linear in the number of envs."""
    from gpd_b200.params import load_drone_params
    from gpd_b200.utils.enums import DroneModel
    from oracle import oracle as orc
    E = a.envs
    threads = orc.max_threads()
    sim = orc.OracleSim(load_drone_params(DroneModel.CF2X), E, ctrl_freq=a.ctrl_freq)
    rng = np.random.default_rng(0)
    pool = [rng.uniform(-1, 1, size=(E, 1, 4)).astype(np.float32) for _ in range(4)]
    S = 240 // a.ctrl_freq

    def one(k):
        _, _, te, tr = sim.step(pool[k % 4], nthreads=threads)
        done = (te | tr)
        if done.any():
            sim.reset(done)
        return sim
    for k in range(warmup):
        one(k)
    if steps is not None:
        # size the per-step sample from two calibration steps of the real loop; never below 8192 envs, where the
        # per-step thread fork/join would start to dominate and under-state the CPU
        t0 = time.perf_counter()
        one(0); one(1)
        per_step = (time.perf_counter() - t0) / 2
        if per_step * steps > budget_s and E > 8192:
            E = max(8192, int(E * budget_s / (per_step * steps)))
            sim = orc.OracleSim(load_drone_params(DroneModel.CF2X), E, ctrl_freq=a.ctrl_freq)
            pool = [p[:E].copy() for p in pool]
            for k in range(warmup):
                one(k)
    t0 = time.perf_counter()
    n = 0
    while True:
        one(n)
        n += 1
        el = time.perf_counter() - t0
        if steps is not None and n >= steps:
            break
        if steps is None and el >= seconds:
            break
    el = time.perf_counter() - t0
    return dict(value=E * S * n / el, steps=n, seconds=el, cores=threads, E=E, S=S)


def port_baseline(a, seconds=None, steps=None, warmup=2):
    r = cpu_port_run(a, seconds=seconds, steps=steps, warmup=warmup)
    return {"value": r["value"], "unit": "drone-substeps/s", "cores": r["cores"], "kind": "port",
            "sample": f"{r['steps']} env.step() of {r['E']} envs in {r['seconds']:.1f} s (FP64 C oracle port, pthreads, auto-reset)"}, r


def python_reference_baseline(a, steps, warmup, budget_s):
    from oracle import ref_python
    r = ref_python.run(steps=steps, warmup=warmup, ctrl_freq=a.ctrl_freq, budget_s=budget_s)
    n = r["workers"] * r["envs_per_worker"]
    return {"value": r["value"], "unit": "drone-substeps/s", "cores": r["workers"], "kind": "reference",
            "sample": (f"{r['steps']} vec-steps of {n} envs ({r['workers']} worker processes x {r['envs_per_worker']} reference "
                       f"HoverAviary(physics=DYN) instances, SubprocVecEnv-style, auto-reset; {r['resets']} resets) in {r['seconds']:.1f} s; "
                       "unmodified reference Python (oracle/_ref) under the pybullet/gymnasium stand-ins of oracle/refshim"),
            "per_core": r["per_core"]}, r


def have_python_reference(a):
    if a.ref_kind == "port":
        return False
    try:
        from oracle import ref_python
        ok = ref_python.available()
    except Exception:
        ok = False
    if a.ref_kind == "python" and not ok:
        raise SystemExit("bench.py: --ref-kind python but oracle/_ref is not staged (python oracle/stage_reference.py)")
    return ok


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = max(1, a.steps), max(1, a.warmup)
    world = int(os.environ.get("WORLD_SIZE", str(a.gpus)))
    extra = {}
    if have_python_reference(a):
        cpu, r = python_reference_baseline(a, steps=K, warmup=min(W, 3), budget_s=40.0)
        ms = 1e3 * r["seconds"] / r["steps"]
        if a.cpu_seconds > 0:      # the C restatement beside it, for scale (never the arm's value when the reference itself runs)
            extra["cpu_port"], _ = port_baseline(a, seconds=min(a.cpu_seconds, 5.0))
    else:
        cpu, r = port_baseline(a, steps=K, warmup=W)
        ms = 1e3 * r["seconds"] / r["steps"]
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "drone-substeps/s", "n_gpus": a.gpus,
        "steps": r["steps"], "warmup": a.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(a, world),
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "drone-substeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    line.update(extra)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi style clock/throttle sampling (NVML) while the GPU is busy."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:        # every sample between start() and stop() is taken while the GPU is under the bench's load
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append(mhz)
                for k, bit in names.items():
                    if rs & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=1)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_from_profile():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class Timer:
    """Device-side timing of a replayable unit: events around `fn()` enqueued behind a short GPU sleep, so that the launches
    are already queued when the first event fires (no host latency inside the window)."""

    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def window(self, fn, sleep_cycles=400_000, events=None):
        """`events`: a pair of external events that `fn`'s CUDA graph records itself, as its first and last node (the window
        then starts when the device starts the graph, not when the host asked for it)."""
        torch = self.torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()
        torch.cuda._sleep(sleep_cycles)
        if events is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
        else:
            e0, e1 = events
            fn()
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        return e0.elapsed_time(e1)

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms, [ms]
        t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        per = [float(x.item()) for x in out]
        return max(per), per


def graph_of(torch, fn):
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.synchronize()
    return g


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, outputs):
    """Writes `outputs` (name -> array with the env axis first) as DIR/<name>.npy in float64 (float64 arrays) or float32 (the
    rest).  Beyond DUMP_MAX_BYTES in all, every array keeps the same fixed, seeded sample of envs, listed in env_index.npy."""
    arrs = {k: np.ascontiguousarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in outputs.items()}
    E = len(next(iter(arrs.values())))
    per_env = sum(v.nbytes for v in arrs.values()) / E
    if per_env * E > DUMP_MAX_BYTES:
        n = int((DUMP_MAX_BYTES - 4096) // (per_env + 8))          # 4 KB for the .npy headers, 8 B per env for env_index
        idx = np.sort(np.random.default_rng(0).choice(E, n, replace=False))
        arrs = {k: v[idx] for k, v in arrs.items()}
        arrs["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def measure_config(torch, timer, make_env, make_action, nsets, steps, trials=3):
    """µs per step of one BASELINE shape: `nsets` rotating env sets, `steps` steps in one CUDA graph, best of `trials` windows,
    max over ranks."""
    envs = [make_env() for _ in range(nsets)]
    acts = [make_action(envs[0], k) for k in range(2 * nsets)]
    for e in envs:
        e.reset()
        e._sim.set_step_chaining(True)      # pre-generated actions (see b200_arm)
    period = 2 * nsets
    steps = max(period, (steps // period) * period)

    def run(n):
        for k in range(n):
            envs[k % nsets]._sim.step(acts[k % period])
    run(period)
    torch.cuda.synchronize()
    g = graph_of(torch, lambda: run(steps))
    g.replay()
    torch.cuda.synchronize()
    best = min(timer.window(g.replay) for _ in range(trials))
    ms, per = timer.max_over_ranks(best)
    sim = envs[0]._sim
    info = dict(E=sim.E, N=sim.N, S=sim.S, us_per_step=1e3 * ms / steps, steps=steps,
                us_per_step_ranks=[1e3 * p / steps for p in per] if len(per) > 1 else None)
    for e in envs:
        e.close()
    del envs, acts, g
    torch.cuda.empty_cache()
    return info


def other_configs(torch, timer, world, rank, local, peak):
    """BASELINE.json configs[2..4] in the driver-run line (VERDICT r1 item 4).  C3/C5 weak (per-GPU sizes fixed), C4 strong."""
    from gpd_b200.distributed import shard_range
    from gpd_b200.envs import CtrlAviary, HoverAviary, MultiHoverAviary
    from gpd_b200.utils.enums import ActionType, DroneModel, Physics

    def rand(shape, seed, dtype=torch.float32):
        g = torch.Generator(device="cuda")
        g.manual_seed(seed + 1000 * rank)
        return (torch.rand(shape, generator=g, device="cuda") * 2 - 1).to(dtype)
    out = {}
    try:    # C3: MultiHoverAviary x2, DYN+GND+DRAG, FP64 parity mode, 32,768 envs per GPU
        E = 32768
        r = measure_config(torch, timer, lambda: MultiHoverAviary(num_envs=E, num_drones=2, physics=Physics.DYN_GND_DRAG, ctrl_freq=30,
                                                                   precision="f64", auto_reset=True, device=local),
                           lambda env, k: rand((E, 2, 4), k), nsets=6, steps=48)
        algo = 2 * 1292     # SURVEY §8d: 1,292 B per drone-ctrl-step in FP64
        gbs = algo * E / (r["us_per_step"] * 1e-6) / 1e9
        r.update(workload="C3 MultiHoverAviary 32,768 envs/GPU x 2 drones DYN+GND+DRAG f64 240/30", scaling="weak",
                 drone_substeps_per_s=world * E * 2 * r["S"] / (r["us_per_step"] * 1e-6),
                 roofline={"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                           "algorithmic_bytes_per_env_step": algo})
        out["c3_multihover2_gnd_drag_f64"] = r
    except Exception as ex:
        out["c3_multihover2_gnd_drag_f64"] = {"error": repr(ex)[:300]}
        torch.cuda.synchronize()
    try:    # C4: 4,096 envs x 64 drones in total (strong scaling: split over the ranks), DYN + O(N^2) downwash, FP32
        Etot, N = 4096, 64
        lo, El = shard_range(Etot, rank, world)
        rng = np.random.default_rng(1)
        xyz = np.concatenate([rng.uniform(-2, 2, size=(Etot, N, 2)), rng.uniform(0.2, 3, size=(Etot, N, 1))], axis=-1)[lo:lo + El]
        r = measure_config(torch, timer, lambda: CtrlAviary(num_envs=El, num_drones=N, physics=Physics.DYN_DW, pyb_freq=240, ctrl_freq=48,
                                                             initial_xyzs=xyz, precision="f32", device=local),
                           lambda env, k: (env.HOVER_RPM * (1 + 0.02 * rand((El, N, 4), k))).float(), nsets=4, steps=16)
        pairs = Etot * N * N * r["S"] / (r["us_per_step"] * 1e-6)      # job-wide pair evaluations per second
        instr_per_pair, mufu_per_pair = 22, 2                             # SASS count of downwash_pair, FP32 (DESIGN §3.6)
        fi = pairs * instr_per_pair / (world * ISSUE_PEAK_FFMA_LANE_OPS)
        r.update(workload="C4 CtrlAviary 4,096 envs x 64 drones in total DYN+DW f32 240/48 (O(N^2) downwash)", scaling="strong",
                 envs_this_rank=El, drone_substeps_per_s=Etot * N * r["S"] / (r["us_per_step"] * 1e-6), pair_evals_per_s=pairs,
                 roofline={"bound": "issue", "achieved": pairs * instr_per_pair / world, "peak": ISSUE_PEAK_FFMA_LANE_OPS,
                           "unit": "FP32 lane-instr/s per GPU", "frac": fi,
                           "mufu_frac": pairs * mufu_per_pair / (world * MUFU_PEAK_OPS),
                           "peak_source": "profiles/r01/microbench.jsonl (FFMA issue, MUFU.EX2)"})
        out["c4_ctrl64_dw_f32"] = r
    except Exception as ex:
        out["c4_ctrl64_dw_f32"] = {"error": repr(ex)[:300]}
        torch.cuda.synchronize()
    try:    # C5: 2,097,152 envs per GPU, FP32, DSLPIDControl in the loop (ActionType.PID), 240/48
        E = 2097152
        r = measure_config(torch, timer, lambda: HoverAviary(num_envs=E, drone_model=DroneModel.CF2P, ctrl_freq=48, act=ActionType.PID,
                                                              precision="f32", auto_reset=True, device=local),
                           lambda env, k: rand((E, 1, 3), k), nsets=1, steps=6)
        algo = 814
        gbs = algo * E / (r["us_per_step"] * 1e-6) / 1e9
        r.update(workload="C5 HoverAviary 2,097,152 envs/GPU ActionType.PID (DSLPIDControl in-loop) f32 240/48", scaling="weak",
                 drone_substeps_per_s=world * E * r["S"] / (r["us_per_step"] * 1e-6),
                 roofline={"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                           "algorithmic_bytes_per_env_step": algo})
        out["c5_hover_pid_48hz_f32"] = r
    except Exception as ex:
        out["c5_hover_pid_48hz_f32"] = {"error": repr(ex)[:300]}
        torch.cuda.synchronize()
    return out


def b200_arm(a):
    import torch
    import torch.distributed as dist

    import gpd_b200  # noqa: F401
    from gpd_b200.distributed import NcclStatsComm
    from gpd_b200.envs import HoverAviary
    from gpd_b200.utils.enums import ActionType, ObservationType, Physics

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    timer = Timer(torch, dist, world, dev)
    sampler = ClockSampler(local)
    sampler.start()                 # well before the timed windows: it samples the pre-warm, the windows and the e2e loop
    E, S, nsets = a.envs, 240 // a.ctrl_freq, a.sets

    envs = [HoverAviary(physics=Physics.DYN, ctrl_freq=a.ctrl_freq, obs=ObservationType.KIN, act=ActionType.RPM,
                        num_envs=E, device=local, precision=a.precision, auto_reset=True, threads_per_block=a.tpb)
            for _ in range(nsets)]
    g = torch.Generator(device=dev)
    g.manual_seed(rank)
    acts = [(torch.rand((E, 1, 4), generator=g, device=dev) * 2 - 1) for _ in range(2 * nsets)]
    for e in envs:
        e.reset()
        # the K timed steps are launched back to back from action buffers generated long before: chained stepping is valid
        # (gpd_set_step_chaining): consecutive launches overlap across the kernel boundary, each tile ordered behind its own
        # previous step.  A policy-in-the-loop rollout (rollout.py) does not chain.
        e._sim.set_step_chaining(True)
    period = 2 * nsets

    nstreams = max(1, min(a.streams, nsets))
    pool = [torch.cuda.Stream(device=dev) for _ in range(nstreams - 1)]

    def run_steps(n, nstreams=nstreams, pool=pool, k0=0):
        """Steps k0 .. k0+n-1; returns what the last step returned (views of the buffers it writes, also under capture)."""
        out = None
        if nstreams == 1:
            for k in range(k0, k0 + n):
                out = envs[k % nsets]._sim.step(acts[k % period])
            return out
        # fork: every pool stream waits for the caller's stream; set j always runs on stream j % nstreams (its own steps stay
        # ordered); join: the caller's stream waits for every pool stream.  All of it is capturable.
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        for st in pool:
            st.wait_event(fork)
        for k in range(k0, k0 + n):
            j = (k % nsets) % nstreams
            with torch.cuda.stream(main if j == 0 else pool[j - 1]):
                out = envs[k % nsets]._sim.step(acts[k % period])
        for st in pool:
            ev = torch.cuda.Event()
            ev.record(st)
            main.wait_event(ev)
        return out

    # warm-up (also touches every buffer); whole cycles so that the observation ping-pong phase is back where it started
    wu = max(3, a.warmup)
    for _ in range((wu + period - 1) // period):
        run_steps(period)
    torch.cuda.synchronize()
    K = max(1, a.steps)
    # EXACTLY K steps per timed window.  Three launch modes (--launch auto picks by K):
    #   single  K <= 1024 (default): ONE graph = [event record, K step kernels, event record].  The two CUDA events are nodes of
    #           the graph, so the window is the device time of exactly the K steps — the ~8 us the device needs to start a
    #           graph (measured, profiles/r02) is launch latency, not step time, and stays outside.  The observation ping-pong
    #           and the set rotation repeat every `period` steps, so m = period / gcd(K, period) such graphs are captured back
    #           to back and replayed round-robin: every replay continues the simulation exactly where the previous one stopped
    #   direct  K plain stream launches enqueued while the device sleeps (Timer.window), events recorded on the stream
    #   cycles  longer runs: `reps` replays of a 128-step graph + a tail graph inside the window and, outside it, the complement
    #           that completes the tail's cycle
    from math import gcd
    mode = a.launch
    if mode == "auto":
        mode = "single" if K <= 1024 else "cycles"
    if a.no_graph:
        mode = "direct"
    gper = period * 8
    m = period // gcd(K, period)
    reps, tail = divmod(K, gper) if mode == "cycles" else (0, 0)
    graphs = None
    graph_error = None
    last = {}           # timed unit -> what its last step returned

    def unit_steps(key, n, k0=0):
        last[key] = run_steps(n, k0=k0)
    if mode != "direct":
        try:
            if mode == "single":
                # the two timing events are the first and the last node of each graph (external events: real record nodes)
                gev = [(torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
                       for _ in range(m)]

                def unit(i):
                    gev[i][0].record()
                    unit_steps(i, K, k0=i * K)
                    gev[i][1].record()
                graphs = [graph_of(torch, (lambda i=i: unit(i))) for i in range(m)]
            else:
                graphs = {"main": graph_of(torch, lambda: unit_steps("main", gper)),
                          "tail": graph_of(torch, lambda: unit_steps("tail", tail)) if tail else None,
                          "comp": graph_of(torch, lambda: run_steps(gper - tail, k0=tail)) if tail else None}
        except Exception as ex:          # never lose the measurement to a capture problem: fall back to direct launches
            graphs = None
            mode = "direct"
            graph_error = repr(ex)[:200]
            torch.cuda.synchronize()
    nxt = [0]           # which of the m units (graphs, or K-step groups of direct launches) comes next

    def timed_unit():
        if mode == "direct":
            unit_steps("direct", K, k0=nxt[0] * K)
            nxt[0] = (nxt[0] + 1) % m
        elif mode == "single":
            graphs[nxt[0]].replay()
            nxt[0] = (nxt[0] + 1) % m
        else:
            for _ in range(reps):
                graphs["main"].replay()
            if tail:
                graphs["tail"].replay()

    def after_unit():       # untimed: bring the rotation back to a cycle boundary
        if mode == "cycles" and tail:
            graphs["comp"].replay()

    def finish_cycle():
        while nxt[0] != 0:
            timed_unit()

    def last_key():     # the unit whose last step was the last timed step
        if mode == "single":
            return (nxt[0] - 1) % m
        return "direct" if mode == "direct" else ("tail" if tail else "main")

    # bring the clocks to their loaded state (untimed): the same work for ~0.3 s on a B200 (34,880 steps at 65,536 envs,
    # launch-bound below).  Counted in steps, not timed, so that every run steps the env sets through the same sequence
    # and the outputs of the timed steps do not depend on the speed of the build.  Auto-resets come in bursts, so where
    # the timed windows fall in an episode moves the figure by ~1 %: the count is what 0.3 s of timed pre-warm reached
    # on a B200 (1000 W limit) with 20-step windows, 1,744 of them (profiles/bench_prewarm.txt).  A faster build
    # pre-warms for proportionally less time.
    pre_steps = 34_880 * 65_536 // max(E, 65_536)
    for n_pre in range(1, max(2, -(-pre_steps // K)) + 1):
        timed_unit()
        after_unit()
        if n_pre % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    est_ms = K * 0.012
    trials = a.trials or (5 if est_ms < 50 else 1)
    windows, per_rank_all = [], []
    # long enough for the host to enqueue the whole window behind it (direct mode: ~10 us of host time per launch)
    sleep_cycles = 400_000 + (40_000 * K if mode == "direct" else 60 * min(K, 4096))
    dumped = None
    for i in range(trials):
        ms_local = timer.window(timed_unit, sleep_cycles, events=gev[nxt[0]] if mode == "single" else None)
        if a.dump_outputs and rank == 0 and i == trials - 1:     # before any later step overwrites the buffers
            dumped = dict(zip(("obs", "reward", "terminated", "truncated"), (t.cpu().numpy() for t in last[last_key()])))
        after_unit()
        ms_max, per = timer.max_over_ranks(ms_local)
        windows.append(ms_max)
        per_rank_all.append(per)
    finish_cycle()
    torch.cuda.synchronize()
    order = sorted(range(trials), key=lambda i: windows[i])
    pick = order[len(order) // 2]                       # median window
    ms = windows[pick]
    per_rank = per_rank_all[pick]
    value = world * E * 1 * S * K / (ms * 1e-3)

    # ---- informational: the same job with the env sets as async pools on their own streams (never the headline) ----
    async_info = l2_info = None
    if nstreams == 1 and not a.no_graph and nsets >= 2 and not a.no_extra:
        try:
            ns2 = min(8, nsets)
            pool2 = [torch.cuda.Stream(device=dev) for _ in range(ns2 - 1)]
            g2 = graph_of(torch, lambda: run_steps(period, ns2, pool2))
            reps2 = 64
            for _ in range(8):
                g2.replay()
            ms2 = min(timer.window(lambda: [g2.replay() for _ in range(reps2)]) for _ in range(3)) / (reps2 * period)
            async_info = {"streams": ns2, "ms_per_step": ms2, "steps": reps2 * period,
                          "value_this_rank": E * S / (ms2 * 1e-3),
                          "note": "env set j steps on stream j % streams (its own steps stay ordered, independent sets overlap): "
                                  "what a trainer with several env pools gets (pool.py); informational, not the headline"}
        except Exception as ex:
            async_info = {"error": repr(ex)[:200]}
            torch.cuda.synchronize()
        try:    # one env set alone (46 MB working set: L2-resident; SURVEY 8d asks for flushed AND unflushed)
            def one_set():
                for k in range(period):
                    envs[0]._sim.step(acts[k % 2])
            g3 = graph_of(torch, one_set)
            reps3 = 64
            for _ in range(8):
                g3.replay()
            ms3 = min(timer.window(lambda: [g3.replay() for _ in range(reps3)]) for _ in range(3)) / (reps3 * period)
            l2_info = {"ms_per_step": ms3, "steps": reps3 * period,
                       "note": "ONE env set stepped back to back (working set < 126 MB L2, no rotation; consecutive steps depend on "
                               "each other tile by tile): what a single-set rollout sees; not an HBM number, informational"}
        except Exception as ex:
            l2_info = {"error": repr(ex)[:200]}
            torch.cuda.synchronize()

    # ---- episode statistics: the only collective — ONE NCCL all-gather inside gpd_episode_stats, off the step path ----
    stats = np.zeros(8)
    comm = None
    stats_how = "gpd_episode_stats (single rank)"
    try:
        if world > 1:
            comm = NcclStatsComm(device=local)
            stats_how = "gpd_episode_stats(..., ncclComm_t): one ncclAllGather of 8 doubles + device combine, in the library"
        for e in envs:
            s = e._sim.episode_stats(nccl_comm=comm.handle if comm else None)
            stats[[0, 1, 2, 3, 6, 7]] += s[[0, 1, 2, 3, 6, 7]]
    except Exception as ex:
        stats_how = "failed: " + repr(ex)[:200]
    finally:
        if comm is not None:
            comm.close()

    # ---- end to end through the public API with host buffers (rank-local; aggregate = sum over ranks) ----
    env = envs[0]
    pinned_act = [torch.empty((E, 1, 4), dtype=torch.float32).pin_memory() for _ in range(4)]
    rng = np.random.default_rng(rank)
    for p in pinned_act:
        p.copy_(torch.from_numpy(rng.uniform(-1, 1, size=(E, 1, 4)).astype(np.float32)))
    np_act = [p.numpy() for p in pinned_act]
    for k in range(5):
        env.step(np_act[k % 4])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    chk = 0.0
    for k in range(a.e2e_steps):
        obs, rew, term, trunc, _ = env.step(np_act[k % 4])
        chk += float(rew[0]) + float(obs[0, 0, 2])          # the step's result is read on the host every step
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_s, e2e_ranks = timer.max_over_ranks(e2e_s)
    e2e_val = world * E * S * a.e2e_steps / e2e_s
    # host obs == device obs (the mirror is not a different observation)
    mirror_ok = bool(np.array_equal(np.ascontiguousarray(obs), env._sim.obs.cpu().numpy()))
    h2d = E * 4 * 4
    d2h = E * (12 * 4 + 4 + 1 + 1)     # kin + reward + terminated + truncated: everything the device computed, nothing echoed
    slide = env._sim._mirror.rows - env._sim.W
    d2h_amortised = d2h + E * env._sim.W * 4 / (slide / env._sim.A)     # + the window rebuild every `slide/A` steps

    # ---- informational: the same numpy batch through a 2-pool VecEnv (one pool's H2D overlaps the other's D2H) ----
    pools_info = None
    if not a.no_extra:
        try:
            from gpd_b200.vec_env import GpdVecEnv
            venv = GpdVecEnv(HoverAviary, E, num_pools=2, physics=Physics.DYN, ctrl_freq=a.ctrl_freq, device=local,
                             precision=a.precision)
            venv.reset()
            for k in range(5):
                venv.step(np_act[k % 4])
            t0 = time.perf_counter()
            for k in range(100):
                o, r_, d_, _i = venv.step(np_act[k % 4])
            dt = time.perf_counter() - t0
            pools_info = {"pools": 2, "ms_per_step": 1e3 * dt / 100, "value_this_rank": E * S * 100 / dt,
                          "api": "GpdVecEnv(num_pools=2).step(numpy): SB3 VecEnv protocol incl. terminal_kin transfer and episode bookkeeping",
                          "note": "informational"}
            venv.close()
        except Exception as ex:
            pools_info = {"error": repr(ex)[:200]}
            torch.cuda.synchronize()

    peak, peak_src = peaks()
    others = None
    if not a.no_extra and not a.no_others:
        for e in envs:
            e.close()
        envs = []
        torch.cuda.empty_cache()
        others = other_configs(torch, timer, world, rank, local, peak)
    clocks = sampler.stop()

    if rank == 0:
        per_launch_ms = ms / K
        algo = (ALGO_BYTES_PER_ENV_STEP_F64 if a.precision == "f64" else ALGO_BYTES_PER_ENV_STEP).get(a.ctrl_freq, None)
        achieved = (algo * E / (per_launch_ms * 1e-3) / 1e9) if algo else None
        tr = traffic_from_profile()
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None,
                "traffic": (tr or {}).get("dram_bytes_per_launch"), "traffic_note": (tr or {}).get("note"),
                "traffic_steady_state": ((tr or {}).get("steady_state_bytes_per_env_step") or 0) * E or None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo * E if algo else None, "kernel": "gpd::step_kernel_bulk<%s,LEAN,N=1>" % ("double" if a.precision == "f64" else "float"),
                "kernel_ms_per_launch": per_launch_ms,
                "note": "consecutive launches overlap across the kernel boundary (chained stepping: programmatic dependent launch + "
                        "per-tile acquire/release sequencing, two tiles per CTA): kernel_ms_per_launch is the time per launch on ONE "
                        "stream over the timed window, not one launch's span"}
        if nstreams > 1:
            roof["note"] = (f"{nstreams} streams: launches of independent env sets overlap, so kernel_ms_per_launch is the "
                            "throughput-equivalent time per launch, not one launch's duration")
        if async_info and "ms_per_step" in async_info and algo:
            async_info["frac_of_hbm_peak"] = algo * E / (async_info["ms_per_step"] * 1e-3) / 1e9 / peak
        cpu = cpu_port = None
        if not a.no_cpu and world == 1:
            try:
                if have_python_reference(a):
                    cpu, _ = python_reference_baseline(a, steps=12, warmup=2, budget_s=max(5.0, a.cpu_seconds))
                    cpu_port, _ = port_baseline(a, seconds=min(a.cpu_seconds, 5.0))
                else:
                    cpu, _ = port_baseline(a, seconds=a.cpu_seconds)
            except Exception as ex:
                cpu = {"error": repr(ex)[:300]}
        if mode == "direct":
            launch = (f"{K} direct stream launches per timed window, enqueued behind a device-side sleep"
                      + (f" (graph capture failed: {graph_error})" if graph_error else ""))
        elif mode == "single":
            launch = (f"ONE CUDA graph per timed window: [event record, {K} step kernels, event record] "
                      f"({m} such graphs replayed round-robin)")
        else:
            launch = "CUDA graph of %d step kernels x %d replays + %d-step tail graph" % (gper, reps, tail)
        line = {
            "metric": METRIC, "value": value, "unit": "drone-substeps/s", "n_gpus": world, "steps": K, "warmup": wu,
            "ms_per_step": per_launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": a.precision, "data": "synthetic",
            "config": config_dict(a, world),        # the same dict on both arms (the driver compares them)
            "measurement": {
                "launch": launch, "streams": nstreams,
                "timing": f"median of {trials} windows of exactly {K} steps, each behind a device-side sleep and "
                          "bracketed by barrier + synchronize; CUDA events"
                          + (" recorded by the graph itself (first and last node)" if mode == "single" else "")
                          + "; max over ranks"},
            "trials_ms": windows,
            "rank_ms": {"min": min(per_rank), "median": float(np.median(per_rank)), "max": max(per_rank), "per_rank": per_rank},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "drone-substeps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "d2h_bytes_per_step_incl_window_rebuild": d2h_amortised,
                    "steps": a.e2e_steps, "ms_per_step": 1e3 * e2e_s / a.e2e_steps, "rank_s": e2e_ranks,
                    "host_obs_equals_device_obs": mirror_ok,
                    "api": "HoverAviary.step(numpy) -> gpd_step_mirror: the step kernel reads the actions from pinned host memory and "
                           "writes kin/reward/flags into the pinned feature-major host observation log over PCIe itself (zero-copy: "
                           "h2d/d2h bytes are what crosses the bus every step; the action ring is the host's own data and is never "
                           "echoed); obs is a strided (E,1,72) view of that log"},
            "gpu_launches": K,
            "roofline": roof,
            "async_pools": async_info,
            "l2_resident": l2_info,
            "e2e_pools": pools_info,
            "other_configs": others,
            "cpu_baseline": cpu,
            "cpu_port": cpu_port,
            "episode_stats": {"episodes": stats[0], "mean_return": stats[1] / max(stats[0], 1),
                              "mean_length": stats[2] / max(stats[0], 1), "env_steps": stats[6], "how": stats_how},
        }
        if dumped is not None:
            dump_outputs(a.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    for e in envs:
        e.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True      # the project's modules are imported below: the bench writes nothing into the tree
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    else:
        b200_arm(a)


if __name__ == "__main__":
    main()
