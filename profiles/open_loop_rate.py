#!/usr/bin/env python
"""Open-loop rollouts: the same precomputed action schedule run (a) as K chained gpd_step calls captured in one CUDA graph
(the best step path for a schedule fixed in advance) and (b) as one gpd_rollout launch, with traj off and on.

Per shape and K: microseconds per control step from CUDA events over >= 0.5 s of work after warm-up, drone-substeps/s, the
algorithmic bytes per env-step (from the shapes, below) with the bandwidth they imply, and which bound applies.  The card name
and power limit are read in the same run.  One JSON line per measurement (stdout, and --out if given).

Bytes per env-step (what the algorithm must move, not what the hardware moved):
  step    : observation row read + written (2 N W 4), the action row (N A 4), reward + 2 flags, and the persistent state read
            + written (13 Real per drone; DSLPID 9 Real more; step counter and episode return 4 B each per env)
  rollout : the action row, reward + 2 flags, (traj) the 12 kin floats per drone (20 Real for the Ctrl env); the state and
            the final observation once per rollout, amortised over K
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpd_b200  # noqa: E402,F401
from gpd_b200.params import load_drone_params  # noqa: E402
from gpd_b200.sim import BatchedSim  # noqa: E402
from gpd_b200.utils.enums import DroneModel  # noqa: E402

HBM_BPS = 7.7e12        # HGX B200 data sheet, per GPU (1000 W); a bound, not a measured rate

SHAPES = {
    "C2": dict(env_kind="hover", action_type="rpm", N=1, pyb=240, ctrl=30, phy=0, precision="f32"),
    "C5": dict(env_kind="hover", action_type="pid", N=1, pyb=240, ctrl=48, phy=0, precision="f32"),
    "C3": dict(env_kind="multihover", action_type="rpm", N=2, pyb=240, ctrl=30, phy=3, precision="f64"),
}
RUNS = [("C2", 65536, 8), ("C2", 65536, 32), ("C2", 65536, 128), ("C2", 1048576, 8), ("C2", 1048576, 32),
        ("C2", 1048576, 128), ("C5", 2097152, 32), ("C3", 32768, 32)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # the measurement still stands; say that the card could not be read
        q = f"{torch.cuda.get_device_name(0)}, power limit unreadable ({type(e).__name__})"
    return q


def make(sh, E):
    kw = dict(SHAPES[sh])
    dp = load_drone_params(DroneModel.CF2X)
    N = kw["N"]
    if kw["env_kind"] == "hover":
        tgt = np.array([[0.0, 0.0, 1.0]])
    else:
        init = np.stack([np.arange(N) * 4 * dp.L, np.arange(N) * 4 * dp.L,
                         np.full(N, dp.COLLISION_H / 2 - dp.COLLISION_Z_OFFSET + .1)], 1)
        tgt = init + np.array([[0, 0, 1 / (i + 1)] for i in range(N)])
    return BatchedSim(dp, E, N, kw["env_kind"], kw["action_type"], kw["pyb"], kw["ctrl"], kw["phy"], kw["precision"], 0,
                      auto_reset=True, target_pos=tgt)


def bytes_per_env_step(s, K, mode):
    rs = 8 if s.precision == "f64" else 4
    N, A, W = s.N, s.A, s.W
    pid = s.action_type in ("pid", "vel", "one_d_pid")
    state = N * (13 + (9 if pid else 0)) * rs + 8          # + step counter and episode return
    act, outs = N * A * 4, rs + 2
    if mode == "step":
        return 2 * N * W * 4 + act + outs + 2 * state
    traj = N * 12 * 4 if mode == "rollout_traj" else 0
    return act + outs + traj + (2 * state + N * W * 4) / K


def time_it(fn, K, min_s=0.5):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    reps = max(3, math.ceil(min_s / max(e0.elapsed_time(e1) * 1e-3, 1e-6)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return ms * 1e3 / (reps * K), ms * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated shape names")
    args = ap.parse_args()
    gpu = card()
    fout = open(args.out, "w") if args.out else None
    for sh, E, K in RUNS:
        if args.only and sh not in args.only.split(","):
            continue
        s = make(sh, E)
        g = torch.Generator(device="cuda").manual_seed(0)
        shape = (K, E, s.N, s.A)
        if s.action_type == "pid":
            acts = (torch.rand(shape, device="cuda", generator=g) - 0.5) * 0.2 + torch.tensor([0, 0, 1.0], device="cuda")
        else:
            acts = (torch.rand(shape, device="cuda", generator=g) - 0.5) * 0.2
        acts = acts.to(s.act_dtype).contiguous()
        # (a) K chained steps in one graph (K even: the ping-pong ends where it started, so replays chain)
        s.set_step_chaining(True)
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            for k in range(K):
                s.step(acts[k])
        torch.cuda.current_stream().wait_stream(st)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for k in range(K):
                s.step(acts[k])
        res = {}
        res["step_graph"] = time_it(graph.replay, K)
        del graph
        # (b) one gpd_rollout per K steps, caller-owned outputs
        out = s.alloc_rollout_outputs(K, traj=True)
        res["rollout"] = time_it(lambda: s.rollout(acts, out=out), K)
        res["rollout_traj"] = time_it(lambda: s.rollout(acts, traj=True, out=out), K)
        sub_per_step = E * s.N * s.S
        for mode, (us, secs) in res.items():
            b = bytes_per_env_step(s, K, "step" if mode == "step_graph" else mode)
            bw = b * E / (us * 1e-6)
            rec = dict(shape=sh, envs=E, K=K, mode=mode, us_per_ctrl_step=round(us, 3),
                       drone_substeps_per_s=float(f"{sub_per_step / (us * 1e-6):.4g}"), bytes_per_env_step=round(b, 1),
                       algorithmic_GBps=round(bw / 1e9, 1), hbm_share=round(bw / HBM_BPS, 3),
                       bound=("HBM bytes" if bw / HBM_BPS > 0.5 else
                              ("FP64 issue / latency" if s.precision == "f64" else "FP32 issue / latency")),
                       timed_s=round(secs, 3), gpu=gpu)
            if mode != "step_graph":
                rec["speedup_vs_step_graph"] = round(res["step_graph"][0] / us, 2)
            line = json.dumps(rec)
            print(line, flush=True)
            if fout:
                fout.write(line + "\n"); fout.flush()
        s.close()
        del acts, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
