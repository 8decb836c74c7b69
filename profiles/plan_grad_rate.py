#!/usr/bin/env python
"""Planning gradients (gpd_plan_grad): microseconds per call next to gpd_plan on the same shapes, and the torch-autograd
restatement of the same gradient (tests/plan_grad_ref.py) on the GPU at the largest of these shapes that fits in memory.

Per shape: median of 5 windows of >= n calls (CUDA events) after warm-up, sample-steps/s, the tape bytes, and the bytes
per sample-step the algorithm must move (not what the hardware moved): the action row read by the forward and again by the
backward (2 N A 4), the tape written and read back (2 x 13 N Real), the gradient row written (N A Real).  The card's name,
power limit and max SM clock are read in the same run.  One JSON line per measurement (stdout, and --out if given).
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from plan_rate import SHAPES, card, make, timed  # noqa: E402
import gpd_b200  # noqa: E402,F401
from gpd_b200.params import load_drone_params  # noqa: E402
from gpd_b200.utils.enums import DroneModel  # noqa: E402
from plan_grad_ref import LeanRef, start_state  # noqa: E402

RUNS = [("C2", 1024, 256, 32), ("C2", 64, 4096, 16), ("C3dyn", 1024, 32, 32)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--n", type=int, default=50)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    info = card()
    lines = []

    def emit(d):
        d["card"] = info
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))
    made = {}
    for sh, E, S, K in RUNS:
        src = make(sh, E)
        tgt = src._target
        src.reset()
        for _ in range(3):
            src.step(torch.as_tensor(rng.uniform(-0.1, 0.1, (E, src.N, src.A)), dtype=torch.float32, device="cuda"))
        acts = torch.as_tensor(rng.uniform(-0.1, 0.1, (K, E, S, src.N, src.A)), dtype=torch.float32,
                               device="cuda").contiguous()
        pout = src.alloc_plan_outputs(K, S)
        gout = src.alloc_plan_grad_outputs(K, S)
        us_plan = timed(lambda: src.plan(acts, gamma=0.99, out=pout), args.n)
        us_grad = timed(lambda: src.plan_grad(acts, gamma=0.99, out=gout), args.n)
        rs = 8 if src.precision == "f64" else 4
        ss = E * S * K
        emit(dict(shape=sh, E=E, S=S, K=K, precision=src.precision, us_per_plan=round(us_plan, 2),
                  us_per_plan_grad=round(us_grad, 2), grad_over_plan=round(us_grad / us_plan, 2),
                  sample_steps_per_s=ss / (us_grad * 1e-6), tape_bytes=src.plan_grad_tape_bytes(K, S),
                  bytes_per_sample_step=dict(actions=2 * src.N * src.A * 4, tape=2 * 13 * src.N * rs,
                                             grad=src.N * src.A * rs)))
        made[(sh, E, S, K)] = (src, tgt, acts)
        del pout, gout
        torch.cuda.empty_cache()
    # the torch-autograd restatement (FP64, one elementwise kernel per operation), largest shape first
    for (sh, E, S, K) in sorted(made, key=lambda r: -r[1] * r[2] * r[3] * SHAPES[r[0]]["N"]):
        src, tgt, acts = made[(sh, E, S, K)]
        kw = dict(SHAPES[sh], num_drones=src.N, pyb_freq=SHAPES[sh]["pyb"], ctrl_freq=SHAPES[sh]["ctrl"], episode_len_sec=8.0)
        ref = LeanRef(load_drone_params(DroneModel.CF2X), kw)
        st, rr, _, cnt = src.get_state()
        st0 = start_state(st.double().repeat_interleave(S, 0), rr.double().repeat_interleave(S, 0))
        c0 = cnt.repeat_interleave(S, 0)
        tg = torch.as_tensor(np.broadcast_to(tgt, (E * S, src.N, 3)).copy(), dtype=torch.float64, device="cuda")

        def autograd():
            a = acts.double().reshape(K, E * S, src.N, src.A).requires_grad_(True)
            G = ref.plan(st0, c0, a, tg, 0.99)[0]
            G.sum().backward()
            return a.grad
        try:
            autograd()
            torch.cuda.synchronize()
            t = []
            for _ in range(3):
                t0 = time.perf_counter()
                autograd()
                torch.cuda.synchronize()
                t.append(time.perf_counter() - t0)
        except torch.cuda.OutOfMemoryError:
            emit(dict(what="torch_autograd_restatement", shape=sh, E=E, S=S, K=K, fits=False))
            torch.cuda.empty_cache()
            continue
        emit(dict(what="torch_autograd_restatement", shape=sh, E=E, S=S, K=K, fits=True, precision="f64",
                  us_per_call=round(float(np.median(t)) * 1e6, 1),
                  peak_mem_gib=round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)))
        break
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
