#!/usr/bin/env python
"""Planning rollouts (gpd_plan): S candidate schedules of K control steps per env, scored from the env's current state.

Per shape: microseconds per plan from CUDA events (median of 5 windows of >= 50 plans after warm-up), sample-steps/s and
drone-substeps/s, against
  (a) the workaround without gpd_plan: get_state -> repeat_interleave -> set_state on an E*S handle -> gpd_rollout -> masked
      sum of the (K, E*S) rewards; timed with its synchronisation (BatchedSim.set_state synchronises the stream);
  (b) gpd_rollout alone on a pre-filled E*S handle: the kernel-only lower bound of (a).
Also the MPPI control step of examples/mppi.py end to end, eager and graphed.  The card name, power limit and max SM clock
are read in the same run.  One JSON line per measurement (stdout, and --out if given).

Bytes per sample-step (what the algorithm must move, not what the hardware moved): the action row (N A 4; 16 B per drone
for 4-wide actions), the reward when asked for (Real), and the copy's state once per plan amortised over K (read only: 13
Real per drone, DSLPID 9 more, the counter 4 B; returns + done_step written once).
"""
import argparse
import json
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
    "C3dyn": dict(env_kind="multihover", action_type="rpm", N=2, pyb=240, ctrl=30, phy=0, precision="f64"),   # plan_grad_rate.py
}
RUNS = [("C2", 1024, 256, 32), ("C2", 64, 4096, 16), ("C5", 1024, 256, 16), ("C3", 1024, 32, 32)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:
        return f"{torch.cuda.get_device_name(0)}, power limit unreadable ({type(e).__name__})"


def make(sh, E, auto_reset=True):
    kw = SHAPES[sh]
    dp = load_drone_params(DroneModel.CF2X)
    N = kw["N"]
    if kw["env_kind"] == "hover":
        tgt = np.array([[0.0, 0.0, 1.0]])
    else:
        init = np.stack([np.arange(N) * 4 * dp.L, np.arange(N) * 4 * dp.L,
                         np.full(N, dp.COLLISION_H / 2 - dp.COLLISION_Z_OFFSET + .1)], 1)
        tgt = init + np.array([[0, 0, 1 / (i + 1)] for i in range(N)])
    return BatchedSim(dp, E, N, kw["env_kind"], kw["action_type"], kw["pyb"], kw["ctrl"], kw["phy"], kw["precision"], 0,
                      auto_reset=auto_reset, target_pos=tgt)


def actions(s, K, S, rng):
    a = rng.uniform(-0.3, 0.3, (K, s.E, S, s.N, s.A))
    if s.action_type == "pid":
        a = a + np.array([0, 0, 0.5])
    return torch.as_tensor(a, dtype=torch.float32, device="cuda").contiguous()


def timed(fn, n, windows=5):
    """Median microseconds per call over `windows` windows of n calls (CUDA events; fn may synchronise itself)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        res.append(a.elapsed_time(b) * 1e3 / n)
    return float(np.median(res))


def bytes_per_sample_step(s, K):
    rs = 8 if s.precision == "f64" else 4
    pid = s.action_type in ("pid", "vel", "one_d_pid")
    state = s.N * (13 + (9 if pid else 0)) * rs + 4 + rs + 4
    return s.N * s.A * 4, rs, state / K


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
    for sh, E, S, K in RUNS:
        src = make(sh, E)
        src.reset()
        for _ in range(3):
            src.step(actions(src, 1, 1, rng)[0, :, 0])
        acts = actions(src, K, S, rng)
        out = src.alloc_plan_outputs(K, S)
        us_plan = timed(lambda: src.plan(acts, gamma=0.99, out=out), args.n)
        # (a) and (b): an E*S handle
        rep = make(sh, E * S, auto_reset=False)
        ra = acts.reshape(K, E * S, src.N, src.A)
        rout = rep.alloc_rollout_outputs(K)
        g = torch.tensor(0.99, dtype=rep.real, device="cuda")
        disc = g ** torch.arange(K, device="cuda", dtype=rep.real)

        def workaround():
            st, rr, ps, cnt = src.get_state()
            rep.set_state(st.repeat_interleave(S, 0), rr.repeat_interleave(S, 0), ps.repeat_interleave(S, 0),
                          cnt.repeat_interleave(S, 0))
            _, rew, te, tr = rep.rollout(ra, out=rout)
            done = (te | tr).bool()
            alive = torch.cumprod(torch.cat([torch.ones_like(done[:1]), ~done[:-1]]).to(rew.dtype), 0)
            return (rew * disc[:, None] * alive).sum(0)
        us_a = timed(workaround, max(5, args.n // 5))
        # a handle with auto-reset, so that repeated rollouts keep the copies in their episodes (a drone that flew off would
        # put FP64 libm calls on their slow paths)
        rep_b = make(sh, E * S)
        st, rr, ps, cnt = src.get_state()
        rep_b.set_state(st.repeat_interleave(S, 0), rr.repeat_interleave(S, 0), ps.repeat_interleave(S, 0),
                        cnt.repeat_interleave(S, 0))
        us_b = timed(lambda: rep_b.rollout(ra, out=rout), args.n)
        act_b, rew_b, st_b = bytes_per_sample_step(src, K)
        ss = E * S * K
        d = dict(shape=sh, E=E, S=S, K=K, precision=src.precision, us_per_plan=round(us_plan, 2),
                 sample_steps_per_s=ss / (us_plan * 1e-6), drone_substeps_per_s=ss * src.N * src.S / (us_plan * 1e-6),
                 us_workaround=round(us_a, 2), us_rollout_only=round(us_b, 2),
                 bytes_per_sample_step=dict(action=act_b, reward_if_asked=rew_b, state_amortised=round(st_b, 2)),
                 hbm_share_of_plan_time=(ss * (act_b + st_b)) / HBM_BPS / (us_plan * 1e-6))
        emit(d)
        del rep, rep_b, src
        torch.cuda.empty_cache()
    from gpd_b200.examples import mppi
    import time
    mppi.run(num_envs=1024, samples=256, horizon=16, steps=4, graph=True)        # warm-up: modules, allocator
    for graph in (False, True):         # run(60 steps) - run(10 steps): the set-up cancels
        t = []
        for steps in (10, 60):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mppi.run(num_envs=1024, samples=256, horizon=16, steps=steps, graph=graph)
            torch.cuda.synchronize()
            t.append(time.perf_counter() - t0)
        emit(dict(what="mppi_control_step", E=1024, S=256, H=16, graph=graph, us_per_control_step=round((t[1] - t[0]) * 1e6 / 50, 1)))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
