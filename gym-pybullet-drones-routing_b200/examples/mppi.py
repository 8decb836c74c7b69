"""Batched MPPI on ``HoverAviary(act=RPM)``: every env keeps a nominal H-step action schedule and, at each control step,
scores S Gaussian perturbations of it with ``env.plan`` (one launch for all envs and samples), moves the nominal to the
softmax(returns / lambda)-weighted mean, steps the env with its first action and shifts it by one step.

    python -m gpd_b200.examples.mppi --num_envs 1024 --samples 256 --horizon 16 --steps 90 [--graph]

``--graph`` captures plan + update + step of one control step in a CUDA graph (one per observation ping-pong parity).
"""
import argparse
import time

import numpy as np
import torch

from ..envs.HoverAviary import HoverAviary
from ..utils.enums import ActionType, Physics


def mppi_update(nominal, eps, returns, lam):
    """nominal (H, E, A), eps (H, E, S, A) perturbations, returns (E, S) -> the new nominal: nominal + sum_s w_s eps_s with
    w = softmax(returns / lam) over the samples of each env."""
    w = torch.softmax(returns / lam, dim=1).to(nominal.dtype)
    return nominal + torch.einsum("es,hesa->hea", w, eps)


def run(num_envs=1024, samples=256, horizon=16, steps=90, lam=1e-4, sigma=0.3, start_offset=0.3, seed=0, graph=False,
        precision="f32", device=0):
    """Returns the mean distance to the target over the envs after each control step (numpy, ``steps`` values)."""
    E, S, H = int(num_envs), int(samples), int(horizon)
    init = np.array([[start_offset, 0.0, 1.0]])          # HoverAviary's target is (0, 0, 1)
    env = HoverAviary(initial_xyzs=init, physics=Physics.DYN, pyb_freq=240, ctrl_freq=30, act=ActionType.RPM,
                      num_envs=E, precision=precision, device=device)
    dev = env._sim.device
    target = torch.tensor([0.0, 0.0, 1.0], device=dev)
    torch.cuda.manual_seed(seed)                           # the default generator: graph-capture safe
    nominal = torch.zeros((H, E, 4), device=dev)
    cand = torch.empty((H, E, S, 1, 4), device=dev)
    out = env._sim.alloc_plan_outputs(H, S)
    dist = torch.zeros((), device=dev)
    obs, _ = env.reset()
    dist.copy_((obs[:, 0, :3] - target).norm(dim=-1).mean())

    def control_step():
        eps = sigma * torch.randn((H, E, S, 4), device=dev)
        cand.copy_((nominal[:, :, None] + eps).clamp(-1, 1)[:, :, :, None])
        res = env.plan(cand, out=out)
        nominal.copy_(mppi_update(nominal, cand[:, :, :, 0] - nominal[:, :, None], res["returns"], lam))
        o = env.step(nominal[0][:, None].contiguous())[0]
        dist.copy_((o[:, 0, :3] - target).norm(dim=-1).mean())
        nominal.copy_(torch.cat([nominal[1:], torch.zeros_like(nominal[:1])]))

    trace = []
    if graph:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graphs = []
        with torch.cuda.stream(side):
            control_step()                                     # warm-up outside the capture (allocator, modules)
            trace.append(dist.item())
            for _ in range(2):                                 # the env's observation ping-pong: one graph per parity
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    control_step()
                graphs.append(g)
        torch.cuda.current_stream(dev).wait_stream(side)
        for k in range(1, steps):
            graphs[(k - 1) % 2].replay()
            trace.append(dist.item())
    else:
        for _ in range(steps):
            control_step()
            trace.append(dist.item())
    env.close()
    return np.array(trace)


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description="Batched MPPI hover on Physics.DYN with env.plan")
    ap.add_argument("--num_envs", default=1024, type=int)
    ap.add_argument("--samples", default=256, type=int)
    ap.add_argument("--horizon", default=16, type=int)
    ap.add_argument("--steps", default=90, type=int)
    ap.add_argument("--lam", default=1e-4, type=float)
    ap.add_argument("--sigma", default=0.3, type=float)
    ap.add_argument("--graph", action="store_true")
    args = ap.parse_args()
    t0 = time.time()
    d = run(args.num_envs, args.samples, args.horizon, args.steps, args.lam, args.sigma, graph=args.graph)
    print(f"mean distance to target: {d[0]:.4f} m after 1 step, {d[-1]:.4f} m after {len(d)} ({time.time() - t0:.1f} s)")
