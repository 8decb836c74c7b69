"""Gradient-based shooting MPC on ``HoverAviary(act=RPM)``: every env keeps a nominal H-step action schedule.  At each
control step it starts ``restarts`` candidates from the nominal (the first unperturbed, the others with Gaussian
perturbations), runs ``n_iter`` Adam ascent steps on their discounted returns through ``plan_return`` (the gradient comes
from ``gpd_plan_grad``, one launch for all envs and candidates), keeps per candidate the best schedule any iterate reached,
and adopts the candidate with the highest return.  It then steps the env with the first action and shifts the schedule.

The gradient holds the episode-end flags constant, so an ascent step alone cannot see that tilting the drone past the
truncation angle ends the episode; the return it is judged by can, since it is cut at the end step.  Keeping the best
iterate makes each control step's plan at least as good as the shifted nominal it started from.  With one candidate and
no perturbation (``--restarts 1 --sigma 0``) the example is plain Adam shooting, which on this reward reaches about
0.05 m and then tilts the drone away; ``--lr 0`` leaves random shooting over the restarts.

    python -m gpd_b200.examples.grad_mpc --num_envs 1024 --horizon 16 --restarts 16 --n_iter 4 --steps 90 [--graph]

``--graph`` captures the whole control step (restarts, Adam iterations, selection, env step) in a CUDA graph (one per
observation ping-pong parity), as ``examples/mppi.py`` does.
"""
import argparse
import time

import numpy as np
import torch

from ..envs.HoverAviary import HoverAviary
from ..utils.enums import ActionType, Physics


def run(num_envs=1024, horizon=16, restarts=16, n_iter=4, steps=90, lr=0.05, sigma=0.3, gamma=1.0, start_offset=0.3,
        seed=0, graph=False, precision="f32", device=0):
    """Returns the mean distance to the target over the envs after each control step (numpy, ``steps`` values)."""
    E, H, S = int(num_envs), int(horizon), int(restarts)
    init = np.array([[start_offset, 0.0, 1.0]])          # HoverAviary's target is (0, 0, 1)
    env = HoverAviary(initial_xyzs=init, physics=Physics.DYN, pyb_freq=240, ctrl_freq=30, act=ActionType.RPM,
                      num_envs=E, precision=precision, device=device)
    sim = env._sim
    dev = sim.device
    target = torch.tensor([0.0, 0.0, 1.0], device=dev)
    torch.cuda.manual_seed(seed)                           # the default generator: graph-capture safe
    nominal = torch.zeros((H, E, 4), device=dev)
    cand = torch.zeros((H, E, S, 1, 4), device=dev, requires_grad=True)     # (K, E, S, N, A)
    best = torch.zeros_like(cand, requires_grad=False)
    best_G = torch.zeros((E, S), device=dev, dtype=sim.real)
    opt = torch.optim.Adam([cand], lr=lr, maximize=True, capturable=True)
    envs = torch.arange(E, device=dev)
    dist = torch.zeros((), device=dev)
    obs, _ = env.reset()
    dist.copy_((obs[:, 0, :3] - target).norm(dim=-1).mean())

    def control_step():
        with torch.no_grad():
            noise = sigma * torch.randn((H, E, S, 4), device=dev)
            noise[:, :, 0] = 0
            cand.copy_((nominal[:, :, None] + noise).clamp(-1, 1)[:, :, :, None])
            best_G.fill_(-float("inf"))
            for st in opt.state.values():                  # a fresh Adam for each control step's problem
                for v in st.values():
                    v.zero_()
        for i in range(n_iter + 1):
            opt.zero_grad(set_to_none=False)
            G = sim.plan_return(cand, gamma)
            with torch.no_grad():                          # the best iterate of each candidate, by its return
                better = G > best_G
                best.copy_(torch.where(better[None, :, :, None, None], cand, best))
                best_G.copy_(torch.where(better, G, best_G))
            if i < n_iter:
                G.sum().backward()
                opt.step()
                with torch.no_grad():
                    cand.clamp_(-1, 1)
        with torch.no_grad():
            nominal.copy_(best[:, envs, best_G.argmax(1), 0])
            o = env.step(nominal[0][:, None].contiguous())[0]
            dist.copy_((o[:, 0, :3] - target).norm(dim=-1).mean())
            nominal.copy_(torch.cat([nominal[1:], torch.zeros_like(nominal[:1])]))

    trace = []
    if graph:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graphs = []
        with torch.cuda.stream(side):
            control_step()                                     # warm-up outside the capture (allocator, Adam state)
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
    ap = argparse.ArgumentParser(description="Gradient-based shooting MPC hover on Physics.DYN with plan_return")
    ap.add_argument("--num_envs", default=1024, type=int)
    ap.add_argument("--horizon", default=16, type=int)
    ap.add_argument("--restarts", default=16, type=int)
    ap.add_argument("--n_iter", default=4, type=int)
    ap.add_argument("--steps", default=90, type=int)
    ap.add_argument("--lr", default=0.05, type=float)
    ap.add_argument("--sigma", default=0.3, type=float)
    ap.add_argument("--graph", action="store_true")
    args = ap.parse_args()
    t0 = time.time()
    d = run(args.num_envs, args.horizon, args.restarts, args.n_iter, args.steps, args.lr, args.sigma, graph=args.graph)
    print(f"mean distance to target: {d[0]:.4f} m after 1 step, {d[-1]:.4f} m after {len(d)} ({time.time() - t0:.1f} s)")
