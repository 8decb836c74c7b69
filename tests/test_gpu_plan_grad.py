"""-m gpu: planning gradients (gpd_plan_grad).  Returns and done_step are held to gpd_plan's (FP64 bit for bit); the
gradient to the torch FP64 restatement (plan_grad_ref.py) replayed on the device from the handle's exported state, to
three-point differences of gpd_plan's own returns, and in FP32 to the FP64 kernel."""
import ctypes as C
import zlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import state_edges as se
from helpers import default_targets
from plan_grad_ref import LeanRef, central_difference, start_state
from test_gpu_plan import _snapshot, make, plan_actions, shape
from test_gpu_rollout import bits, schedule
from gpd_b200 import _lib
from gpd_b200.params import load_drone_params
from gpd_b200.sim import BatchedSim
from gpd_b200.utils.enums import DroneModel

pytestmark = pytest.mark.gpu

MODELS = {"cf2x": DroneModel.CF2X, "cf2p": DroneModel.CF2P, "race": DroneModel.RACE}
# (model, shape, ctrl_freq, S, E, K, gamma): both action types, Hover and MultiHover x3, every model, 1 / 8 / 24
# substeps, ragged E and S (multi-drone copies not a multiple of the copies per CTA)
CASES = [("cf2x", "hover30", 30, 64, 37, 16, 0.9), ("cf2x", "hover30", 30, 1, 1, 1, 1.0),
         ("cf2p", "hover30", 240, 3, 37, 16, 1.0), ("race", "hover30", 10, 5, 19, 16, 0.9),
         ("cf2x", "one_d_rpm", 10, 3, 37, 16, 0.9), ("race", "one_d_rpm", 30, 7, 5, 16, 1.0),
         ("cf2x", "multi3", 30, 3, 37, 16, 1.0), ("cf2p", "multi3", 10, 5, 13, 16, 0.9),
         ("race", "multi3", 240, 64, 1, 8, 0.9)]


def kw_of(model, name, ctrl, **over):
    return shape(name, model=MODELS[model], ctrl_freq=ctrl, **over)


def source(kw, E, precision, seed, n=5, scale=0.1):
    s = make(kw, E, precision)
    s.reset()
    rng = np.random.default_rng(seed)
    for _ in range(n):
        s.step(schedule(rng, s, 1, scale)[0])
    return s, rng


def restated_grad(src, kw, acts, gamma, targets=None):
    """The restatement's returns, done_step and gradient (K, E, S, N, A), replayed in FP64 on the device."""
    K, E, S, N, A = acts.shape
    st, rr, _, cnt = src.get_state()
    rep = lambda t: t.double().repeat_interleave(S, 0)
    st0 = start_state(rep(st), rep(rr))
    tg = torch.as_tensor(np.broadcast_to(default_targets(kw), (E, N, 3)) if targets is None else targets,
                         dtype=torch.float64, device="cuda").repeat_interleave(S, 0)
    a = acts.double().reshape(K, E * S, N, A).clone().requires_grad_(True)
    G, done, *_ = LeanRef(load_drone_params(kw["model"]), kw).plan(st0, cnt.repeat_interleave(S, 0), a, tg, gamma)
    G.sum().backward()
    return G.detach().reshape(E, S), done.reshape(E, S), a.grad.reshape(K, E, S, N, A)


def rel_to_copy(x, y):
    """max over copies of max|x - y| / max|y| (per copy (e, s), over k, i, j)."""
    d = (x - y).abs().permute(1, 2, 0, 3, 4).flatten(2).amax(-1)
    n = y.abs().permute(1, 2, 0, 3, 4).flatten(2).amax(-1).clamp_min(1e-300)
    return (d / n).max().item()


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("model,name,ctrl,S,E,K,gamma", CASES)
def test_plan_grad_returns_match_plan(precision, model, name, ctrl, S, E, K, gamma):
    kw = kw_of(model, name, ctrl)
    src, rng = source(kw, E, precision, zlib.crc32(f"{model} {name} {ctrl} {S} {E}".encode()))
    acts = plan_actions(rng, src, K, S)
    for tg in (None, torch.as_tensor(np.array(default_targets(kw))[None] + rng.uniform(-0.3, 0.3, (E, kw["num_drones"], 3)),
                                     dtype=src.real, device="cuda").contiguous()):
        ref = {k: v.clone() for k, v in src.plan(acts, gamma=gamma, targets=tg).items()}
        res = src.plan_grad(acts, gamma=gamma, targets=tg)
        if precision == "f64":
            assert torch.equal(bits(res["returns"]), bits(ref["returns"]))
        else:
            same = torch.equal(bits(res["returns"]), bits(ref["returns"]))
            print(f"[plan_grad] f32 {model} {name} {ctrl}: returns bit-identical to gpd_plan: {same}")
            assert torch.allclose(res["returns"], ref["returns"], rtol=1e-4, atol=1e-4)
        assert torch.equal(res["done_step"], ref["done_step"])


@pytest.mark.parametrize("model,name,ctrl,S,E,K,gamma", CASES)
def test_plan_grad_matches_restatement(model, name, ctrl, S, E, K, gamma):
    kw = kw_of(model, name, ctrl)
    src, rng = source(kw, E, "f64", zlib.crc32(f"{model} {name} {ctrl} {S} {E} g".encode()))
    acts = plan_actions(rng, src, K, S, scale=0.1)
    res = src.plan_grad(acts, gamma=gamma)
    G, done, g = restated_grad(src, kw, acts, gamma)
    assert torch.equal(res["done_step"], done.to(torch.int32))
    assert (res["returns"] - G).abs().max().item() <= 1e-9
    err = rel_to_copy(res["grad"], g)
    print(f"[plan_grad] f64 {model} {name} {ctrl}: gradient vs the restatement {err:.2e} of each copy's max-norm")
    assert err <= 1e-9


@pytest.mark.parametrize("name", ["hover30", "one_d_rpm", "multi3"])
def test_plan_grad_f32_against_f64(name):
    kw = kw_of("cf2x", name, 30)
    E, S, K = 64, 4, 16
    a, rng = source(kw, E, "f64", 21, n=2, scale=0.05)
    b = make(kw, E, "f32")
    b.reset()
    b.set_state(*a.get_state())
    acts = plan_actions(rng, a, K, S, scale=0.05)
    g64 = a.plan_grad(acts, gamma=0.95)["grad"].reshape(K, E * S, -1).permute(1, 0, 2).flatten(1)
    g32 = b.plan_grad(acts, gamma=0.95)["grad"].double().reshape(K, E * S, -1).permute(1, 0, 2).flatten(1)
    cos = torch.nn.functional.cosine_similarity(g32, g64, dim=1)
    ratio = g32.norm(dim=1) / g64.norm(dim=1)
    print(f"[plan_grad] f32 vs f64 {name}: 1 - cosine <= {(1 - cos).max().item():.1e}, |norm ratio - 1| <= "
          f"{(ratio - 1).abs().max().item():.1e}")
    # measured on a B200: 1 - cosine ~1e-12, |ratio - 1| <= 1.0e-6 near hover at K = 16; bounds with a 10x margin
    assert (1 - cos).max().item() <= 1e-5 and (ratio - 1).abs().max().item() <= 1e-5


@pytest.mark.parametrize("name,ctrl", [("hover30", 30), ("one_d_rpm", 10), ("multi3", 240)])
def test_plan_grad_matches_plan_differences(name, ctrl):
    """Three-point differences of gpd_plan's own FP64 returns with h = 2^-10 (exact in the float32 actions): copy 5j
    unperturbed, 5j+1..5j+4 at +h, -h, +2h, -2h on one entry.  The O(h^2) budget is estimated from the same differences
    at 2h (Richardson: the error at h is a third of the change from 2h to h)."""
    kw = kw_of("cf2x", name, ctrl)
    E, K, n, h = 4, 12, 6, 2.0 ** -10
    src, rng = source(kw, E, "f64", 31, n=2, scale=0.02)
    N, A = src.N, src.A
    base = plan_actions(rng, src, K, 1, scale=0.02)
    grad = src.plan_grad(base, gamma=0.95)["grad"][:, :, 0]
    coords = [(int(rng.integers(K)), int(rng.integers(N)), int(rng.integers(A))) for _ in range(n)]
    acts = base.repeat(1, 1, 5 * n, 1, 1)
    for j, (k, i, c) in enumerate(coords):
        for m, step in enumerate((h, -h, 2 * h, -2 * h)):
            acts[k, :, 5 * j + 1 + m, i, c] += step
    res = src.plan(acts, gamma=0.95, reward=True)
    G = res["returns"].cpu().numpy()
    rew = res["reward"].cpu().numpy()
    done = res["done_step"].cpu().numpy()
    assert (done == done[:, :1]).all(), "a flag changed within +-2h"
    worst = 0.0
    for e in range(E):
        kend = min(done[e, 0], K - 1)
        assert (rew[:kend + 1, e] > 0).all(), "the reward's clip changed within +-2h"
        scale = grad[:, e].abs().max().item()
        for j, (k, i, c) in enumerate(coords):
            a = acts[k, e, 5 * j:5 * j + 5, i, c].cpu().numpy()
            g5 = G[e, 5 * j:5 * j + 5]
            fd_h = central_difference(g5[[0, 1, 2]], a[[0, 1, 2]])
            fd_2h = central_difference(g5[[0, 3, 4]], a[[0, 3, 4]])
            budget = abs(fd_2h - fd_h) / 3
            assert budget <= 1e-3 * scale, (e, k, i, c, budget, scale)         # the budget itself is O(h^2) small
            tol = 1.5 * budget + 1e-8 * scale + 64 * 2.0 ** -52 * abs(g5[0]) / h
            err = abs(fd_h - grad[k, e, i, c].item())
            assert err <= tol, (e, k, i, c, fd_h, grad[k, e, i, c].item(), budget, scale)
            worst = max(worst, err / max(scale, 1e-300))
    print(f"[plan_grad] {name}: gradient vs three-point differences (h = 2^-10) within {worst:.1e} of the max-norm")


@pytest.mark.parametrize("fam", ["F5", "F7"])
@pytest.mark.parametrize("name", ["hover30", "multi3"])
def test_plan_grad_episode_ends(fam, name):
    K, S, E = 16, 3, 96
    seen = set()
    for ep in (8.0, 1 / 3):
        kw = shape(name, episode_len_sec=ep)
        f = se.FAMILIES[fam](np.random.default_rng(7), kw, E, "f64")
        src = make(kw, E, "f64")
        src.reset()
        src.set_state(torch.as_tensor(f["state20"]), torch.as_tensor(f["rpy_rates"]), torch.as_tensor(f["pid_state"]),
                      torch.as_tensor(f["step_counter"]))
        a2 = torch.as_tensor(f["actions"], dtype=torch.float32, device="cuda")
        acts = a2[torch.arange(K) % 2][:, :, None].expand(K, E, S, kw["num_drones"], src.A).contiguous()
        ref = {k: v.clone() for k, v in src.plan(acts, gamma=0.9).items()}
        res = src.plan_grad(acts, gamma=0.9)
        assert torch.equal(bits(res["returns"]), bits(ref["returns"])) and torch.equal(res["done_step"], ref["done_step"])
        done = res["done_step"].long()
        rows = torch.arange(K, device="cuda")[:, None, None] > done[None]
        g = res["grad"].flatten(3)
        assert (g[rows] == 0).all(), "rows after the end step"
        fin = torch.stack([torch.isfinite(x).all(-1).all(-1) for x in src.get_state()[:2]]).all(0)
        if fin.all():
            # copies that end at k = 0 have a gradient in row 0 only; finite starts have finite gradients
            assert torch.isfinite(g).all()
        seen |= set(np.unique(done.cpu().numpy()).tolist())
    if fam == "F5":
        assert 0 in seen and K in seen and any(0 < k < K for k in seen), sorted(seen)


@pytest.mark.parametrize("kind", ["f32_chained_65536", "f64_multihover"])
def test_plan_grad_leaves_the_source_untouched(kind):
    if kind == "f32_chained_65536":
        kw, E, prec, chaining = shape("hover30"), 65536, "f32", True
    else:
        kw, E, prec, chaining = shape("multi3", episode_len_sec=0.3), 37, "f64", False
    a, b = make(kw, E, prec, chaining=chaining), make(kw, E, prec, chaining=chaining)
    rng = np.random.default_rng(11)
    sched = [schedule(rng, a, 1)[0] for _ in range(12)]
    for s in (a, b):
        s.reset()
        for k in range(7):
            s.step(sched[k])
    before = _snapshot(a)
    a.plan_grad(plan_actions(rng, a, 8, 4), gamma=0.9)
    for x, y in zip(before, _snapshot(a)):
        assert torch.equal(x, y)
    for s in (a, b):
        for k in range(7, 12):
            s.step(sched[k])
    torch.cuda.synchronize()
    for x, y in zip(_snapshot(a), _snapshot(b)):
        assert torch.equal(x, y)
    assert np.array_equal(a.episode_stats(), b.episode_stats())


def test_plan_return_graph_replay():
    kw = shape("hover30")
    s = make(kw, 65536, "f32", chaining=True)
    s.reset()
    rng = np.random.default_rng(9)
    for _ in range(4):
        s.step(schedule(rng, s, 1)[0])
    acts = plan_actions(rng, s, 16, 2)
    eager = {k: v.clone() for k, v in s.plan_grad(acts, gamma=0.9).items()}
    x = acts.clone().requires_grad_(True)
    s.plan_return(x, 0.9).sum().backward()
    assert torch.equal(x.grad, eager["grad"])
    out = s.alloc_plan_grad_outputs(16, 2)
    y = acts.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            s.plan_grad(acts, gamma=0.9, out=out)
            G = s.plan_return(y, 0.9)
            G.sum().backward()
    torch.cuda.current_stream().wait_stream(side)
    for v in (out["returns"], out["grad"]):
        v.zero_()
    g.replay()
    torch.cuda.synchronize()
    for k in ("returns", "done_step", "grad"):
        assert torch.equal(bits(eager[k]), bits(out[k])), k
    assert torch.equal(bits(G), bits(eager["returns"])) and torch.equal(bits(y.grad), bits(eager["grad"]))


def test_plan_grad_invalid_arguments():
    L = _lib.load()
    kw = shape("hover30")
    s = make(kw, 4096, "f32")
    s.reset()
    E, N, A, K, S = s.E, s.N, s.A, 4, 2
    acts = torch.zeros((K, E, S, N, A), device="cuda")
    big = torch.zeros(K * E * S * N * A + 4, device="cuda")
    ret = torch.zeros((E, S), device="cuda")
    done = torch.zeros((E, S), dtype=torch.int32, device="cuda")
    grad = torch.zeros((K, E, S, N, A), device="cuda")
    nb = s.plan_grad_tape_bytes(K, S)
    print(f"[plan_grad] tape of {E} envs x {S} samples x {K} steps: {nb} B")
    assert nb == K * 13 * E * S * N * 4
    tape = torch.zeros(nb + 16, dtype=torch.uint8, device="cuda")
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)
    st = s._stream()
    ok = (s.h, K, S, p(acts), None, 0.9, p(ret), p(done), p(grad), p(tape), nb, st)
    assert L.gpd_plan_grad(*ok) == 0
    names = ["h", "K", "S", "actions", "targets", "gamma", "returns", "done_step", "grad", "tape", "tape_bytes", "stream"]

    def bad(**kv):
        args = list(ok)
        for k, v in kv.items():
            args[names.index(k)] = v
        return L.gpd_plan_grad(*args)
    cases = [dict(K=0), dict(S=0), dict(K=-1), dict(gamma=float("nan")), dict(gamma=float("inf")), dict(gamma=-0.1),
             dict(gamma=1.5), dict(actions=None), dict(returns=None), dict(grad=None), dict(tape=None),
             dict(tape_bytes=nb - 1), dict(actions=p(big, 4)), dict(tape=p(tape, 4)), dict(done_step=p(ret)),
             dict(grad=p(ret)), dict(tape=p(grad)), dict(returns=p(acts)), dict(targets=p(grad)), dict(S=2 ** 31 - 1)]
    for c in cases:
        assert bad(**c) == -1, c
        assert L.gpd_plan_grad(*ok) == 0, f"handle unusable after {c}"
    # a tape size that matches 2^31 - 1 samples reaches the grid check (rejected before any launch, nothing is touched)
    huge = L.gpd_plan_grad_tape_bytes(s.h, K, 2 ** 31 - 1)
    assert huge > 0 and bad(S=2 ** 31 - 1, tape_bytes=huge) == -1
    assert b"INT32_MAX" in L.gpd_last_error()
    assert L.gpd_plan_grad(*ok) == 0
    assert L.gpd_plan_grad_tape_bytes(s.h, 0, S) == -1 and L.gpd_plan_grad_tape_bytes(s.h, K, 0) == -1
    dp = load_drone_params(DroneModel.CF2X)
    others = [BatchedSim(dp, 4, 1, env_kind="ctrl", action_type="ctrl_rpm", pyb_freq=240, ctrl_freq=48, precision="f32")]
    for at in ("pid", "vel", "one_d_pid"):
        others.append(BatchedSim(dp, 4, 1, env_kind="hover", action_type=at, precision="f32", target_pos=[[0, 0, 1]]))
    multi2 = default_targets(dict(model=DroneModel.CF2X, num_drones=2, env_kind="multihover"))
    for phy in (1, 2, 4):
        others.append(BatchedSim(dp, 4, 2, env_kind="multihover", action_type="rpm", physics_flags=phy, precision="f64",
                                 target_pos=multi2))
    for o in others:
        Eo, No, Ao = o.E, o.N, o.A
        ao = torch.zeros((K, Eo, S, No, Ao), dtype=o.act_dtype, device="cuda")
        ro = torch.zeros((Eo, S), dtype=o.real, device="cuda")
        go = torch.zeros((K, Eo, S, No, Ao), dtype=o.real, device="cuda")
        assert L.gpd_plan_grad(o.h, K, S, p(ao), None, 1.0, p(ro), None, p(go), p(tape), nb, st) == -1
        assert b"gpd_plan_grad" in L.gpd_last_error()
        with pytest.raises(ValueError):
            o.plan_grad(ao)
    s.step(torch.zeros((E, N, A), device="cuda"))
    torch.cuda.synchronize()


def test_plan_grad_large_copy_count():
    kw = shape("hover30")
    E, S, K = 4096, 256, 16
    src, rng = source(kw, E, "f32", 12)
    acts = plan_actions(rng, src, K, S, scale=0.1)
    nb = src.plan_grad_tape_bytes(K, S)
    print(f"[plan_grad] {E * S} copies x {K} steps: tape {nb / 2 ** 20:.0f} MiB")
    res = src.plan_grad(acts, gamma=0.99)
    ref = src.plan(acts, gamma=0.99)
    assert torch.equal(res["done_step"], ref["done_step"])
    assert torch.allclose(res["returns"], ref["returns"], rtol=1e-4, atol=1e-4)
    envs = [0, 1111, 4095]
    b = make(kw, len(envs), "f64")
    b.reset()
    b.set_state(*(x[envs] for x in src.get_state()))
    sub = acts[:, envs, :8].contiguous()
    g64 = b.plan_grad(sub, gamma=0.99)["grad"]
    g32 = res["grad"][:, envs, :8].double()
    cos = torch.nn.functional.cosine_similarity(g32.permute(1, 2, 0, 3, 4).flatten(2), g64.permute(1, 2, 0, 3, 4).flatten(2), dim=-1)
    assert (1 - cos).max().item() <= 1e-5


def test_grad_mpc_example():
    from gpd_b200.examples import grad_mpc
    d = grad_mpc.run(num_envs=64, horizon=16, steps=90, start_offset=0.3)
    print(f"[plan_grad] grad MPC 64 envs, 16 restarts x 4 Adam steps, H=16: mean distance {d[0]:.4f} m after 1 step, "
          f"{d[-1]:.4f} m after 90 steps")
    assert d[-1] < 0.15, d[::10]
    g = grad_mpc.run(num_envs=64, horizon=16, steps=90, start_offset=0.3, graph=True)
    print(f"[plan_grad] grad MPC graphed: {g[-1]:.4f} m after 90 steps")
    assert g[-1] < 0.15, g[::10]
    r = grad_mpc.run(num_envs=64, horizon=16, steps=90, start_offset=0.3, lr=0.0)
    print(f"[plan_grad] the same restarts without gradient steps (lr = 0): {r[-1]:.4f} m after 90 steps")
    p = grad_mpc.run(num_envs=64, horizon=16, steps=90, start_offset=0.3, restarts=1, sigma=0.0)
    print(f"[plan_grad] one candidate, plain Adam shooting: {p.min():.4f} m at best, {p[-1]:.4f} m after 90 steps")
    z = grad_mpc.run(num_envs=64, horizon=4, n_iter=2, steps=30, start_offset=0.3, lr=0.0, sigma=0.0)
    assert np.allclose(z, 0.3, atol=1e-3), z[::5]
