"""Planning gradients without a GPU: the torch restatement (plan_grad_ref.py) the GPU tests hold gpd_plan_grad to, checked
against the CPU oracle (values to 1e-12 over 32 control steps, gradients against central differences of the oracle's
return), BatchedSim.plan_grad's argument checks (on a stub that has no handle) and plan_return's backward."""
import types
import zlib

import numpy as np
import pytest
import torch

import state_edges as se
from plan_grad_ref import LeanRef, central_difference, start_state
from helpers import default_targets
from plan_ref import plan_returns
from gpd_b200.params import load_drone_params
from gpd_b200.sim import BatchedSim, _PlanReturn
from gpd_b200.utils.enums import DroneModel

MODELS = {"cf2x": DroneModel.CF2X, "cf2p": DroneModel.CF2P, "race": DroneModel.RACE}
# (model, shape, ctrl_freq): every model, both action types, Hover and MultiHover x3, 1 / 8 / 24 substeps
CASES = [("cf2x", "hover30", 30), ("cf2p", "hover30", 240), ("race", "hover30", 10), ("cf2x", "one_d_rpm", 10),
         ("race", "one_d_rpm", 30), ("cf2x", "multi3", 30), ("cf2p", "multi3", 10), ("race", "multi3", 240)]


def _setup(model, name, ctrl, E, rng, near=False):
    kw = se.shape(name, model=MODELS[model], ctrl_freq=ctrl)
    N = kw["num_drones"]
    tgt = default_targets(kw)
    init_xyz = init_rpy = None
    if near:        # near hover around the target: no clip or flag changes under small perturbations
        init_xyz = tgt[None] + rng.uniform(-0.1, 0.1, (E, N, 3))
        init_rpy = rng.uniform(-0.05, 0.05, (E, N, 3))
    ref = se.oracle_sim(kw, E, init_xyz=init_xyz, init_rpy=init_rpy)
    ref.reset()
    return kw, ref, np.broadcast_to(tgt, (E, N, 3))


def _oracle_plan(ref, acts, gamma):
    """acts (K, E, N, A) float32 -> the oracle's rewards, flags, states and the recurrence's returns."""
    rew, done, st = [], [], []
    for k in range(acts.shape[0]):
        _, r, te, tr = ref.step(acts[k])
        rew.append(r.copy())
        done.append((te | tr).astype(bool))
        st.append((ref.state20.copy(), ref.rpy_rates.copy(), te.copy(), tr.copy()))
    G, step = plan_returns(torch.tensor(np.stack(rew)), torch.tensor(np.stack(done)), gamma)
    return G.numpy(), step.numpy(), np.stack(rew), st


def _start(ref):
    return start_state(torch.tensor(ref.state20), torch.tensor(ref.rpy_rates)), torch.tensor(ref.step_counter)


@pytest.mark.parametrize("model,name,ctrl", CASES)
def test_restatement_matches_oracle(model, name, ctrl):
    rng = np.random.default_rng(zlib.crc32(f"{model} {name} {ctrl}".encode()))
    E, K = 6, 32
    kw, ref, tgt = _setup(model, name, ctrl, E, rng)
    A = se.A_WIDTH[kw["action_type"]]
    acts = rng.uniform(-0.4, 0.4, (K, E, kw["num_drones"], A)).astype(np.float32)
    lr = LeanRef(load_drone_params(kw["model"]), kw)
    st0, cnt = _start(ref)
    G, done, states, rew, term, trunc = lr.plan(st0, cnt, torch.tensor(acts, dtype=torch.float64), torch.tensor(tgt), 0.9)
    Go, do, rewo, sto = _oracle_plan(ref, acts, 0.9)
    for k in range(K):
        s20, rr, te, tr = sto[k]
        s = states[k]
        got = torch.cat([s["p"], s["q"], s["rpy"], s["v"], s["av"]], -1).numpy()
        want = s20[..., :16]
        d = np.abs(got - want)
        d[..., 7:10] = np.minimum(d[..., 7:10], np.abs(2 * np.pi - d[..., 7:10]))
        assert d.max() <= 1e-12, (k, d.max(axis=(0, 1)))
        assert np.abs(s["w"].numpy() - rr).max() <= 1e-12, k
        assert np.array_equal(term[k].numpy(), te.astype(bool)) and np.array_equal(trunc[k].numpy(), tr.astype(bool)), k
    assert np.abs(rew.numpy() - rewo).max() <= 1e-12
    assert np.array_equal(done.numpy(), do) and np.abs(G.numpy() - Go).max() <= 1e-12


@pytest.mark.parametrize("model,name,ctrl", CASES)
def test_restatement_gradient_matches_oracle_differences(model, name, ctrl):
    rng = np.random.default_rng(zlib.crc32(f"{model} {name} {ctrl} grad".encode()))
    E, K, n, h, gamma = 3, 16, 8, 2.0 ** -14, 0.95
    kw, ref, tgt = _setup(model, name, ctrl, E, rng, near=True)
    N, A = kw["num_drones"], se.A_WIDTH[kw["action_type"]]
    acts = (np.round(rng.uniform(-0.02, 0.02, (K, E, N, A)) * 2 ** 20) / 2 ** 20).astype(np.float32)
    lr = LeanRef(load_drone_params(kw["model"]), kw)
    st0, cnt = _start(ref)
    a = torch.tensor(acts, dtype=torch.float64, requires_grad=True)
    G, done, _, rew, _, _ = lr.plan(st0, cnt, a, torch.tensor(tgt), gamma)
    assert (rew > 0).all()
    G.sum().backward()
    grad = a.grad.numpy()
    # n random coordinates per env, each run unperturbed, at +h and at -h on copies of its env in one oracle batch
    coords = [(int(rng.integers(K)), e, int(rng.integers(N)), int(rng.integers(A))) for e in range(E) for _ in range(n)]
    sub = [c[1] for c in coords for _ in range(3)]
    big = se.oracle_sim(kw, len(sub))
    big.state20[...], big.rpy_rates[...], big.step_counter[...] = ref.state20[sub], ref.rpy_rates[sub], ref.step_counter[sub]
    pa = acts[:, sub].copy()
    for j, (k, e, i, c) in enumerate(coords):
        pa[k, 3 * j + 1, i, c] += np.float32(h)
        pa[k, 3 * j + 2, i, c] -= np.float32(h)
    Gp, dp, rp, _ = _oracle_plan(big, pa, gamma)
    assert np.array_equal(dp, done.numpy()[sub]) and (rp > 0).all(), "a flag or the clip changed within +-h"
    for j, (k, e, i, c) in enumerate(coords):
        fd = central_difference(Gp[3 * j:3 * j + 3], pa[k, 3 * j:3 * j + 3, i, c])
        # O(h^2) truncation, and the returns' rounding (~64 ulp of |G|) over the step in u
        tol = 1e-6 * np.abs(grad[:, e]).max() + 64 * 2.0 ** -52 * abs(Gp[3 * j]) / h
        assert abs(fd - grad[k, e, i, c]) <= tol, (k, e, i, c, fd, grad[k, e, i, c], tol)


# ---- BatchedSim.plan_grad's checks, on a stub without a handle ----
def _stub(E=3, N=1, A=4, ctrl=False, action_type="rpm", physics_flags=0):
    return types.SimpleNamespace(E=E, N=N, A=A, is_ctrl=ctrl, real=torch.float32, act_dtype=torch.float32,
                                 device=torch.device("cpu"), action_type=action_type, physics_flags=physics_flags,
                                 plan_grad_tape_bytes=lambda K, S: 13 * 4 * K * S * E * N)


@pytest.mark.parametrize("kw", [dict(ctrl=True), dict(action_type="pid"), dict(action_type="vel"),
                                dict(action_type="one_d_pid"), dict(physics_flags=1), dict(physics_flags=4)])
def test_plan_grad_rejects_configurations(kw):
    with pytest.raises(ValueError, match="plan_grad differentiates"):
        BatchedSim.plan_grad(_stub(**kw), torch.zeros((2, 3, 5, 1, 4)))


@pytest.mark.parametrize("shape", [(2, 3, 4, 1), (2, 4, 5, 1, 4), (2, 3, 5, 2, 4), (0, 3, 5, 1, 4), (2, 3, 0, 1, 4)])
def test_plan_grad_rejects_action_shapes(shape):
    with pytest.raises(ValueError, match="actions must have shape"):
        BatchedSim.plan_grad(_stub(), torch.zeros(shape))


def test_plan_grad_rejects_targets():
    with pytest.raises(ValueError, match="targets must be"):
        BatchedSim.plan_grad(_stub(), torch.zeros((2, 3, 5, 1, 4)), targets=torch.zeros((3, 1, 3), dtype=torch.float64))


def _out(K=2, E=3, S=5, N=1, A=4):
    return {"returns": torch.zeros((E, S)), "done_step": torch.zeros((E, S), dtype=torch.int32),
            "grad": torch.zeros((K, E, S, N, A)), "tape": torch.zeros(13 * 4 * K * S * E * N, dtype=torch.uint8)}


@pytest.mark.parametrize("name,bad", [("grad", torch.zeros((2, 3, 5, 1, 3))), ("grad", torch.zeros((2, 3, 5, 1, 4),
                                      dtype=torch.float64)), ("grad", torch.zeros((2, 3, 5, 1, 8))[..., ::2]),
                                      ("returns", torch.zeros((3, 4))), ("done_step", torch.zeros((3, 5)))])
def test_plan_grad_rejects_out_buffers(name, bad):
    out = _out()
    out[name] = bad
    with pytest.raises(ValueError, match=f"out\\['{name}'\\]"):
        BatchedSim.plan_grad(_stub(), torch.zeros((2, 3, 5, 1, 4)), out=out)


def test_plan_grad_out_buffers_must_be_cuda():
    with pytest.raises(ValueError, match="CUDA"):
        BatchedSim.plan_grad(_stub(), torch.zeros((2, 3, 5, 1, 4)), out=_out())


def test_plan_return_backward_scales_the_kernel_gradient():
    E, S, K = 3, 5, 2
    grad = torch.randn((K, E, S, 1, 4), dtype=torch.float64)
    ret = torch.randn((E, S), dtype=torch.float64)
    stub = types.SimpleNamespace(plan_grad=lambda a, gamma, targets: {"returns": ret.clone(), "grad": grad})
    a = torch.zeros((K, E, S, 1, 4), requires_grad=True)
    G = _PlanReturn.apply(stub, a, 0.9, None)
    assert torch.equal(G, ret)
    w = torch.randn((E, S), dtype=torch.float64)
    (G * w).sum().backward()
    assert a.grad.dtype == torch.float32
    assert torch.equal(a.grad, (w[None, :, :, None, None] * grad).float())
