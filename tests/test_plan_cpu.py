"""Planning rollouts without a GPU: the return recurrence the GPU tests hold gpd_plan to, BatchedSim.plan's argument checks
(on a stub that has no handle), and the MPPI example's weighted update."""
import math
import types

import numpy as np
import pytest
import torch

from plan_ref import plan_returns
from gpd_b200.examples.mppi import mppi_update
from gpd_b200.sim import BatchedSim


def _ret(rew, done, gamma, dtype=torch.float64):
    return plan_returns(torch.tensor(rew, dtype=dtype)[:, None], torch.tensor(done)[:, None], gamma)


def test_returns_gamma_one_no_end():
    G, k = _ret([1.0, 2.0, 3.0], [False, False, False], 1.0)
    assert G.item() == 6.0 and k.item() == 3


def test_returns_gamma_half_end_mid():
    # 1 + 0.5*2 + 0.25*4 (the ending step's reward counts), then nothing
    G, k = _ret([1.0, 2.0, 4.0, 8.0, 16.0], [False, False, True, False, True], 0.5)
    assert G.item() == 3.0 and k.item() == 2


def test_returns_end_at_zero():
    G, k = _ret([1.5, 2.0, 3.0], [True, True, False], 0.5)
    assert G.item() == 1.5 and k.item() == 0


def test_returns_end_last_step():
    G, k = _ret([1.0, 1.0, 1.0], [False, False, True], 0.5)
    assert G.item() == 1.75 and k.item() == 2


def test_returns_nan_reward():
    G, k = _ret([1.0, float("nan"), 1.0], [False, False, False], 0.9)
    assert math.isnan(G.item()) and k.item() == 3
    G, k = _ret([1.0, 1.0, float("nan")], [False, True, False], 0.9)       # after the end: not summed
    assert G.item() == 1.9 and k.item() == 1


def test_returns_rounded_per_operation_float32():
    r = np.float32([0.1, 0.7, 1.3, 0.2])
    g = np.float32(0.9)
    G, w = np.float32(0), np.float32(1)
    for x in r:
        G = np.float32(G + np.float32(w * x))
        w = np.float32(w * g)
    out, _ = _ret(r.tolist(), [False] * 4, 0.9, torch.float32)
    assert out.item() == float(G)


def _stub(E=3, N=1, A=4, ctrl=False):
    return types.SimpleNamespace(E=E, N=N, A=A, is_ctrl=ctrl, real=torch.float32, act_dtype=torch.float32,
                                 device=torch.device("cpu"))


@pytest.mark.parametrize("shape", [(2, 3, 4, 1), (2, 4, 5, 1, 4), (2, 3, 5, 2, 4), (2, 3, 5, 1, 3), (0, 3, 5, 1, 4),
                                   (2, 3, 0, 1, 4)])
def test_plan_rejects_action_shapes(shape):
    with pytest.raises(ValueError, match="actions must have shape"):
        BatchedSim.plan(_stub(), torch.zeros(shape))


def test_plan_rejects_ctrl_env():
    with pytest.raises(ValueError, match="Ctrl"):
        BatchedSim.plan(_stub(ctrl=True), torch.zeros((2, 3, 5, 1, 4)))


@pytest.mark.parametrize("t", [torch.zeros((3, 1, 2)), torch.zeros((3, 1, 3), dtype=torch.float64),
                               torch.zeros((3, 1, 6))[..., ::2]])
def test_plan_rejects_targets(t):
    with pytest.raises(ValueError, match="targets must be"):
        BatchedSim.plan(_stub(), torch.zeros((2, 3, 5, 1, 4)), targets=t)


def _out(K, E, S, N, real=torch.float32):
    return {"returns": torch.zeros((E, S), dtype=real), "done_step": torch.zeros((E, S), dtype=torch.int32),
            "reward": torch.zeros((K, E, S), dtype=real), "final_kin": torch.zeros((E, S, N, 12))}


@pytest.mark.parametrize("name,bad", [("returns", torch.zeros((3, 4))), ("returns", torch.zeros((3, 5), dtype=torch.float64)),
                                      ("done_step", torch.zeros((3, 5))), ("reward", torch.zeros((3, 3, 5))),
                                      ("final_kin", torch.zeros((3, 5, 1, 13))),
                                      ("returns", torch.zeros((5, 3)).t())])
def test_plan_rejects_out_buffers(name, bad):
    out = _out(2, 3, 5, 1)
    out[name] = bad
    with pytest.raises(ValueError, match=f"out\\['{name}'\\]"):
        BatchedSim.plan(_stub(), torch.zeros((2, 3, 5, 1, 4)), reward=True, final_kin=True, out=out)


def test_plan_out_buffers_must_be_cuda():
    with pytest.raises(ValueError, match="CUDA"):
        BatchedSim.plan(_stub(), torch.zeros((2, 3, 5, 1, 4)), out=_out(2, 3, 5, 1))


def test_mppi_update_matches_numpy():
    rng = np.random.default_rng(3)
    H, E, S, A = 4, 5, 7, 4
    nom = rng.normal(size=(H, E, A)).astype(np.float32)
    eps = rng.normal(size=(H, E, S, A)).astype(np.float32)
    ret = rng.normal(size=(E, S)).astype(np.float32) * 3
    lam = 0.5
    got = mppi_update(torch.from_numpy(nom), torch.from_numpy(eps), torch.from_numpy(ret), lam).numpy()
    z = ret.astype(np.float64) / lam
    w = np.exp(z - z.max(1, keepdims=True))
    w /= w.sum(1, keepdims=True)
    want = nom + np.einsum("es,hesa->hea", w, eps)
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)
    # a dominant sample takes the whole update
    ret2 = np.zeros((E, S), np.float32)
    ret2[:, 2] = 100.0
    got2 = mppi_update(torch.from_numpy(nom), torch.from_numpy(eps), torch.from_numpy(ret2), 0.01).numpy()
    np.testing.assert_allclose(got2, nom + eps[:, :, 2], rtol=1e-6, atol=1e-6)
