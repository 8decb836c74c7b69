"""The state families of tests/state_edges.py cover the branches they claim (computed in numpy in the kernels' order of
operations, and with the CPU oracle), so that tests/test_gpu_state_edges.py cannot quietly stop reaching a branch when a
generator drifts; and the oracle's Bullet conversions agree bit for bit with the pybullet stand-in on those attitudes."""
import importlib.util
import os

import numpy as np
import pytest

import state_edges as se
from helpers import ROOT
from gpd_b200.params import load_drone_params
from oracle import oracle as orc

PRECISIONS = ("f64", "f32")


def _pybullet_shim():
    spec = importlib.util.spec_from_file_location("_refshim_pybullet", os.path.join(ROOT, "oracle", "refshim", "pybullet.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("fam", ["F2", "F3", "F4"])
def test_oracle_conversions_match_pybullet_stand_in(fam, precision):
    pb = _pybullet_shim()
    d = se.FAMILIES[fam](np.random.default_rng(1), se.shape("hover30"), 257, precision)
    for q in d["state20"][..., 3:7].reshape(-1, 4):
        e_o, e_p = orc.euler_from_quaternion(q), np.array(pb.getEulerFromQuaternion(q))
        assert np.array_equal(e_o, e_p), (q, e_o, e_p)
        assert np.array_equal(orc.matrix_from_quaternion(q).ravel(), np.array(pb.getMatrixFromQuaternion(q))), q


def _t32(rates, pyb):
    h = np.float32(np.float32(1.0 / pyb) * np.float32(.5))            # LeanStep::h, hh; integrate_q<float>'s h*h
    r = rates.astype(np.float32)
    return (r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1] + r[..., 2] * r[..., 2]) * (h * h)


def _t64(rates, pyb):
    h = (1.0 / pyb) * .5
    return (rates ** 2).sum(-1) * (h * h)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["hover30", "hover60_20", "hover240", "one_d_rpm", "multi3", "ctrl1"])
def test_f1_straddles_the_quaternion_update_switches(name, precision):
    """Envs strictly on both sides of t = 0.04 (lean_substep_f32) and t = 0.25 (integrate_q<float>), within 1e-4 of each,
    at every frequency; |w| on both sides of the reference's 1e-8 early return; all of it constant over the step."""
    kw = se.shape(name)
    d = se.f1_rates(np.random.default_rng(2), kw, 257, precision)
    rr = d["rpy_rates"]
    for t in (_t32(rr, kw["pyb_freq"]).astype(np.float64), _t64(rr, kw["pyb_freq"])):
        for thr in (0.04, 0.25):
            assert np.any((t < thr) & (t > thr * (1 - 1e-4))) and np.any((t > thr) & (t < thr * (1 + 1e-4))), (thr, name)
    n = np.linalg.norm(rr, axis=-1)
    assert np.any((n > 0) & (n < 1e-8)) and np.any((n > 1e-8) & (n < 1e-7)) and np.any(n == 0)
    assert np.any(n == 1e-8) or precision == "f32"         # float32(1e-8) lies just below 1e-8
    # principal-axis envs: balanced rotors keep |w| (and so t) the same through every substep
    ref = se.oracle_sim(kw, 257)
    se.inject_oracle(ref, d)
    ax = d["groups"]["axis"]
    ref.step(d["actions"][0])
    assert np.array_equal(ref.rpy_rates[ax], d["rpy_rates"][ax])
    assert len(d["groups"]["generic"]) >= 100


@pytest.mark.parametrize("precision", PRECISIONS)
def test_f2_sarg_straddles_the_gimbal_threshold(precision):
    """sarg on both sides of +-0.99999 (float64, the FP64 kernels) and of +-float32(0.99999) (float32, the FP32 kernels),
    with envs outside the FP32 band of 64 ulp on both sides; the band holds < 5 % of the drones."""
    d = se.f2_attitudes(np.random.default_rng(3), se.shape("hover30"), 513, precision)
    q = d["state20"][..., 3:7].reshape(-1, 4)
    if precision == "f64":
        s = se.sarg(q)
        for sg in (1, -1):
            v = sg * s
            assert np.any((v >= se.SARG_T) & (v < se.SARG_T + 1e-12)) and np.any((v < se.SARG_T) & (v > se.SARG_T - 1e-12))
    else:
        s = se.sarg(q, np.float32)
        thr, ulp = np.float32(se.SARG_T32), np.spacing(np.float32(1))
        for sg in (1, -1):
            v = (sg * s).astype(np.float64)
            assert np.any(v >= thr + 64 * ulp) and np.any((v < thr - 64 * ulp) & (v > 0.9999))
            assert np.any((v >= thr) & (v < thr + 64 * ulp)) and np.any((v < thr) & (v > thr - 64 * ulp))
        band = np.abs(np.abs(se.sarg(q)) - se.SARG_T) <= 64 * np.spacing(np.float32(se.SARG_T))
        assert 0 < band.mean() < 0.05
    # roll / yaw at +-pi and roll at +-pi/2: the x < 0 and |y| > |x| quadrants of atan2
    e = d["state20"][..., 7:10].reshape(-1, 3)
    assert np.sum(np.abs(e[:, 0]) > 3.1) >= 4 and np.sum(np.abs(e[:, 2]) > 3.1) >= 4
    assert np.sum(np.abs(np.abs(e[:, 0]) - np.pi / 2) < 2e-3) >= 3


@pytest.mark.parametrize("precision", PRECISIONS)
def test_f3_quaternion_norms(precision):
    d = se.f3_quat_norm(np.random.default_rng(4), se.shape("hover30"), 257, precision)
    q = d["state20"][..., 3:7].reshape(-1, 4)
    n = np.linalg.norm(q, axis=-1)
    for v in se.NORMS:
        assert np.sum(np.abs(n - v) < 1e-6) >= 30, v
    s = np.abs(se.sarg(q))
    assert np.any(s > 1.0) and np.any((s > 0.99999) & (s <= 1.0)) and np.all(np.isfinite(d["state20"][..., 7:10]))


def _gate_sign_rule(q):
    """The in-step ground-effect gate of step_substep (gpd_kernels.cuh), float64 in the kernel's order of operations."""
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    s = -2.0 * (x * z - w * y)
    rx = w * w - x * x - y * y + z * z
    ry = 2.0 * (y * z + w * x)
    gimbal = (s <= -0.99999) | (s >= 0.99999)
    upright = (rx > 0) & (np.abs(ry) * 1.7225464241988331e-16 < rx)     # atan2 does not round to +-pi/2
    return ~gimbal & (upright | ((rx == 0) & (ry == 0)))


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["gnd", "gnd_drag", "multi3_gd", "ctrl3_dw"])
def test_f4_ground_gate_true_and_false(name, precision):
    """The oracle's gate |roll|, |pitch| < pi/2 (BaseAviary.py:742) is true for >= 20 % and false for >= 20 % of the drones,
    and gimbal attitudes (sarg past the threshold) sit near the ground; the rotors of >= 20 % of the drones are at or
    below the clip height."""
    kw = se.shape(name)
    d = se.f4_ground(np.random.default_rng(5), kw, 257, precision)
    q = d["state20"][..., 3:7].reshape(-1, 4)
    e = d["state20"][..., 7:10].reshape(-1, 3)
    gate = (np.abs(e[:, 0]) < np.pi / 2) & (np.abs(e[:, 1]) < np.pi / 2)
    assert 0.2 <= gate.mean() <= 0.8, gate.mean()
    assert np.array_equal(_gate_sign_rule(q), gate)           # the FP64 kernel's shortcut agrees with the oracle's libm gate
    low = d["state20"][..., 2].reshape(-1) <= 1.5 * load_drone_params(kw["model"]).GND_EFF_H_CLIP
    assert low.mean() >= 0.2 / kw["num_drones"]
    assert np.sum(low & (np.abs(se.sarg(q)) >= 0.99999)) >= 2


F5_CONFIGS = [(L, f) for L in se.EPISODE_LENS for f in (240, 96, 60)]
F5_CTRL = {240: 30, 96: 48, 60: 30}


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("env", ["hover30", "multi3"])
@pytest.mark.parametrize("length,pyb", F5_CONFIGS)
def test_f5_flags_on_both_sides_of_each_boundary(env, length, pyb, precision):
    """The oracle's flags come out both true and false inside every boundary group, over both ctrl steps; the placed x, y
    and attitudes do not move during a step; max_counter is the last counter the reference does not truncate."""
    kw = se.shape(env, pyb_freq=pyb, ctrl_freq=F5_CTRL[pyb], episode_len_sec=length)
    S = pyb // kw["ctrl_freq"]
    mc = se.max_counter(length, pyb)
    assert mc / pyb <= length < (mc + 1) / pyb
    E = 513
    d = se.f5_episode_end(np.random.default_rng(6), kw, E, precision)
    ref = se.oracle_sim(kw, E)
    se.inject_oracle(ref, d)
    g = d["groups"]
    flags = []
    for t in range(2):
        pos0, q0 = ref.state20[..., 0:3].copy(), ref.state20[..., 3:7].copy()
        _, _, te, tr = ref.step(d["actions"][t])
        flags.append((te.copy(), tr.copy()))
        for k in ("xy0", "xy1"):
            assert np.array_equal(ref.state20[g[k], :, 0:2], pos0[g[k], :, 0:2])
        for k in ("rp0", "rp1", "xy0", "xy1", "z"):
            assert np.array_equal(ref.state20[g[k], :, 3:7], q0[g[k]])
    for k in ("xy0", "xy1", "z", "rp0", "rp1", "counter"):
        tr = flags[0][1][g[k]]
        assert tr.any() and not tr.all(), k
    te = flags[0][0][g["dist"]]
    assert te.any() and not te.all()
    c = g["counter"]                                     # max_counter - S, max_counter, max_counter + 1 (3 envs each)
    assert list(flags[0][1][c]) == [0, 0, 0, 0, 0, 0, 1, 1, 1] and list(flags[1][1][c]) == [0, 0, 0, 1, 1, 1, 1, 1, 1]
    assert np.all(d["step_counter"][c] == np.repeat([mc - S, mc, mc + 1], 3))


@pytest.mark.parametrize("name", ["pid", "vel", "one_d_pid"])
def test_f6_controller_edges(name):
    """Yaw and last yaw across +-pi saturate the yaw torque; integrators sit at and beyond their clips; inverted drones
    give sthr <= 0; PID destinations at distance exactly 1; VEL actions with a zero direction or negative speed."""
    kw = se.shape(name)
    d = se.f6_controller(np.random.default_rng(7), kw, 257, "f64")
    g = d["groups"]
    pid = orc.make_pid(__import__("gpd_b200.params", fromlist=["x"]).default_pid_params(kw["model"]))
    sat = 0
    for e in g["yaw_wrap"]:
        st = d["pid_state"][e, 0].copy()
        s = d["state20"][e, 0]
        _, _, _ = orc.pid_compute(pid, 1 / 30, s[0:3], s[3:7], s[10:13], s[0:3], pid_state=st)
        rate = (s[9] - d["pid_state"][e, 0, 8]) * 30
        sat += abs(pid.D_TOR[2] * -rate) > 3200
    assert sat >= len(g["yaw_wrap"]) - 2
    ps = d["pid_state"][g["clips"]][:, 0]
    assert np.any(np.abs(ps[:, 5]) > 1500) and np.any(np.abs(ps[:, 5]) == 1500) and np.any(np.abs(ps[:, 0]) > 2)
    inv = d["state20"][g["inverted"]][:, 0]
    m8 = np.array([orc.matrix_from_quaternion(q)[2, 2] for q in inv[:, 3:7]])
    assert np.all(m8 < 0)
    if name == "pid":
        a = d["actions"][0][g["dist1"]][:, 0].astype(np.float64)
        dist = np.linalg.norm(a - d["state20"][g["dist1"]][:, 0, 0:3], axis=-1)
        assert np.any(dist == 1.0) and np.any(dist > 1.0)
    if name == "vel":
        a = d["actions"][0][g["vel_edge"]][:, 0]
        assert np.any(np.all(a[:, :3] == 0, axis=-1)) and np.any(a[:, 3] < 0)


@pytest.mark.parametrize("name", ["hover30", "one_d_rpm", "gnd_drag", "multi3_gd", "ctrl1"])
def test_f7_value_edges(name):
    kw = se.shape(name)
    d = se.f7_values(np.random.default_rng(8), kw, 257, "f32")
    a = d["actions"]
    if kw["action_type"] == "ctrl_rpm":
        assert np.any(a < 0) and np.any(a > load_drone_params(kw["model"]).MAX_RPM)
    else:
        for v in (30, -30, 1, -1):
            assert np.any(a == v)
        assert np.any((a == 0) & np.signbit(a)) and np.any((a == 0) & ~np.signbit(a))
    bad = ~np.isfinite(d["state20"][..., :13]).all(-1)
    assert bad.sum() == 2 and set(np.nonzero(bad.any(-1))[0]) == set(d["groups"]["nonfinite"])
