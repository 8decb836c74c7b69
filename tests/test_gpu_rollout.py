"""-m gpu: open-loop rollouts (gpd_rollout).  Two identical handles start from the same state; one runs K control steps of
an action schedule in one gpd_rollout, the other K gpd_step calls on the same actions.  They must agree on the final
observation (action ring included), every per-step reward / flag / traj / terminal_kin row, the exported state, the change
in the episode statistics, and on 3 more steps afterwards (chain, counters and aux copies intact).  FP64: bit for bit (the
FP64 build has -fmad=false and both kernels share the device functions).  FP32: within the FP32 ceilings of
test_gpu_state_edges.py, flags and counters exact outside the threshold bands (the two kernels may contract FMAs
differently); the share of bit-identical envs is printed."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import state_edges as se
from helpers import default_targets
from gpd_b200 import _lib
from gpd_b200.params import load_drone_params
from gpd_b200.sim import BatchedSim
from gpd_b200.utils.enums import DroneModel

pytestmark = pytest.mark.gpu

# FP32 ceilings of test_gpu_state_edges.py (F32_CEIL) per observation / state quantity
F32_KIN_ATOL = np.array([1e-4] * 9 + [2e-3] * 3)
F32_ATOL = {12: F32_KIN_ATOL,                                                        # obs kin / traj / terminal_kin
            20: np.array([1e-4] * 13 + [2e-3] * 3 + [0.05] * 4),                     # state20 (RPM ~1e4: 5e-6 relative)
            3: np.full(3, 2e-3), 9: np.full(9, 1e-4)}                                # rpy_rates, pid_state
SHORT_EP = 0.3          # 72 substeps at 240 Hz: several auto-resets fall inside a 40-step rollout


def kwargs(name, **over):
    return se.shape(name, **over)


CTRL_VEL = dict(env_kind="ctrl", action_type="ctrl_vel", num_drones=1, pyb_freq=240, ctrl_freq=48, physics_flags=0)
CTRL64_DW = dict(env_kind="ctrl", action_type="ctrl_rpm", num_drones=64, pyb_freq=240, ctrl_freq=48, physics_flags=4)
MULTI2_GD = dict(env_kind="multihover", action_type="rpm", num_drones=2, pyb_freq=240, ctrl_freq=30, physics_flags=3)


def make(kw, E, precision, auto_reset=True, ep_len=SHORT_EP, chaining=False):
    s = BatchedSim(load_drone_params(kw["model"]), E, kw["num_drones"], env_kind=kw["env_kind"],
                   action_type=kw["action_type"], pyb_freq=kw["pyb_freq"], ctrl_freq=kw["ctrl_freq"],
                   physics_flags=kw["physics_flags"], precision=precision, auto_reset=auto_reset,
                   target_pos=default_targets(kw), episode_len_sec=ep_len)
    if chaining:
        s.set_step_chaining(True)
    return s


def bits(x):
    x = x.contiguous()
    return x.view({8: torch.int64, 4: torch.int32, 2: torch.int16, 1: torch.uint8}[x.element_size()])


def schedule(rng, s, K, scale=0.3):
    """Actions (K, E, N, A) in the sim's action dtype: small RPM offsets, targets near the drone, controller inputs."""
    E, N, A = s.E, s.N, s.A
    if s.action_type == "ctrl_rpm":
        hover = load_drone_params(DroneModel.CF2X).HOVER_RPM
        a = hover * (1 + 0.05 * scale * rng.uniform(-1, 1, (K, E, N, A)))
    elif s.action_type == "pid":
        a = rng.uniform(-0.5, 0.5, (K, E, N, A)) + np.array([0, 0, 0.5])
    else:
        a = scale * rng.uniform(-1, 1, (K, E, N, A))
    return torch.as_tensor(a).to(device="cuda", dtype=s.act_dtype).contiguous()


class Result:
    def __init__(self, obs, rew, te, tr, traj, tkin):
        self.obs, self.rew, self.te, self.tr, self.traj, self.tkin = obs, rew, te, tr, traj, tkin


def run_rollout(s, acts):
    K = acts.shape[0]
    tk = s.auto_reset and not s.is_ctrl
    out = s.alloc_rollout_outputs(K, traj=True, terminal_kin=tk)
    if tk:
        out["terminal_kin"].fill_(float("nan"))        # rows of steps where an env did not finish stay untouched
    r = s.rollout(acts, traj=True, terminal_kin=tk, out=out)
    return Result(r[0].clone(), r[1], r[2], r[3], r[4], r[5] if tk else None)


def run_steps(s, acts):
    K = acts.shape[0]
    rew, te, tr, traj, tkin = [], [], [], [], []
    for k in range(K):
        if s.terminal_kin is not None:
            s.terminal_kin.fill_(float("nan"))
        obs, r, a, b = s.step(acts[k])
        rew.append(r.clone()); te.append(a.clone()); tr.append(b.clone())
        traj.append(obs.clone() if s.is_ctrl else obs[..., :12].clone())
        if s.terminal_kin is not None:
            tkin.append(s.terminal_kin.clone())
    return Result(obs.clone(), torch.stack(rew), torch.stack(te), torch.stack(tr), torch.stack(traj),
                  torch.stack(tkin) if tkin else None)


def flag_band(s, kin):
    """Envs whose step is within 1e-5 of a Hover / MultiHover threshold (FP32: the two kernels may round across it)."""
    if s.is_ctrl:
        return np.zeros(kin.shape[:-2], bool)
    lim = 1.5 if s.env_kind == "hover" else 2.0
    near = lambda v, c: np.abs(v - c) < 1e-5
    b = (near(np.abs(kin[..., 0]), lim) | near(np.abs(kin[..., 1]), lim) | near(kin[..., 2], 2.0) |
         near(np.abs(kin[..., 3]), .4) | near(np.abs(kin[..., 4]), .4)).any(-1)
    return b


class Checker:
    def __init__(self, s, precision):
        self.s, self.f64 = s, precision == "f64"
        self.skip = np.zeros(s.E, bool)         # FP32: envs that crossed a threshold band (their episodes may split differently)
        self.n_bit, self.n_tot = 0, 0

    def kin(self, what, x, y, per_env_axis=1):
        """x, y: (..., E, N, C) kin / state rows."""
        if self.f64:
            assert torch.equal(bits(x), bits(y)), what
            return
        xa, ya = x.double().cpu().numpy(), y.double().cpu().numpy()
        C_ = xa.shape[-1]
        atol = F32_ATOL[C_]
        d = np.abs(xa - ya)
        if C_ in (12, 20):                       # angles: +-pi wrap
            cols = [3, 4, 5] if C_ == 12 else [7, 8, 9]
            d[..., cols] = np.minimum(d[..., cols], np.abs(2 * np.pi - d[..., cols]))
        ok = (d <= atol) | (np.isnan(xa) & np.isnan(ya))
        env_ok = ok.reshape(ok.shape[:-2] + (-1,)).all(-1)
        env_ok = env_ok if env_ok.ndim == 1 else env_ok.all(0)
        bad = ~env_ok & ~self.skip
        assert not bad.any(), f"{what}: {int(bad.sum())} envs beyond the FP32 ceilings, e.g. env {int(np.argmax(bad))}: " \
                              f"max diff {np.nanmax(d)}"
        same = (xa.view(np.uint64) == ya.view(np.uint64)).reshape(xa.shape[:-2] + (-1,)).all(-1)
        same = same if same.ndim == 1 else same.all(0)
        self.n_bit += int(same.sum()); self.n_tot += same.size

    def flags(self, what, x, y, ref_kin=None):
        """x, y: (K, E) per-step outputs; ref_kin (K, E, N, 12) of the step path marks FP32 threshold bands."""
        if self.f64:
            assert torch.equal(bits(x), bits(y)), what
            return
        xa, ya = x.cpu().numpy(), y.cpu().numpy()
        if ref_kin is not None:
            for k in range(xa.shape[0]):
                self.skip |= flag_band(self.s, ref_kin[k])
                bad = (xa[k] != ya[k]) if xa.dtype != np.float32 else ~np.isclose(xa[k], ya[k], rtol=1e-4, atol=1e-4)
                bad &= ~self.skip
                assert not bad.any(), f"{what}[{k}]: envs {np.nonzero(bad)[0][:8]}"
        else:
            bad = ((xa != ya) if xa.dtype != np.float32 else ~np.isclose(xa, ya, rtol=1e-4, atol=1e-4))
            bad = bad.any(0) & ~self.skip if bad.ndim == 2 else bad & ~self.skip
            assert not bad.any(), what

    def report(self, tag):
        if not self.f64 and self.n_tot:
            print(f"[rollout] {tag}: {100.0 * self.n_bit / self.n_tot:.1f} % of the compared env rows bit-identical "
                  f"({int(self.skip.sum())} of {self.s.E} envs in an FP32 threshold band)")


def compare(ra, rb, a, b, chk):
    ref_kin = None
    if not a.is_ctrl:                           # the step path's kin before any auto-reset marks the FP32 bands
        ref_kin = rb.traj.cpu().numpy()
        if rb.tkin is not None:
            tk = rb.tkin.cpu().numpy()
            fin = ~np.isnan(tk[..., 0])
            ref_kin[fin] = tk[fin]
    chk.flags("terminated", ra.te, rb.te, ref_kin)
    chk.flags("truncated", ra.tr, rb.tr)
    chk.flags("reward", ra.rew, rb.rew)
    chk.kin("traj", ra.traj, rb.traj)
    if ra.tkin is not None:
        if chk.f64:
            assert torch.equal(bits(ra.tkin), bits(rb.tkin)), "terminal_kin"
        else:
            fin_a, fin_b = ~torch.isnan(ra.tkin[..., 0]), ~torch.isnan(rb.tkin[..., 0])
            diff = (fin_a != fin_b).any(-1).any(0).cpu().numpy() & ~chk.skip
            assert not diff.any(), "terminal_kin rows written at different steps"
            chk.kin("terminal_kin", torch.nan_to_num(ra.tkin, nan=0.0), torch.nan_to_num(rb.tkin, nan=0.0))
    if a.is_ctrl:
        chk.kin("obs", ra.obs, rb.obs)
    else:
        chk.kin("obs kin", ra.obs[..., :12], rb.obs[..., :12])
        assert torch.equal(bits(ra.obs[..., 12:]), bits(rb.obs[..., 12:])), "action ring"
    sa, sb = a.get_state(), b.get_state()
    chk.kin("state20", sa[0], sb[0])
    chk.kin("rpy_rates", sa[1], sb[1])
    chk.kin("pid_state", sa[2], sb[2])
    cnt_a, cnt_b = sa[3].cpu().numpy(), sb[3].cpu().numpy()
    assert np.array_equal(cnt_a[~chk.skip], cnt_b[~chk.skip]), "step counters"


def compare_stats(a, b, chk):
    if not a.auto_reset:
        return
    x, y = a.episode_stats(clear=True), b.episode_stats(clear=True)
    if chk.skip.any():
        return                                 # FP32 envs in a threshold band may end episodes at different steps
    for j in (0, 2, 6, 7):                      # episodes, lengths, env-steps, terminated: exact
        assert x[j] == y[j], (j, x, y)
    if x[0] > 0:
        assert x[4] == y[4] and x[5] == y[5], (x, y)          # min / max
        for j in (1, 3):
            assert abs(x[j] - y[j]) <= 1e-6 * max(1.0, abs(y[j])), (j, x, y)


def drive(kw, E, precision, K, auto_reset=True, seed=0, warm=2, per_env=False, family=None, ep_len=SHORT_EP, tag=""):
    rng = np.random.default_rng(seed)
    a, b = make(kw, E, precision, auto_reset, ep_len), make(kw, E, precision, auto_reset, ep_len)
    if per_env:
        N = kw["num_drones"]
        xyz = np.stack([rng.uniform(-.5, .5, (E, N)), rng.uniform(-.5, .5, (E, N)), rng.uniform(.3, 1.2, (E, N))], -1)
        rpy = rng.uniform(-.1, .1, (E, N, 3))
        for s in (a, b):
            s.set_init_poses(xyz, rpy)
            if not s.is_ctrl:
                s.set_targets(xyz + np.array([0, 0, 0.3]))
            s.reset()
    if family is not None:
        fam = se.FAMILIES[family](rng, kw, E, precision)
        rdt = a.real
        dev = lambda v, dt=rdt: torch.as_tensor(np.ascontiguousarray(v)).to(device="cuda", dtype=dt)
        for s in (a, b):
            s.set_state(dev(fam["state20"]), dev(fam["rpy_rates"]), dev(fam["pid_state"]), dev(fam["step_counter"], torch.int32))
    chk = Checker(a, precision)
    for _ in range(warm):                       # a non-zero ring and a previous observation
        w = schedule(rng, a, 1)[0]
        a.step(w); b.step(w)
    if auto_reset:
        a.episode_stats(clear=True); b.episode_stats(clear=True)
    acts = schedule(rng, a, K)
    if family is not None:                      # the family's own first actions (e.g. +-30 RPM offsets, NaN / Inf states)
        fa = torch.as_tensor(fam["actions"][:min(2, K)]).to(device="cuda", dtype=a.act_dtype)
        acts[:fa.shape[0]] = fa
    ra, rb = run_rollout(a, acts), run_steps(b, acts)
    torch.cuda.synchronize()
    compare(ra, rb, a, b, chk)
    compare_stats(a, b, chk)
    after = schedule(rng, a, 3)                 # the chain, counters and aux copies are intact after the rollout
    rb2 = run_steps(b, after)
    ra2 = run_steps(a, after)
    compare(ra2, rb2, a, b, chk)
    chk.report(tag or f"{kw['env_kind']} {kw['action_type']} {precision} E={E} K={K}")
    return a, b


# ---- action types, physics, drone models ---------------------------------------------------------------------------
ACTION_CASES = ["hover30", "one_d_rpm", "pid", "vel", "one_d_pid", "ctrl1"]


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ACTION_CASES)
def test_rollout_action_types(name, precision):
    drive(kwargs(name), 37, precision, vel_steps(name == "vel", precision))


def vel_steps(vel, precision):
    """Velocity commands in FP32: 8 steps.  Over 40 steps of random velocity targets the controller amplifies the two
    kernels' FP32 contraction differences beyond the ceilings (measured on a B200: 0.06 / 0.12 in 3 of 37 envs); FP64 runs
    the full 40 steps bit for bit."""
    return 8 if vel and precision == "f32" else 40


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_rollout_ctrl_vel(precision):
    drive(dict(CTRL_VEL, model=DroneModel.CF2X), 37, precision, vel_steps(True, precision))


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("shape", ["multi2_gd", "multi3", "ctrl64_dw"])
def test_rollout_physics(shape, precision):
    kw = {"multi2_gd": dict(MULTI2_GD, model=DroneModel.CF2X), "multi3": kwargs("multi3"),
          "ctrl64_dw": dict(CTRL64_DW, model=DroneModel.CF2X)}[shape]
    if shape == "ctrl64_dw" and precision == "f32":
        pytest.skip("FP32 downwash: the stiff field exceeds the FP32 ceilings within a window (DESIGN.md); FP64 is bit-exact")
    drive(kw, 37 if shape != "ctrl64_dw" else 9, precision, 40, ep_len=SHORT_EP if shape != "ctrl64_dw" else 8.0)


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("model", [DroneModel.CF2P, DroneModel.RACE])
def test_rollout_drone_models(model, precision):
    drive(kwargs("hover30", model=model), 37, precision, 40)


# ---- K against the ring length, ragged env counts, auto-reset, per-env poses ---------------------------------------------
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("K", [1, 14, 15, 16, 40])      # B = 15 at 30 Hz
def test_rollout_ring_lengths(K, precision):
    drive(kwargs("hover30"), 37, precision, K)


@pytest.mark.parametrize("K", [1, 5, 6, 7])             # B = 6 at 12 Hz; A = 1 and A = 3 rows (scalar ring copies)
def test_rollout_ring_narrow_actions(K):
    drive(kwargs("one_d_rpm", ctrl_freq=12), 37, "f64", K)
    drive(kwargs("pid", ctrl_freq=12), 37, "f64", K)


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("E", [1, 37, 4097])
def test_rollout_ragged_env_counts(E, precision):
    drive(kwargs("hover30"), E, precision, 20)
    drive(kwargs("multi3"), E, precision, 20)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_rollout_without_auto_reset_and_without_obs_prev(precision):
    drive(kwargs("hover30"), 37, precision, 20, auto_reset=False)
    drive(kwargs("hover30"), 37, precision, 3, auto_reset=False, warm=0)     # ring from the reset observation
    drive(kwargs("pid"), 37, precision, 20, auto_reset=False)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_rollout_per_env_poses_and_targets(precision):
    drive(kwargs("hover30"), 37, precision, 40, per_env=True)
    drive(kwargs("multi3"), 37, precision, 40, per_env=True)


@pytest.mark.parametrize("fam", ["F1", "F2", "F7"])
@pytest.mark.parametrize("name", ["hover30", "multi3"])
def test_rollout_from_edge_states_f64(fam, name):
    """Injected off-nominal starts: fast spins, any attitude, NaN / Inf values.  FP64 bit for bit (NaN / Inf bits too)."""
    drive(kwargs(name), 513, "f64", 8, family=fam, warm=0, ep_len=8.0)


# ---- interaction with the rest of the library ------------------------------------------------------------------------
def test_rollout_chained_state_on_off_and_chained_steps(monkeypatch):
    """Lean FP32 (C2-like tiles): chained gpd_step -> gpd_rollout -> chained gpd_step on one stream, with the chained state
    (GPD_STATE_IN_OBS) on and off: the same bits.  Against plain unchained steps: within the FP32 ceilings.  Nothing else
    runs on the stream between chained steps (the chaining contract)."""
    kw = kwargs("hover30")
    E = 4 * 148 * 64
    rng = np.random.default_rng(3)
    sims = {}
    for on in (1, 0):
        monkeypatch.setenv("GPD_STATE_IN_OBS", str(on))
        sims[on] = make(kw, E, "f32", chaining=True)
    monkeypatch.delenv("GPD_STATE_IN_OBS")
    ref = make(kw, E, "f32")
    pre, acts, post = schedule(rng, ref, 4), schedule(rng, ref, 24), schedule(rng, ref, 4)
    torch.cuda.synchronize()
    outs = {}
    for on, s in sims.items():
        K = acts.shape[0]
        out = s.alloc_rollout_outputs(K, traj=True, terminal_kin=True)
        out["terminal_kin"].fill_(float("nan"))
        torch.cuda.synchronize()
        for k in range(4):
            s.step(pre[k])
        s.rollout(acts, traj=True, terminal_kin=True, out=out)
        for k in range(4):
            obs = s.step(post[k])[0]
        outs[on] = (out, obs.clone(), s.reward.clone(), s.get_state())
    for k in range(4):
        ref.step(pre[k])
    rr = run_steps(ref, acts)
    for k in range(4):
        ref_obs = ref.step(post[k])[0]
    torch.cuda.synchronize()
    (o1, obs1, rew1, st1), (o0, obs0, rew0, st0) = outs[1], outs[0]
    for f in o1:
        assert torch.equal(bits(o1[f]), bits(o0[f])), f
    assert torch.equal(bits(obs1), bits(obs0)) and torch.equal(bits(rew1), bits(rew0))
    for x, y in zip(st1, st0):
        assert torch.equal(bits(x), bits(y))
    chk = Checker(sims[1], "f32")
    chk.flags("terminated", o1["terminated"], rr.te, rr.traj.cpu().numpy())
    chk.flags("truncated", o1["truncated"], rr.tr)
    chk.kin("traj", o1["traj"], rr.traj)
    chk.kin("obs after the chained steps", obs1[..., :12], ref_obs[..., :12])
    assert torch.equal(bits(obs1[..., 12:]), bits(ref_obs[..., 12:]))
    chk.report("chained C2-like")


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_rollout_masked_reset_between_rollouts(precision):
    kw = kwargs("hover30")
    E = 37
    rng = np.random.default_rng(5)
    a, b = make(kw, E, precision), make(kw, E, precision)
    chk = Checker(a, precision)
    for it in range(2):
        acts = schedule(rng, a, 12)
        ra, rb = run_rollout(a, acts), run_steps(b, acts)
        compare(ra, rb, a, b, chk)
        mask = torch.as_tensor(rng.random(E) < 0.4, device="cuda")
        oa, ob = a.reset(mask), b.reset(mask)
        chk.kin("obs after masked reset", oa[..., :12], ob[..., :12])
        assert torch.equal(bits(oa[..., 12:]), bits(ob[..., 12:]))
    chk.report("masked reset")


def test_rollout_then_host_mirror_step():
    """A host-mirror step after a rollout: the mirror rebuilds itself from the rollout's observation."""
    kw = kwargs("hover30")
    E = 37
    rng = np.random.default_rng(6)
    a, b = make(kw, E, "f64"), make(kw, E, "f64")
    w = schedule(rng, a, 1)[0].cpu().numpy()
    a.step_host(w); b.step_host(w)                        # both mirrors attached and in sync
    acts = schedule(rng, a, 10)
    a.rollout(acts)
    for k in range(10):
        b.step(acts[k])
    w = schedule(rng, a, 1)[0].cpu().numpy()
    oa, ra = a.step_host(w)[:2]
    ob, rb = b.step_host(w)[:2]
    assert np.array_equal(np.asarray(oa).view(np.uint32), np.asarray(ob).view(np.uint32))
    assert np.array_equal(ra, rb)
    torch.cuda.synchronize()
    assert torch.equal(bits(a.obs), bits(b.obs))


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_rollout_graph_capture_replay(precision):
    """A rollout captured in a CUDA graph (caller-owned outputs: nothing allocated) and replayed equals the eager run."""
    kw = kwargs("pid")
    E, K = 37, 16
    rng = np.random.default_rng(7)
    g_sim, e_sim = make(kw, E, precision), make(kw, E, precision)
    w = schedule(rng, g_sim, 1)[0]
    g_sim.step(w); e_sim.step(w)
    acts = schedule(rng, g_sim, K)
    out = g_sim.alloc_rollout_outputs(K, traj=True, terminal_kin=True)
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(st):
        with torch.cuda.graph(graph, stream=st):
            g_obs = g_sim.rollout(acts, traj=True, terminal_kin=True, out=out)[0]
    out["terminal_kin"].fill_(float("nan"))
    graph.replay()
    re = run_rollout(e_sim, acts)
    torch.cuda.synchronize()
    assert torch.equal(bits(g_obs), bits(re.obs))
    for x, y in ((out["reward"], re.rew), (out["terminated"], re.te), (out["truncated"], re.tr), (out["traj"], re.traj),
                 (out["terminal_kin"], re.tkin)):
        assert torch.equal(bits(x), bits(y))
    for x, y in zip(g_sim.get_state(), e_sim.get_state()):
        assert torch.equal(bits(x), bits(y))


def test_rollout_invalid_arguments():
    kw = kwargs("hover30")
    s = make(kw, 37, "f32")
    L = _lib.load()
    K = 4
    acts = torch.zeros((K, 37, 1, 4), device="cuda")
    obs = torch.zeros((37, 1, s.W), device="cuda")
    prev = s.obs
    big = torch.zeros(acts.numel() + 4, device="cuda")
    big_obs = torch.zeros(obs.numel() + 4, device="cuda")
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cases = [
        (0, p(acts), p(prev), p(obs)),                 # n_steps < 1
        (-3, p(acts), p(prev), p(obs)),
        (K, None, p(prev), p(obs)),                    # null actions
        (K, p(acts), p(prev), None),                   # null obs_out
        (K, p(acts), p(obs), p(obs)),                  # obs_out aliases obs_prev
        (K, p(acts), p(prev), p(acts)),                # obs_out aliases actions
        (K, p(big, 4), p(prev), p(obs)),               # misaligned actions
        (K, p(acts), p(prev), p(big_obs, 8)),          # misaligned obs_out
    ]
    for n, ac, pr, ob in cases:
        rc = L.gpd_rollout(s.h, n, ac, pr, ob, None, None, None, None, None, stream)
        assert rc == -1, (n, rc)
    rc = L.gpd_rollout(s.h, K, p(acts), p(prev), p(obs), None, None, None, p(big_obs, 4), None, stream)
    assert rc == -1                                    # misaligned traj
    assert L.gpd_rollout(None, K, p(acts), p(prev), p(obs), None, None, None, None, None, stream) == -1
    assert L.gpd_rollout(s.h, K, p(acts), p(prev), p(obs), None, None, None, None, None, stream) == 0
    torch.cuda.synchronize()


def test_base_aviary_rollout():
    from gpd_b200.envs.HoverAviary import HoverAviary
    env_a, env_b = HoverAviary(num_envs=37), HoverAviary(num_envs=37)
    rng = np.random.default_rng(8)
    acts = torch.as_tensor(rng.uniform(-.3, .3, (12, 37, 1, 4)), dtype=torch.float32, device="cuda")
    obs, rew, te, tr, info = env_a.rollout(acts, return_traj=True)
    assert rew.shape == (12, 37) and te.dtype == torch.bool and tr.dtype == torch.bool
    assert info["traj"].shape == (12, 37, 1, 12)
    for k in range(12):
        ob = env_b.step(acts[k])[0]
    torch.cuda.synchronize()
    assert torch.allclose(obs[..., :12], ob[..., :12], atol=1e-4)
    assert torch.equal(obs[..., 12:], ob[..., 12:])
