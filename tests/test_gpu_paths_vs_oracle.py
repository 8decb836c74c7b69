"""-m gpu: every size- and layout-selected data path of the step, in the launch pattern that selects it, against the CPU
oracle on every env of every set.

gpd_create and step_impl pick a step's data path from the env count, the buffer alignment and the launch pattern: bulk or
per-thread kernel, 64- or 128-env tiles, one or two tiles per CTA, per-tile sequencing and PDL, the chained state
(position and velocity read from the previous observation row), the TMA ring copy and its whole-sector split, the
shared-memory fallback, plain stores for misaligned outputs.  Each case below runs in the pattern that reaches its path
(chained rotations of several handles from one replayed CUDA graph, or eager steps) and is compared with the oracle at
window ends (tests/paths_harness.py): the oracle is teacher-forced from the GPU's exported state at each window start and
stepped over the same actions, so no state is read between the checked steps.  At every window end: state and rpy_rates,
the whole observation (its action ring bit for bit), the last step's reward and flags, terminal_kin of the envs that ended,
the counters and the change in episode_stats.

Bounds: FP64 the fuzz tests' (1e-9 on state, flags exact).  FP32 the ceilings of test_gpu_state_edges.py (1e-4 on pos /
vel / quat / rpy, 2e-3 on rates / ang_v) with its exemption bands, each under 5 % of a case; an env whose flag decision
falls in a band drops out until the next window.

Witnesses: the create-time choices are read from the GPD_DEBUG_LAYOUT line, the per-launch ones (kernel, grid) from one
extra window run under torch.profiler after the checked windows; a retune that moves a case off its path fails here.
Runtime-selected variants of one kernel instance (GPD_TMA, GPD_TMA_EDGE) must give the same bits as the default.
"""
import json
import os
import re
import zlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import state_edges as se
from helpers import S_ANGV, S_POS, S_QUAT, S_RPM, S_RPY, S_VEL, angle_err, default_targets, quat_err, rel_err
from paths_harness import Track, load_oracle, step_window
from test_gpu_state_edges import F32_CEIL, F64_TOL, _flag_band, _rpy_band
from gpd_b200.params import load_drone_params

pytestmark = pytest.mark.gpu

LAYOUT = re.compile(r"\[gpd\] (\d+) CTAs/SM, ([\d.]+) waves: tile_dep (\d), pdl (\d), bulk path (\d), tile (\d+), tiles (\d+), "
                    r"tma (\d), tma_edge (\d), bulk_tpc (\d), state_in_obs (\d)")
LAYOUT_KEYS = ("tile_dep", "pdl", "bulk", "tile", "tiles", "tma", "tma_edge", "bulk_tpc", "state_in_obs")


def bits(x):
    x = x.contiguous()
    return x.view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))


def _shape(env_kind, act, N, pyb, ctrl, flags, **over):
    kw = dict(env_kind=env_kind, action_type=act, num_drones=N, pyb_freq=pyb, ctrl_freq=ctrl, physics_flags=flags)
    kw = dict(kw, model=se.shape("hover30")["model"], init_xyz=None, init_rpy=None, episode_len_sec=8.0)
    kw.update(over)
    return kw


def _spaced_heights(E, N, seed):
    """test_cuda_full_size_properties_other_configs' C4 FP32 poses: every drone of an env at its own height, 0.045 m apart."""
    rng = np.random.default_rng(seed)
    z = 0.2 + 0.045 * np.argsort(rng.random((E, N)), axis=1)[..., None].astype(np.float64)
    return np.concatenate([rng.uniform(-2, 2, (E, N, 2)), z], -1), np.zeros((E, N, 3))


class Case:
    """One data path: the env, its size and precision, the launch pattern and what the witnesses must show.
    pattern "graph": `steps` steps rotating over `nsets` chained handles captured once, `replays` replays per window.
    pattern "eager": `steps` eager steps per handle per window (`align` cycles the step over misaligned buffers)."""

    def __init__(self, kw, E, precision, nsets=1, pattern="graph", steps=2, replays=1, windows=2, env=None, layout=None,
                 kernel=None, grids=None, variants=(), spaced=False, align=False):
        self.kw, self.E, self.precision, self.nsets = kw, E, precision, nsets
        self.pattern, self.steps, self.replays, self.windows = pattern, steps, replays, windows
        self.env, self.layout, self.kernel, self.grids = dict(env or {}), dict(layout or {}), kernel, grids
        self.variants, self.spaced, self.align = variants, spaced, align
        self.ctrl = kw["env_kind"] == "ctrl"
        self.auto_reset = not self.ctrl
        # FP32 downwash is held to the oracle by test_gpu_parity.py at its own documented bound (a stiff field: rounding
        # differences grow ~10x per 5 ctrl steps, beyond the FP32 ceilings used here, as in test_gpu_state_edges.py); its
        # cases here check the path witnesses and the bit-identity of the runtime variants only
        self.dw32 = precision == "f32" and bool(kw["physics_flags"] & 4)


HOVER = _shape("hover", "rpm", 1, 240, 30, 0)
# bulk kernel names: step_kernel_bulk<R, KIND, MULTI>, KIND 0 force models, 1 lean, 2 DSLPID; per-thread kernel
# step_kernel<R, KIND, MULTI, VEC>
CASES = {
    # the benchmark: 8 x 65,536 lean FP32 envs, chained rotation, 16-step graph
    "c2_f32": Case(HOVER, 65536, "f32", nsets=8, steps=16, replays=2, windows=3,
                   layout=dict(bulk=1, tile=128, tiles=512, bulk_tpc=2, state_in_obs=1, tile_dep=1, pdl=1),
                   kernel="step_kernel_bulk<float, 1, false>", grids=(256, 512)),
    "c2_f64": Case(HOVER, 65536, "f64", nsets=8, steps=16, replays=2, windows=2,
                   layout=dict(bulk=1, tile=128, tiles=512, bulk_tpc=1, state_in_obs=0, tile_dep=1),
                   kernel="step_kernel_bulk<double, 1, false>", grids=(512,)),
    # tile-size edges of the lean FP32 bulk kernel (37,888 <= D <= 262,144: 128-env tiles), ragged and odd tile counts
    "tiles_37887": Case(HOVER, 37887, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=64, tiles=592, bulk_tpc=2, state_in_obs=1),
                        kernel="step_kernel_bulk<float, 1, false>", grids=(296, 592)),
    "tiles_37888": Case(HOVER, 37888, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=128, tiles=296, bulk_tpc=1, state_in_obs=1),
                        kernel="step_kernel_bulk<float, 1, false>", grids=(296,)),
    "tiles_37933": Case(HOVER, 37933, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=128, tiles=297, bulk_tpc=1, state_in_obs=1),
                        kernel="step_kernel_bulk<float, 1, false>", grids=(297,)),
    "tiles_65581": Case(HOVER, 65581, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=128, tiles=513, bulk_tpc=2, state_in_obs=1),
                        kernel="step_kernel_bulk<float, 1, false>", grids=(257, 513)),
    "tiles_262144": Case(HOVER, 262144, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=128, tiles=2048, bulk_tpc=2, state_in_obs=1),
                         kernel="step_kernel_bulk<float, 1, false>", grids=(1024, 2048)),
    "tiles_262145": Case(HOVER, 262145, "f32", nsets=3, steps=6, layout=dict(bulk=1, tile=64, tiles=4097, bulk_tpc=2, state_in_obs=1),
                         kernel="step_kernel_bulk<float, 1, false>", grids=(2049, 4097)),
    # many waves: no per-tile sequencing, no PDL, chained state still on
    "waves_1m": Case(HOVER, 1048576, "f32", nsets=2, steps=4, layout=dict(bulk=1, tile=64, tiles=16384, tile_dep=0, pdl=0, state_in_obs=1),
                     kernel="step_kernel_bulk<float, 1, false>", grids=(16384,)),
    # C3: MultiHover x2 GND+DRAG FP64 on the multi-drone bulk kernel
    "c3_f64": Case(_shape("multihover", "rpm", 2, 240, 30, 3), 32768, "f64", nsets=6, steps=12,
                   layout=dict(bulk=1, state_in_obs=0), kernel="step_kernel_bulk<double, 0, true>"),
    # C4: Ctrl x64 with downwash on gpd::step_kernel
    "c4_f32": Case(_shape("ctrl", "ctrl_rpm", 64, 240, 48, 4), 4096, "f32", nsets=4, steps=8, spaced=True,
                   layout=dict(bulk=0, tma=0), kernel="step_kernel<float, 0, true, false>"),
    "c4_f64": Case(_shape("ctrl", "ctrl_rpm", 64, 240, 48, 4), 4096, "f64", nsets=4, steps=8, spaced=True,
                   layout=dict(bulk=0, tma=0), kernel="step_kernel<double, 0, true, false>"),
    # C5: 2 M HoverAviary PID envs, row-sliding bulk kernel, many waves
    "c5_f32": Case(_shape("hover", "pid", 1, 240, 48, 0), 2097152, "f32", nsets=1, steps=6, windows=1,
                   layout=dict(bulk=1, tile_dep=0, state_in_obs=0), kernel="step_kernel_bulk<float, 2, false>"),
    # whole-sector TMA split (D >= 65,536 with 32-byte ring rows): MultiHover x2 with downwash runs gpd::step_kernel
    "edge_mh_32768_f32": Case(_shape("multihover", "rpm", 2, 240, 30, 4), 32768, "f32", nsets=2, steps=4,
                              layout=dict(bulk=0, tma=1, tma_edge=1), kernel="step_kernel<float, 0, true, true>",
                              variants=({"GPD_TMA_EDGE": "0"}, {"GPD_TMA": "0"})),
    "edge_mh_32767_f32": Case(_shape("multihover", "rpm", 2, 240, 30, 4), 32767, "f32", nsets=2, steps=4,
                              layout=dict(bulk=0, tma=1, tma_edge=0), kernel="step_kernel<float, 0, true, true>",
                              variants=({"GPD_TMA_EDGE": "1"},)),
    "edge_mh_32768_f64": Case(_shape("multihover", "rpm", 2, 240, 30, 4), 32768, "f64", nsets=2, steps=4,
                              layout=dict(bulk=0, tma=1, tma_edge=1), kernel="step_kernel<double, 0, true, true>",
                              variants=({"GPD_TMA_EDGE": "0"}, {"GPD_TMA": "0"})),
    "edge_mh_32767_f64": Case(_shape("multihover", "rpm", 2, 240, 30, 4), 32767, "f64", nsets=2, steps=4, pattern="eager",
                              layout=dict(bulk=0, tma=1, tma_edge=0), kernel="step_kernel<double, 0, true, true>"),
    "edge_hover_65536": Case(HOVER, 65536, "f32", pattern="eager", steps=4, env={"GPD_BULK": "0"},
                             layout=dict(bulk=0, tma=1, tma_edge=1), kernel="step_kernel<float, 1, false, true>",
                             variants=({"GPD_TMA_EDGE": "0"}, {"GPD_TMA": "0"})),
    "edge_hover_1000_forced": Case(HOVER, 1000, "f32", pattern="eager", steps=4, env={"GPD_BULK": "0", "GPD_TMA_EDGE": "1"},
                                   layout=dict(bulk=0, tma=1, tma_edge=1), kernel="step_kernel<float, 1, false, true>",
                                   variants=({"GPD_TMA_EDGE": "0"}, {"GPD_TMA": "0"})),
    # A < 4: the whole old ring through TMA, written out shifted by the copy warp
    "ring_one_d_rpm_240": Case(_shape("hover", "one_d_rpm", 1, 240, 240, 0), 20000, "f32", pattern="eager", steps=4,
                               layout=dict(bulk=0, tma=1), kernel="step_kernel<float, 1, false, false>", variants=({"GPD_TMA": "0"},)),
    "ring_one_d_pid_240": Case(_shape("hover", "one_d_pid", 1, 240, 240, 0), 20000, "f32", pattern="eager", steps=4,
                               layout=dict(bulk=0, tma=1), kernel="step_kernel<float, 2, false, false>", variants=({"GPD_TMA": "0"},)),
    "ring_pid_48": Case(_shape("hover", "pid", 1, 240, 48, 0), 20000, "f32", pattern="eager", steps=4, env={"GPD_BULK": "0"},
                        layout=dict(bulk=0, tma=1), kernel="step_kernel<float, 2, false, false>", variants=({"GPD_TMA": "0"},)),
    # a history tile beyond the shared-memory limit: the register-copy path
    "smem_fallback_mh256": Case(_shape("multihover", "rpm", 256, 240, 120, 0), 48, "f32", pattern="eager", steps=4,
                                layout=dict(bulk=0, tma=0), kernel="step_kernel<float, 1, true, true>"),
    # misaligned buffers: per-thread kernel for that step (after a state sync on a chained-state handle), plain output stores
    "align_f32": Case(HOVER, 20000, "f32", pattern="eager", steps=4, align=True, layout=dict(bulk=1, state_in_obs=1)),
    "align_f64": Case(HOVER, 20000, "f64", pattern="eager", steps=4, align=True, layout=dict(bulk=1, state_in_obs=0)),
}


# ---------------------------------------------------------------------------------------------------------------------
def _make(c, capfd, monkeypatch, extra_env=None):
    from gpd_b200.sim import BatchedSim
    kw = c.kw
    env = dict(c.env, **(extra_env or {}))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("GPD_DEBUG_LAYOUT", "1")
    capfd.readouterr()
    xyz = rpy = None
    if c.spaced:
        xyz, rpy = _spaced_heights(c.E, kw["num_drones"], 5)
    sims = [BatchedSim(load_drone_params(kw["model"]), c.E, kw["num_drones"], env_kind=kw["env_kind"],
                       action_type=kw["action_type"], pyb_freq=kw["pyb_freq"], ctrl_freq=kw["ctrl_freq"],
                       physics_flags=kw["physics_flags"], precision=c.precision, auto_reset=c.auto_reset,
                       target_pos=default_targets(kw), episode_len_sec=kw["episode_len_sec"], init_xyz=xyz, init_rpy=rpy)
            for _ in range(c.nsets)]
    err = capfd.readouterr().err
    for k in list(env) + ["GPD_DEBUG_LAYOUT"]:
        monkeypatch.delenv(k, raising=False)
    lines = [m.groups() for m in LAYOUT.finditer(err)]
    assert len(lines) == c.nsets, err[-2000:]
    lay = [dict(zip(LAYOUT_KEYS, (int(x) for x in g[2:]))) for g in lines]
    assert all(x == lay[0] for x in lay)
    return sims, lay[0], (xyz, rpy)


def _actions(c, rng, sim):
    """Per-step actions of one window, host (what the oracle sees) and device."""
    E, N, A = c.E, c.kw["num_drones"], sim.A
    if c.ctrl:
        hover = load_drone_params(c.kw["model"]).HOVER_RPM
        a = hover * (1 + 0.02 * rng.uniform(-1, 1, (E, N, A)))
        a = a.astype(np.float32).astype(np.float64) if c.precision == "f32" else a
        return a, torch.from_numpy(a).to("cuda", sim.act_dtype)
    a = rng.uniform(-1, 1, (E, N, A)).astype(np.float32)
    return a, torch.from_numpy(a).cuda()


class Runner:
    """The GPU half: handles stepped in the case's pattern; window by window."""

    def __init__(self, c, sims):
        self.c, self.sims = c, sims
        self.dev_acts = None
        self.graph = None
        if c.pattern == "graph":
            for s in sims:
                s.set_step_chaining(True)

    def schedule(self):
        """(set, step slot) of every step of one window, in launch order."""
        c = self.c
        if c.pattern == "graph":
            return [(k % c.nsets, k) for _ in range(c.replays) for k in range(c.steps)]
        return [(j, k) for k in range(c.steps) for j in range(c.nsets)]

    def set_actions(self, dev):
        if self.dev_acts is None:
            self.dev_acts = [d.clone() for d in dev]
        else:
            for x, d in zip(self.dev_acts, dev):
                x.copy_(d)
        torch.cuda.synchronize()

    def run(self):
        """One window; returns per set the (obs, reward, terminated, truncated) of its last step and, for eager steps, every
        step's outputs (cloned)."""
        c = self.c
        per_step = []
        if c.pattern == "graph":
            if self.graph is None:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.stream(side):
                    with torch.cuda.graph(self.graph, stream=side):
                        for k in range(c.steps):
                            self.sims[k % c.nsets].step(self.dev_acts[k])
            for _ in range(c.replays):
                self.graph.replay()
            torch.cuda.synchronize()
            return [(s.obs, s.reward, s.terminated, s.truncated) for s in self.sims], per_step
        last = [None] * c.nsets
        for j, k in self.schedule():
            s = self.sims[j]
            out = _aligned_step(s, self.dev_acts[k], k) if c.align else s.step(self.dev_acts[k])
            last[j] = out
            per_step.append(tuple(x.clone() for x in out[1:]))
        torch.cuda.synchronize()
        return last, per_step


def _aligned_step(s, act, k):
    """Step k of an alignment window: 0 aligned; 1 actions 4 bytes off; 2 obs_prev / obs_out 4 bytes off; 3 reward and
    flags 4 bytes (one element) off.  Steps 1-3 go through step_into and hand the observation back with adopt_obs."""
    if k % 4 == 0:
        return s.step(act)
    E, N, W = s.E, s.N, s.W

    def off(shape, dtype, fill=None):
        n = int(np.prod(shape))
        esz = torch.empty((), dtype=dtype).element_size()
        base = torch.zeros(n + 16 // esz, dtype=dtype, device="cuda")
        sh = max(1, 4 // esz)
        v = base[sh:sh + n].view(shape)
        if fill is not None:
            v.copy_(fill)
        return v
    a = act
    prev = s.obs
    out = torch.empty_like(prev)
    rew, te, tr = torch.empty_like(s.reward), torch.empty_like(s.terminated), torch.empty_like(s.truncated)
    if k % 4 == 1:
        a = off(act.shape, act.dtype, act)
    elif k % 4 == 2:
        prev = off(prev.shape, prev.dtype, prev)
        out = off(prev.shape, prev.dtype)
    else:
        rew, te, tr = off(rew.shape, rew.dtype), off(te.shape, te.dtype), off(tr.shape, tr.dtype)
    s.step_into(a, prev, out, rew, te, tr)
    s.adopt_obs(out)
    return s.obs, rew, te, tr


# ---------------------------------------------------------------------------------------------------------------------
def _bands(c):
    """FP32 exemption bands of test_gpu_state_edges.py, judged on the oracle's state after each step (before its reset)."""
    if c.precision != "f32":
        return None
    kw = c.kw
    has_pid = kw["action_type"] in ("pid", "vel", "one_d_pid")

    def mark(ref, tr):
        with np.errstate(invalid="ignore"):
            tr.ex_rpy |= _rpy_band(ref.state20)
            if has_pid:     # the in-step controller's yaw wrap
                tr.ex_state |= np.abs(np.abs(ref.state20[..., 9]) - np.pi) < 1e-5
            if kw["physics_flags"] & 1:
                tr.ex_state |= tr.ex_rpy
            if not c.ctrl:
                fb = _flag_band(kw, ref.state20)
                tr.ex_flag |= fb
                tr.tainted |= fb
    return mark


def _np(x):
    return x.double().cpu().numpy() if x.dtype not in (torch.int32, torch.uint8) else x.cpu().numpy()


def _check_set(c, ctx, sim, ref, tr, got, want, stats0):
    """Window-end comparison of one env set."""
    f32 = c.precision == "f32"
    tol = F32_CEIL if f32 else F64_TOL
    o_ref, r_ref, te_ref, tr_ref = want
    obs, rew, te, trn = got
    ok_env = ~(tr.ex_flag | tr.ex_state.any(-1))
    ok = ok_env[:, None] & np.ones(c.kw["num_drones"], bool)[None]
    # ---- flags and reward of the last step ----
    if not c.ctrl:
        assert np.array_equal(_np(te)[~tr.ex_flag], te_ref[~tr.ex_flag]), ctx + ("terminated",)
        assert np.array_equal(_np(trn)[~tr.ex_flag], tr_ref[~tr.ex_flag]), ctx + ("truncated",)
    r = _np(rew)
    err = np.max(np.abs(r - r_ref)[ok_env] / np.maximum(np.abs(r_ref[ok_env]), 1.0 if f32 else 1e-3), initial=0)
    assert err <= tol["reward"], ctx + ("reward", err)
    # ---- observation ----
    g = obs.double().cpu().numpy()
    if not c.ctrl:
        assert np.array_equal(obs[..., 12:].cpu().numpy(), o_ref[..., 12:]), ctx + ("ring",)
        fo = 1.2e-7                 # float32 rounding of the RL observation
        sl = dict(pos=slice(0, 3), rpy=slice(3, 6), vel=slice(6, 9), ang_v=slice(9, 12))
    else:
        fo = 0.0
        sl = dict(pos=slice(0, 3), quat=slice(3, 7), rpy=slice(7, 10), vel=slice(10, 13), ang_v=slice(13, 16), rpm=slice(16, 20))
    w = np.asarray(o_ref, np.float64)
    for nm, s_ in sl.items():
        if nm == "rpy":
            m = ok & ~tr.ex_rpy
            e_ = angle_err(g[..., s_][m], w[..., s_][m]) - 4 * fo
        elif nm == "quat":
            e_ = quat_err(g[..., s_][ok], w[..., s_][ok])
        else:
            e_ = rel_err(g[..., s_][ok], w[..., s_][ok], floor=1e-2 if (f32 and nm == "ang_v") else 1e-3) - fo
        lim = tol[nm] if c.ctrl else max(tol[nm], tol["obs"])
        assert e_ <= lim, ctx + ("obs", nm, e_)
    # ---- terminal_kin of the envs that ended in this window (their latest end) ----
    if c.auto_reset and tr.ended.any():
        tk = sim.terminal_kin.double().cpu().numpy()
        m = tr.ended[:, None] & ok & ~tr.ex_rpy
        kd = tk - tr.tkin
        kd[..., 3:6] = (kd[..., 3:6] + np.pi) % (2 * np.pi) - np.pi
        lim = np.repeat([max(tol[q], tol["obs"]) for q in ("pos", "rpy", "vel", "ang_v")], 3)
        assert np.all(np.abs(kd[m]) <= lim * np.maximum(np.abs(tr.tkin[m]), 1)), ctx + ("terminal_kin",)
    # ---- exported state, counters ----
    st20, rr, ps, cnt = (_np(x) for x in sim.get_state())
    rs = ref.state20
    assert np.array_equal(cnt[ok_env], ref.step_counter[ok_env]), ctx + ("counter",)
    fr = 1e-2 if f32 else 1e-3
    if f32 and c.kw["action_type"] in ("pid", "vel", "one_d_pid"):
        tol = dict(tol, rpm=tol["pid"])         # the RPM is the FP32 controller's output: the controller's bound
    for nm, g_, w_, fl in (("pos", st20[..., S_POS], rs[..., S_POS], 1e-3), ("vel", st20[..., S_VEL], rs[..., S_VEL], 1e-3),
                           ("rates", rr, ref.rpy_rates, fr), ("ang_v", st20[..., S_ANGV], rs[..., S_ANGV], fr),
                           ("rpm", st20[..., S_RPM], rs[..., S_RPM], 1e-3)):
        e_ = rel_err(g_[ok], w_[ok], floor=fl)
        assert e_ <= tol[nm], ctx + (nm, e_)
    e_ = quat_err(st20[..., S_QUAT][ok], rs[..., S_QUAT][ok])
    assert e_ <= tol["quat"], ctx + ("quat", e_)
    m = ok & ~tr.ex_rpy
    e_ = angle_err(st20[..., S_RPY][m], rs[..., S_RPY][m])
    assert e_ <= tol["rpy"], ctx + ("rpy", e_)
    if c.kw["action_type"] in ("pid", "vel", "one_d_pid"):
        e_ = max(rel_err(ps[..., 0:6][ok], ref.pid_state[..., 0:6][ok]), angle_err(ps[..., 6:9][m], ref.pid_state[..., 6:9][m]))
        assert e_ <= tol["pid"], ctx + ("pid", e_)
    # ---- episode statistics over the window ----
    if c.auto_reset:
        d = sim.episode_stats() - stats0
        assert d[6] == tr.steps, ctx + ("env_steps", d[6], tr.steps)
        n_band = int(tr.ex_flag.sum())
        if n_band == 0:
            assert d[0] == tr.n_ep and d[2] == tr.sum_len, ctx + ("episodes", d[0], tr.n_ep, d[2], tr.sum_len)
            if tr.ret_ok:
                assert abs(d[1] - tr.sum_ret) <= 1e-5 * max(abs(tr.sum_ret), 1.0), ctx + ("returns", d[1], tr.sum_ret)
        else:
            assert abs(d[0] - tr.n_ep) <= n_band, ctx + ("episodes", d[0], tr.n_ep, n_band)


def _snapshot(sims):
    out = []
    for s in sims:
        out += [x.clone() for x in s.get_state()] + [s.obs.clone(), s.reward.clone(), s.terminated.clone(), s.truncated.clone()]
        if s.auto_reset:
            out.append(torch.from_numpy(s.episode_stats()))
    return out


def _run(c, name, capfd, monkeypatch, extra_env=None, oracle=True):
    """The case's windows; returns the layout witness and the window-end snapshots (for the bit-identity variants)."""
    oracle = oracle and not c.dw32
    sims, lay, (xyz, rpy) = _make(c, capfd, monkeypatch, extra_env)
    kw = c.kw
    refs = tracks = None
    if oracle:
        refs = [se.oracle_sim(kw, c.E, xyz, rpy) for _ in range(c.nsets)]
        tracks = [Track(c.E, kw["num_drones"], kw["pyb_freq"] // kw["ctrl_freq"]) for _ in range(c.nsets)]
    from oracle import oracle as orc
    nth = orc.max_threads()
    for s in sims:
        s.reset()
    run = Runner(c, sims)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    bands = _bands(c)
    snaps = []
    n_slots = c.steps
    for w in range(c.windows):
        host, dev = zip(*[_actions(c, rng, sims[0]) for _ in range(n_slots)])
        run.set_actions(dev)
        stats0 = []
        if oracle:
            for s, ref, tr in zip(sims, refs, tracks):
                st20, rr, ps, cnt = (_np(x) for x in s.get_state())
                load_oracle(ref, st20, rr, ps, cnt, s.obs.cpu().numpy())
                tr.start(cnt)
                stats0.append(s.episode_stats() if c.auto_reset else None)
        last, per_step = run.run()
        snaps.append(_snapshot(sims))
        if not oracle:
            continue
        sched = run.schedule()
        wants = [None] * c.nsets
        for j in range(c.nsets):
            acts = [host[k] for (jj, k) in sched if jj == j]
            if c.pattern == "eager":            # every step's reward and flags (outputs only: no state is read)
                steps_j = [p for (jj, _), p in zip(sched, per_step) if jj == j]
                for t, (a, p) in enumerate(zip(acts, steps_j)):
                    wants[j] = step_window(refs[j], tracks[j], [a], c.auto_reset, nth, bands)
                    _, r_ref, te_ref, tr_ref = wants[j]
                    ok_env = ~(tracks[j].ex_flag | tracks[j].ex_state.any(-1))
                    if not c.ctrl:
                        assert np.array_equal(_np(p[1])[ok_env], te_ref[ok_env]), (name, w, j, t, "terminated")
                        assert np.array_equal(_np(p[2])[ok_env], tr_ref[ok_env]), (name, w, j, t, "truncated")
                    f32 = c.precision == "f32"
                    err = np.max(np.abs(_np(p[0]) - r_ref)[ok_env] / np.maximum(np.abs(r_ref[ok_env]), 1.0 if f32 else 1e-3),
                                 initial=0)
                    assert err <= (F32_CEIL if f32 else F64_TOL)["reward"], (name, w, j, t, "reward", err)
            else:
                wants[j] = step_window(refs[j], tracks[j], acts, c.auto_reset, nth, bands)
            _check_set(c, (name, w, j), sims[j], refs[j], tracks[j], last[j], wants[j], stats0[j])
            if bands is not None:
                tr = tracks[j]
                for m in (tr.ex_state.any(-1), tr.ex_rpy.any(-1), tr.ex_flag):
                    assert m.mean() < 0.05, (name, w, j, m.mean())
    return sims, run, lay, snaps


def _profile_launches(run, tmp_path):
    """One more window under torch.profiler (not compared): (kernel name, grid x) of every step launch."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        run.run()
        torch.cuda.synchronize()
    path = os.path.join(str(tmp_path), "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    out = []
    for e in ev:
        if e.get("cat") == "kernel" and "gpd::" in e.get("name", ""):
            out.append((e["name"], int(e.get("args", {}).get("grid", [0])[0]), int(e.get("args", {}).get("shared memory", -1))))
    return out


@pytest.mark.parametrize("name", list(CASES))
def test_cuda_path_vs_oracle(name, capfd, monkeypatch, tmp_path):
    c = CASES[name]
    sims, run, lay, snaps = _run(c, name, capfd, monkeypatch)
    # ---- create-time witness ----
    for k, v in c.layout.items():
        assert lay[k] == v, (name, k, lay)
    # ---- per-launch witness: one untimed, unchecked window under the profiler ----
    launches = _profile_launches(run, tmp_path)
    steps = [x for x in launches if "step_kernel" in x[0]]
    n_launch = len(run.schedule())
    # the trace may miss one eager launch at its edge, and some of the kernels a replayed graph launches: each recorded launch
    # must show the path
    lo = n_launch - 1 if c.pattern == "eager" else 1
    assert lo <= len(steps) <= n_launch, (name, launches[:8])
    if c.align:
        # aligned steps and misaligned outputs stay on the bulk kernel; misaligned actions or observations take the
        # per-thread kernel (its scalar variant), behind a state sync on a chained-state handle
        n_bulk = sum("step_kernel_bulk" in x[0] for x in steps)
        n_thr = sum(re.search(r"step_kernel<\w+, \d, \w+, false>", x[0]) is not None for x in steps)
        want_bulk = sum(k % 4 in (0, 3) for _, k in run.schedule())
        assert want_bulk - 1 <= n_bulk <= want_bulk and n_bulk + n_thr == len(steps), (name, [x[0] for x in steps])
        syncs = sum("state_sync_kernel" in x[0] for x in launches)
        want = 2 * c.nsets if lay["state_in_obs"] else 0
        assert want - 1 <= syncs <= want, (name, syncs)
    else:
        assert all(c.kernel in x[0] for x in steps), (name, c.kernel, {x[0] for x in steps})
        if c.grids:
            grids = [x[1] for x in steps]
            assert set(grids) <= set(c.grids), (name, sorted(set(grids)))
            if len(c.grids) > 1:            # two tiles per CTA behind another handle: every launch but the graph's first
                assert grids.count(min(c.grids)) >= len(steps) - c.replays, (name, grids)
    for s in sims:
        s.close()
    # ---- runtime-selected variants of the same kernel instance: the same bits ----
    for var in c.variants:
        v_sims, _, v_lay, v_snaps = _run(c, name, capfd, monkeypatch, extra_env=var, oracle=False)
        if "GPD_TMA" in var:
            assert v_lay["tma"] == 0, (name, var, v_lay)
        if "GPD_TMA_EDGE" in var:
            assert v_lay["tma_edge"] == int(var["GPD_TMA_EDGE"]), (name, var, v_lay)
        for wsnap, vsnap in zip(snaps, v_snaps):
            for x, y in zip(wsnap, vsnap):
                if x.dtype == torch.float64 and x.numel() == 8 and x.device.type == "cpu":
                    # episode_stats: counts exact; the sums of returns are FP32 partial sums per CTA, whose grouping
                    # follows the block size the wave search picks for the variant's shared-memory need
                    i = [0, 2, 4, 5, 6, 7]
                    assert torch.equal(x[i], y[i]), (name, var, x, y)
                    assert torch.allclose(x[[1, 3]], y[[1, 3]], rtol=1e-6, atol=0), (name, var, x, y)
                else:
                    assert torch.equal(bits(x), bits(y)), (name, var)
        for s in v_sims:
            s.close()
