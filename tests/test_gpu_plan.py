"""-m gpu: planning rollouts (gpd_plan).  The reference is a replica handle: a BatchedSim of E*S envs of the same
configuration without auto-reset, holding the source handle's exported state repeated S times (state20 with the previous
RPM, rpy_rates, pid_state, counter; per-env targets repeated too), stepped K times by gpd_step on the plan's actions.  Its
returns / done_step come from the recurrence of include/gpd.h restated in torch (plan_ref.py), and its last observation's
kin is the expected final_kin.  FP64: bit for bit.  FP32: within the FP32 ceilings and threshold bands of
test_gpu_rollout.py, done_step exact outside the bands, returns exactly the recurrence over the plan's own rewards."""
import ctypes as C
import types
import zlib

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import state_edges as se
from paths_harness import load_oracle
from plan_ref import plan_returns
from test_gpu_rollout import F32_ATOL, bits, flag_band, schedule
from helpers import default_targets
from gpd_b200 import _lib
from gpd_b200.params import load_drone_params
from gpd_b200.sim import BatchedSim
from gpd_b200.utils.enums import DroneModel

pytestmark = pytest.mark.gpu

MULTI2_DW = dict(env_kind="multihover", action_type="rpm", num_drones=2, pyb_freq=240, ctrl_freq=30, physics_flags=4)
MULTI2_GD = dict(env_kind="multihover", action_type="rpm", num_drones=2, pyb_freq=240, ctrl_freq=30, physics_flags=3)


def shape(name, **over):
    if name in ("multi2_dw", "multi2_gd"):
        kw = dict(MULTI2_DW if name == "multi2_dw" else MULTI2_GD, model=DroneModel.CF2X, episode_len_sec=8.0)
        kw.update(over)
        return kw
    return se.shape(name, **over)


def make(kw, E, precision, auto_reset=True, chaining=False):
    s = BatchedSim(load_drone_params(kw["model"]), E, kw["num_drones"], env_kind=kw["env_kind"],
                   action_type=kw["action_type"], pyb_freq=kw["pyb_freq"], ctrl_freq=kw["ctrl_freq"],
                   physics_flags=kw["physics_flags"], precision=precision, auto_reset=auto_reset,
                   target_pos=default_targets(kw), episode_len_sec=kw["episode_len_sec"])
    if chaining:
        s.set_step_chaining(True)
    return s


def plan_actions(rng, s, K, S, scale=0.3):
    """(K, E, S, N, A) in the action dtype, drawn as test_gpu_rollout.schedule draws them."""
    fake = types.SimpleNamespace(E=s.E * S, N=s.N, A=s.A, action_type=s.action_type, act_dtype=s.act_dtype)
    return schedule(rng, fake, K, scale).reshape(K, s.E, S, s.N, s.A).contiguous()


def advance(s, rng, n=5):
    for _ in range(n):
        s.step(schedule(rng, s, 1)[0])


def replica(src, kw, S, precision, envs=None, targets=None):
    """E*S envs (or len(envs)*S) holding the source's state repeated S times, without auto-reset."""
    st, rr, ps, cnt = src.get_state()
    if envs is not None:
        st, rr, ps, cnt = st[envs], rr[envs], ps[envs], cnt[envs]
    r = make(kw, st.shape[0] * S, precision, auto_reset=False)
    if targets is not None:
        r.set_targets(np.repeat(np.asarray(targets, np.float64), S, axis=0))
    r.set_state(st.repeat_interleave(S, 0), rr.repeat_interleave(S, 0), ps.repeat_interleave(S, 0),
                cnt.repeat_interleave(S, 0))
    return r


def run_replica(r, acts):
    K = acts.shape[0]
    a = acts.reshape(K, r.E, r.N, r.A)
    rew, done, kin = [], [], []
    for k in range(K):
        obs, rw, te, tr = r.step(a[k])
        rew.append(rw.clone())
        done.append((te | tr).bool())
        kin.append(obs[..., :12].clone())
    return torch.stack(rew), torch.stack(done), torch.stack(kin)


def check(src, rep, acts, gamma, res, precision, tag):
    """res: the plan's dict (reward and final_kin included); rep: the replica handle."""
    K, E, S = acts.shape[:3]
    rew, done, kin = run_replica(rep, acts)
    G, step = plan_returns(rew, done, gamma)
    pr, pd, pk, pg = res["reward"].reshape(K, E * S), res["done_step"].reshape(-1), res["final_kin"], res["returns"]
    if precision == "f64":
        assert torch.equal(bits(pr), bits(rew)), f"{tag}: reward"
        assert torch.equal(bits(pg.reshape(-1)), bits(G)), f"{tag}: returns"
        assert torch.equal(pd, step), f"{tag}: done_step"
        assert torch.equal(bits(pk.reshape(kin[-1].shape)), bits(kin[-1])), f"{tag}: final_kin"
        return
    kin_np = kin.double().cpu().numpy()
    band = np.zeros(E * S, bool)
    for k in range(K):
        band |= flag_band(rep, kin_np[k])
    # the recurrence over the plan's own rewards, bit for bit
    ended = torch.arange(K, device=pd.device)[:, None] == pd[None, :].long()
    G_own, step_own = plan_returns(pr, ended, gamma)
    assert torch.equal(step_own, pd)
    assert torch.equal(bits(pg.reshape(-1)), bits(G_own)), f"{tag}: returns vs the recurrence over the plan's rewards"
    ok = ~band
    assert torch.equal(pd[torch.as_tensor(ok, device=pd.device)], step[torch.as_tensor(ok, device=pd.device)]), \
        f"{tag}: done_step outside the FP32 bands"
    a, b = pr.double().cpu().numpy(), rew.double().cpu().numpy()
    badr = ~np.isclose(a, b, rtol=1e-4, atol=1e-4).all(0) & ok
    assert not badr.any(), f"{tag}: reward, copies {np.nonzero(badr)[0][:8]}"
    x, y = pk.reshape(kin[-1].shape).double().cpu().numpy(), kin[-1].double().cpu().numpy()
    d = np.abs(x - y)
    d[..., 3:6] = np.minimum(d[..., 3:6], np.abs(2 * np.pi - d[..., 3:6]))
    badk = ~((d <= F32_ATOL[12]) | (np.isnan(x) & np.isnan(y))).reshape(E * S, -1).all(-1) & ok
    assert not badk.any(), f"{tag}: final_kin beyond the FP32 ceilings, copies {np.nonzero(badk)[0][:8]}, max {np.nanmax(d)}"
    same = (x.view(np.uint64) == y.view(np.uint64)).reshape(E * S, -1).all(-1)
    print(f"[plan] {tag}: {100.0 * same.mean():.1f} % of the copies' final kin bit-identical "
          f"({int(band.sum())} of {E * S} copies in an FP32 threshold band)")


# (shape, S, E, K, gamma, episode_len_sec): every shape once with S > 1 and K = 16; multi-drone shapes with E*S not a
# multiple of the envs per CTA
CASES = [
    ("hover30", 64, 37, 16, 0.9, 8.0), ("hover30", 1, 1, 1, 1.0, 8.0), ("one_d_rpm", 3, 37, 16, 1.0, 0.3),
    ("pid", 3, 37, 16, 0.9, 8.0), ("vel", 64, 1, 16, 1.0, 8.0), ("one_d_pid", 3, 37, 16, 0.9, 0.3),
    ("gnd_drag", 64, 37, 16, 0.9, 8.0), ("multi3", 3, 37, 16, 1.0, 0.3), ("multi3", 64, 1, 1, 0.9, 8.0),
    ("multi3_gd", 64, 37, 16, 0.9, 8.0), ("multi2_dw", 3, 37, 16, 0.9, 8.0), ("cf2p", 3, 37, 16, 1.0, 8.0),
    ("race", 3, 1, 16, 0.9, 0.3),
]


def case_kw(name, ep):
    if name == "cf2p":
        return shape("hover30", model=DroneModel.CF2P, episode_len_sec=ep)
    if name == "race":
        return shape("hover30", model=DroneModel.RACE, episode_len_sec=ep)
    return shape(name, episode_len_sec=ep)


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name,S,E,K,gamma,ep", CASES)
def test_plan_matches_replica(precision, name, S, E, K, gamma, ep):
    kw = case_kw(name, ep)
    rng = np.random.default_rng(zlib.crc32(f"{name} {S} {E} {K}".encode()))
    src = make(kw, E, precision)
    src.reset()
    advance(src, rng)
    acts = plan_actions(rng, src, K, S)
    res = src.plan(acts, gamma=gamma, reward=True, final_kin=True)
    check(src, replica(src, kw, S, precision), acts, gamma, res, precision, f"{precision} {name} S={S} E={E} K={K}")


@pytest.mark.parametrize("fam", ["F5", "F7"])
@pytest.mark.parametrize("name", ["hover30", "multi3"])
def test_plan_episode_ends(fam, name):
    seen = set()
    K, S, E = 16, 3, 96
    for ep in (8.0, 1 / 3):
        kw = shape(name, episode_len_sec=ep)
        rng = np.random.default_rng(7)
        f = se.FAMILIES[fam](rng, kw, E, "f64")
        src = make(kw, E, "f64")
        src.reset()
        src.set_state(torch.as_tensor(f["state20"]), torch.as_tensor(f["rpy_rates"]), torch.as_tensor(f["pid_state"]),
                      torch.as_tensor(f["step_counter"]))
        a2 = torch.as_tensor(f["actions"], dtype=torch.float32, device="cuda")        # (2, E, N, A)
        acts = a2[torch.arange(K) % 2][:, :, None].expand(K, E, S, kw["num_drones"], src.A).contiguous()
        res = src.plan(acts, gamma=0.9, reward=True, final_kin=True)
        check(src, replica(src, kw, S, "f64"), acts, 0.9, res, "f64", f"{fam} {name} ep={ep:.3f}")
        seen |= set(np.unique(res["done_step"].cpu().numpy()).tolist())
    if fam == "F5":
        assert 0 in seen and K in seen and any(0 < k < K for k in seen), sorted(seen)


def _snapshot(s):
    st = s.get_state()
    return [bits(x).clone() for x in (s.obs_buf[0], s.obs_buf[1]) + tuple(st)]


@pytest.mark.parametrize("kind", ["f32_chained_65536", "f64_multihover"])
def test_plan_leaves_the_source_untouched(kind):
    if kind == "f32_chained_65536":
        kw, E, prec, chaining = shape("hover30"), 65536, "f32", True
    else:
        kw, E, prec, chaining = shape("multi3_gd", episode_len_sec=0.3), 37, "f64", False
    a, b = make(kw, E, prec, chaining=chaining), make(kw, E, prec, chaining=chaining)
    rng = np.random.default_rng(11)
    sched = [schedule(rng, a, 1)[0] for _ in range(12)]
    for s in (a, b):
        s.reset()
        for k in range(7):
            s.step(sched[k])
    acts = plan_actions(rng, a, 8, 4)
    a.plan(acts, gamma=0.9, reward=True, final_kin=True)
    for s in (a, b):
        for k in range(7, 12):
            s.step(sched[k])
    torch.cuda.synchronize()
    for x, y in zip(_snapshot(a), _snapshot(b)):
        assert torch.equal(x, y)
    assert np.array_equal(a.episode_stats(), b.episode_stats())


def test_plan_after_steps_same_as_before():
    """The plan itself leaves every buffer of the handle as it found it (before vs after, nothing stepped between)."""
    kw = shape("multi3_gd", episode_len_sec=0.3)
    s = make(kw, 37, "f64")
    s.reset()
    advance(s, np.random.default_rng(2))
    before = _snapshot(s) + [torch.as_tensor(s.episode_stats())]
    s.plan(plan_actions(np.random.default_rng(3), s, 16, 5), reward=True, final_kin=True)
    after = _snapshot(s) + [torch.as_tensor(s.episode_stats())]
    for x, y in zip(before, after):
        assert torch.equal(x, y)


def test_plan_oracle_anchor():
    kw = shape("multi2_gd")
    E, S, K = 16, 8, 16
    rng = np.random.default_rng(5)
    src = make(kw, E, "f64")
    src.reset()
    advance(src, rng)
    acts = plan_actions(rng, src, K, S)
    res = src.plan(acts, reward=True, final_kin=True)
    st, rr, ps, cnt = (x.cpu().numpy() for x in src.get_state())
    obs = src.obs.cpu().numpy()
    pairs = [(e, s) for e in range(E) for s in range(S)][::2][:64]
    ref = se.oracle_sim(kw, len(pairs))
    idx = np.array([e for e, _ in pairs])
    load_oracle(ref, st[idx], rr[idx], ps[idx], cnt[idx], obs[idx])
    a = acts.cpu().numpy()
    rew = []
    for k in range(K):
        o, r, _, _ = ref.step(np.stack([a[k, e, s] for e, s in pairs]))
        rew.append(r.copy())
    pr = res["reward"].cpu().numpy()
    pk = res["final_kin"].cpu().numpy()
    got_r = np.stack([pr[:, e, s] for e, s in pairs], 1)
    got_k = np.stack([pk[e, s] for e, s in pairs])
    assert np.abs(got_r - np.stack(rew)).max() <= 1e-9
    assert np.abs(got_k - o[..., :12]).max() <= 1e-9


def test_plan_target_override():
    kw = shape("hover30")
    E, S, K = 37, 3, 16
    rng = np.random.default_rng(8)
    src = make(kw, E, "f64")
    src.reset()
    advance(src, rng)
    acts = plan_actions(rng, src, K, S)
    own = src.plan(acts, reward=True, final_kin=True)
    own = {k: v.clone() for k, v in own.items()}
    tg = np.array([[0.0, 0.0, 1.0]]) + rng.uniform(-0.3, 0.3, (E, 1, 3))
    res = src.plan(acts, targets=torch.as_tensor(tg, device="cuda"), reward=True, final_kin=True)
    check(src, replica(src, kw, S, "f64", targets=tg), acts, 1.0, res, "f64", "target override")
    again = src.plan(acts, reward=True, final_kin=True)
    for k in own:
        assert torch.equal(bits(own[k]), bits(again[k])), f"handle targets changed: {k}"


def test_plan_graph_replay():
    kw = shape("hover30")
    s = make(kw, 65536, "f32", chaining=True)
    s.reset()
    rng = np.random.default_rng(9)
    for _ in range(4):
        s.step(schedule(rng, s, 1)[0])
    acts = plan_actions(rng, s, 16, 2)
    eager = {k: v.clone() for k, v in s.plan(acts, gamma=0.9, reward=True, final_kin=True).items()}
    out = s.alloc_plan_outputs(16, 2, reward=True, final_kin=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            s.plan(acts, gamma=0.9, reward=True, final_kin=True, out=out)
    torch.cuda.current_stream().wait_stream(side)
    for v in out.values():
        v.zero_()
    g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(bits(eager[k]), bits(out[k])), k


def test_plan_large_copy_count():
    kw = shape("hover30")
    E, S, K = 4096, 256, 32
    rng = np.random.default_rng(12)
    src = make(kw, E, "f32")
    src.reset()
    advance(src, rng)
    acts = plan_actions(rng, src, K, S)
    res = src.plan(acts, gamma=0.99, reward=True, final_kin=True)
    envs = torch.tensor([0, 1111, 2222, 4095], device="cuda")
    sub = {"reward": res["reward"][:, envs].contiguous(), "done_step": res["done_step"][envs].contiguous(),
           "final_kin": res["final_kin"][envs].contiguous(), "returns": res["returns"][envs].contiguous()}
    check(src, replica(src, kw, S, "f32", envs=envs), acts[:, envs].contiguous(), 0.99, sub, "f32", "E=4096 S=256 K=32")


def test_plan_invalid_arguments():
    L = _lib.load()
    kw = shape("hover30")
    s = make(kw, 4096, "f32")
    s.reset()
    E, N, A, K, S = s.E, s.N, s.A, 4, 2
    acts = torch.zeros((K, E, S, N, A), device="cuda")
    big = torch.zeros(K * E * S * N * A + 4, device="cuda")
    ret = torch.zeros((E, S), device="cuda")
    done = torch.zeros((E, S), dtype=torch.int32, device="cuda")
    rew = torch.zeros((K, E, S), device="cuda")
    fk = torch.zeros(E * S * N * 12 + 4, device="cuda")
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)
    st = s._stream()
    ok = (s.h, K, S, p(acts), None, 0.9, p(ret), p(done), p(rew), p(fk), st)
    assert L.gpd_plan(*ok) == 0

    def bad(**kv):
        names = ["h", "K", "S", "actions", "targets", "gamma", "returns", "done_step", "reward", "final_kin", "stream"]
        args = list(ok)
        for k, v in kv.items():
            args[names.index(k)] = v
        return L.gpd_plan(*args)
    cases = [dict(K=0), dict(S=0), dict(K=-1), dict(gamma=float("nan")), dict(gamma=float("inf")), dict(gamma=-0.1),
             dict(gamma=1.5), dict(actions=None), dict(returns=None), dict(actions=p(big, 4)), dict(final_kin=p(fk, 4)),
             dict(reward=p(ret)), dict(done_step=p(ret)), dict(final_kin=p(rew)), dict(returns=p(acts)),
             dict(S=2 ** 31 - 1)]
    for c in cases:
        assert bad(**c) == -1, c
        assert L.gpd_plan(*ok) == 0, f"handle unusable after {c}"
    ctrl = BatchedSim(load_drone_params(DroneModel.CF2X), 4, 1, env_kind="ctrl", action_type="ctrl_rpm", pyb_freq=240,
                      ctrl_freq=48, precision="f32")
    assert L.gpd_plan(ctrl.h, K, S, p(acts), None, 1.0, p(ret), None, None, None, st) == -1
    with pytest.raises(ValueError):
        ctrl.plan(torch.zeros((K, 4, S, 1, 4), device="cuda"))
    s.step(torch.zeros((E, N, A), device="cuda"))
    torch.cuda.synchronize()


def test_mppi_example():
    from gpd_b200.examples import mppi
    d = mppi.run(num_envs=64, samples=256, horizon=16, steps=90, start_offset=0.3, seed=0)
    print(f"[plan] MPPI 64 envs, S=256, H=16: mean distance {d[0]:.4f} m after 1 step, {d[-1]:.4f} m after 90 steps")
    assert d[-1] < 0.15, d[::10]
    g = mppi.run(num_envs=64, samples=256, horizon=16, steps=90, start_offset=0.3, seed=0, graph=True)
    print(f"[plan] MPPI graphed: {g[-1]:.4f} m after 90 steps")
    assert g[-1] < 0.15, g[::10]
    z = mppi.run(num_envs=64, samples=16, horizon=4, steps=30, start_offset=0.3, sigma=0.0)
    assert np.allclose(z, 0.3, atol=1e-3), z[::5]
