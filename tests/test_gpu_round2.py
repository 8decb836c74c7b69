"""Round-2 GPU parity tests: the host observation mirror (gpd_step_mirror), env pools behind the VecEnv adapter, per-CTA
step sequencing (programmatic dependent launch), gpd_adjacency, per-env MultiHover targets, the in-library NCCL statistics
reduce and the legacy row-major gpd_step_host.  All call through the C ABI; the oracle is the checker."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import S_POS, S_VEL, default_targets, make_oracle, rel_err
import gpd_b200  # noqa: F401
from gpd_b200 import _lib
from gpd_b200.params import load_drone_params
from gpd_b200.utils.enums import DroneModel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_sim(kw, num_envs=1, precision="f64", auto_reset=False, tpb=0, target=None):
    from gpd_b200.sim import BatchedSim
    dp = load_drone_params(kw["model"])
    return BatchedSim(dp, num_envs, kw["num_drones"], env_kind=kw["env_kind"], action_type=kw["action_type"],
                      pyb_freq=kw["pyb_freq"], ctrl_freq=kw["ctrl_freq"], physics_flags=kw["physics_flags"], precision=precision,
                      auto_reset=auto_reset, target_pos=default_targets(kw) if target is None else target,
                      init_xyz=kw["init_xyz"], init_rpy=kw["init_rpy"], threads_per_block=tpb)


def _kw(env_kind="hover", act="rpm", N=1, freq=30, flags=0, model=DroneModel.CF2X):
    return dict(model=model, env_kind=env_kind, action_type=act, num_drones=N, pyb_freq=240, ctrl_freq=freq, physics_flags=flags,
                init_xyz=None, init_rpy=None)


@pytest.mark.parametrize("act,N,freq,precision,io", [
    ("rpm", 1, 30, "f32", "zc"), ("rpm", 1, 48, "f64", "zc"), ("pid", 1, 48, "f32", "zc"),
    ("one_d_rpm", 1, 30, "f32", "zc"), ("rpm", 3, 30, "f32", "zc"), ("vel", 2, 30, "f64", "zc"),
    ("rpm", 1, 30, "f32", "zc_pinned_actions"), ("pid", 1, 48, "f64", "zc_pinned_actions"), ("rpm", 2, 30, "f32", "zc_pinned_actions"),
    ("rpm", 1, 30, "f32", "dma"), ("vel", 2, 30, "f64", "dma"), ("rpm", 1, 48, "f32", "dma"),
    ("rpm", 1, 30, "f32", "pageable_outputs")])
def test_cuda_host_mirror_equals_device_observation(act, N, freq, precision, io, monkeypatch):
    """The numpy-facing step returns a strided view of the pinned feature-major log; at every step it must equal, bit for bit,
    the device observation (same chain), through window slides, compactions (16-step log), masked and full resets, and
    tensor-path steps in between (stale mirror -> rebuilt).  io: "zc" = the zero-copy step (pinned result arrays: the kernel
    writes kin rows / reward / flags / terminal rows straight into host memory; pageable actions are staged),
    "zc_pinned_actions" = it also reads the actions from host memory, "dma" = GPD_MIRROR_ZEROCOPY=0 (staging + copies),
    "pageable_outputs" = result arrays the device cannot address (falls back to staging + copies by itself)."""
    rng = np.random.default_rng(3)
    E = 517
    if io == "dma":
        monkeypatch.setenv("GPD_MIRROR_ZEROCOPY", "0")
    kw = _kw("hover" if N == 1 else "multihover", act, N, freq, model=DroneModel.CF2P if act in ("pid", "vel") else DroneModel.CF2X)
    sim = make_sim(kw, E, precision, auto_reset=True)
    twin = make_sim(kw, E, precision, auto_reset=True)      # the same run on device tensors only
    sim.attach_mirror(slide_steps=16)
    A = sim.A
    out = sim.alloc_host_outputs(pinned=io != "pageable_outputs", terminal_kin=True)
    pinned_a = torch.empty((E, N, A), dtype=torch.float32).pin_memory().numpy() if io == "zc_pinned_actions" else None
    obs = sim.reset_host()
    twin.reset()
    assert obs.shape == (E, N, sim.W) and obs.dtype == np.float32 and not obs.flags["C_CONTIGUOUS"]
    assert np.array_equal(obs, sim.obs.cpu().numpy()) and np.array_equal(obs, twin.obs.cpu().numpy())
    for t in range(70):
        a = rng.uniform(-1, 1, (E, N, A)).astype(np.float32)
        if pinned_a is not None:
            pinned_a[...] = a
            a = pinned_a
        od, rd, td, trd = twin.step(torch.from_numpy(a).cuda())
        if t in (23, 24, 40):               # tensor-path steps: the device chain moves without the mirror
            sim.step(torch.from_numpy(a).cuda())
            continue
        obs, rew, term, trunc, tkin = sim.step_host(a, out)
        assert np.array_equal(obs, sim.obs.cpu().numpy()), (t, "host obs == this sim's device obs")
        assert np.array_equal(obs, od.cpu().numpy()), (t, "host obs == the tensor-path twin's obs")
        assert np.array_equal(obs[..., -A:], a), (t, "newest ring slot is this step's action")
        assert np.array_equal(rew, rd.cpu().numpy()) and np.array_equal(term, td.cpu().numpy())
        assert np.array_equal(trunc, trd.cpu().numpy())
        done = (term | trunc).astype(bool)
        if done.any():
            assert np.array_equal(tkin[done], twin.terminal_kin.cpu().numpy()[done])
        if t == 30:                         # masked reset through the host path: ring survives, kin rows refreshed in place
            m = (rng.random(E) < 0.4).astype(np.uint8)
            o2 = sim.reset_host(m)
            twin.reset(torch.from_numpy(m))
            assert np.array_equal(o2, sim.obs.cpu().numpy()) and np.array_equal(o2, twin.obs.cpu().numpy())
            assert np.array_equal(o2[..., 12:], obs[..., 12:])
        if t == 50:
            o3 = sim.reset_host()
            twin.reset()
            assert np.array_equal(o3, sim.obs.cpu().numpy()) and np.array_equal(o3, twin.obs.cpu().numpy())
    sim.close(); twin.close()


def test_cuda_host_mirror_tracks_the_oracle():
    """HoverAviary.step(numpy) (mirror path) against the oracle: obs, reward, flags over 60 steps with auto-reset."""
    from gpd_b200.envs import HoverAviary
    rng = np.random.default_rng(11)
    E = 300
    env = HoverAviary(num_envs=E, precision="f64", auto_reset=True)
    ref = make_oracle(_kw(), num_envs=E)
    obs, _ = env.reset(as_numpy=True)
    assert np.max(np.abs(obs - ref.obs)) <= 1e-6
    for t in range(60):
        a = rng.uniform(-1, 1, (E, 1, 4)).astype(np.float32)
        obs, rew, term, trunc, info = env.step(a)
        o_ref, r_ref, te_ref, tr_ref = ref.step(a)
        o_ref = o_ref.copy()
        d = (te_ref | tr_ref).astype(bool)
        if d.any():
            o_ref[d] = ref.reset(d.astype(np.uint8))[d]
        assert np.max(np.abs(obs - o_ref)) <= 1e-6 and np.max(np.abs(rew - r_ref)) <= 1e-9
        assert np.array_equal(term, te_ref.astype(bool)) and np.array_equal(trunc, tr_ref.astype(bool))
        assert info == {"answer": 42}
    o, _ = env.reset()                    # numpy mode is sticky: reset answers in numpy, ring intact
    assert isinstance(o, np.ndarray) and np.array_equal(o[..., 12:], obs[..., 12:])
    ck = env.checkpoint()
    a = rng.uniform(-1, 1, (E, 1, 4)).astype(np.float32)
    o1 = np.array(env.step(a)[0])
    env.restore(ck)                        # resume bit-exactly, ring included, through the numpy path
    o2 = np.array(env.step(a)[0])
    assert np.array_equal(o1, o2)
    env.close()


def test_cuda_legacy_row_major_step_host_on_rl_env():
    """gpd_step_host / gpd_reset_host (dense row-major host observation, internal device chain) still equal gpd_step."""
    rng = np.random.default_rng(2)
    E = 130
    kw = _kw(act="pid", freq=48, model=DroneModel.CF2P)
    s1, s2 = make_sim(kw, E), make_sim(kw, E)
    L = _lib.load()
    obs = np.empty((E, 1, s2.W), np.float32); rew = np.empty(E); te = np.empty(E, np.uint8); tr = np.empty(E, np.uint8)
    s1.reset()
    _lib.check(L.gpd_reset_host(s2.h, None, C.c_void_p(obs.ctypes.data), None))
    assert np.array_equal(obs, s1.obs.cpu().numpy())
    for t in range(6):
        a = rng.uniform(-1, 1, (E, 1, 3)).astype(np.float32)
        od, rd, td, trd = s1.step(torch.from_numpy(a).cuda())
        _lib.check(L.gpd_step_host(s2.h, C.c_void_p(a.ctypes.data), C.c_void_p(obs.ctypes.data), C.c_void_p(rew.ctypes.data),
                                   C.c_void_p(te.ctypes.data), C.c_void_p(tr.ctypes.data), None, None))
        assert np.array_equal(obs, od.cpu().numpy()) and np.array_equal(rew, rd.cpu().numpy())
        assert np.array_equal(te, td.cpu().numpy()) and np.array_equal(tr, trd.cpu().numpy())
    m = (rng.random(E) < 0.5).astype(np.uint8)
    s1.reset(torch.from_numpy(m))
    _lib.check(L.gpd_reset_host(s2.h, C.c_void_p(m.ctypes.data), C.c_void_p(obs.ctypes.data), None))
    assert np.array_equal(obs, s1.obs.cpu().numpy())
    s1.close(); s2.close()


def test_cuda_mirror_rejects_bad_use():
    kw = _kw("ctrl", "ctrl_rpm")
    s = make_sim(kw, 8)
    with pytest.raises(ValueError):
        s.attach_mirror()
    s.close()
    s = make_sim(_kw(), 8)
    L = _lib.load()
    base = C.c_void_p()
    _lib.check(L.gpd_mirror_alloc(10, 8, C.byref(base)))
    assert L.gpd_mirror_attach(s.h, base, 10, 8, 0) == -1 and b"rows" in L.gpd_last_error()     # needs W + A rows
    assert L.gpd_step_mirror(s.h, base, None, None, None, None, None, None, None, None) == -1    # nothing attached
    _lib.check(L.gpd_mirror_free(base))
    s.close()


@pytest.mark.parametrize("pools", [2, 4])
def test_cuda_vec_env_pools_equal_one_pool(pools):
    """GpdVecEnv over several env pools (own streams, ONE shared host mirror): one numpy batch in, one out, bit-identical to
    the single-pool adapter, including terminal observations and episode infos."""
    from gpd_b200.envs import HoverAviary
    from gpd_b200.vec_env import GpdVecEnv
    rng = np.random.default_rng(17)
    E = 256
    v1 = GpdVecEnv(HoverAviary, E, precision="f32")
    vp = GpdVecEnv(HoverAviary, E, num_pools=pools, slide_steps=8, precision="f32")
    o1, op = v1.reset(), vp.reset()
    assert op.shape == (E, 1, 72) and np.array_equal(o1, op)
    ndone = 0
    for t in range(45):
        a = rng.uniform(-1, 1, (E, 1, 4)).astype(np.float32)
        o1, r1, d1, i1 = v1.step(a)
        op, rp, dp, ip = vp.step(a)
        assert np.array_equal(o1, op) and np.array_equal(r1, rp) and np.array_equal(d1, dp), t
        for e in np.nonzero(d1)[0][:6]:
            x, y = i1[int(e)], ip[int(e)]
            assert np.array_equal(x["terminal_observation"], y["terminal_observation"])
            assert x["TimeLimit.truncated"] == y["TimeLimit.truncated"] and x["episode"]["l"] == y["episode"]["l"]
            assert abs(x["episode"]["r"] - y["episode"]["r"]) < 1e-12
            ndone += 1
    assert ndone > 0
    s1, sp = v1.episode_stats(), vp.episode_stats()
    assert s1[0] == sp[0] and s1[2] == sp[2] and s1[6] == sp[6] and abs(s1[1] - sp[1]) <= 1e-6 * abs(s1[1])
    assert s1[4] == sp[4] and s1[5] == sp[5]
    o, r, te, tr = vp.step_tensor(torch.zeros((E, 1, 4), device="cuda"))
    assert o.shape == (E, 1, 72) and r.shape == (E,)
    v1.close(); vp.close()


@pytest.mark.parametrize("shape", ["hover_f32", "hover_f64", "multihover3_f32", "ctrl2_dw_f32", "hoverpid_f32"])
def test_cuda_per_cta_sequencing_is_bit_identical_to_serial_launches(shape, monkeypatch):
    """Programmatic dependent launch + per-CTA step sequencing (the default) against whole-grid stream ordering
    (GPD_TILE_DEP=0 GPD_PDL=0): identical bits after hundreds of back-to-back dependent steps replayed from CUDA graphs,
    on ONE env set (consecutive steps depend on each other tile by tile) with auto-reset and statistics."""
    rng = np.random.default_rng(5)
    cfg = {"hover_f32": (_kw(), 65536, "f32", True), "hover_f64": (_kw(), 20000, "f64", True),
           "multihover3_f32": (_kw("multihover", "rpm", 3), 9000, "f32", True),
           "ctrl2_dw_f32": (_kw("ctrl", "ctrl_rpm", 2, 48, 4), 5000, "f32", False),
           "hoverpid_f32": (_kw(act="pid", freq=48, model=DroneModel.CF2P), 30000, "f32", True)}[shape]
    kw, E, prec, ar = cfg
    fast = make_sim(kw, E, prec, auto_reset=ar)
    fast.set_step_chaining(True)        # the action buffers below are complete long before the first step is enqueued
    monkeypatch.setenv("GPD_TILE_DEP", "0"); monkeypatch.setenv("GPD_PDL", "0")
    slow = make_sim(kw, E, prec, auto_reset=ar)
    monkeypatch.delenv("GPD_TILE_DEP"); monkeypatch.delenv("GPD_PDL")
    A, N = fast.A, fast.N
    if kw["env_kind"] == "ctrl":
        hov = load_drone_params(kw["model"]).HOVER_RPM
        acts = [torch.from_numpy((hov * (1 + 0.05 * rng.uniform(-1, 1, (E, N, A)))).astype(np.float32)).cuda() for _ in range(4)]
    else:
        acts = [torch.from_numpy(rng.uniform(-1, 1, (E, N, A)).astype(np.float32)).cuda() for _ in range(4)]
    outs = []
    for sim in (fast, slow):
        sim.reset()
        for k in range(4):
            sim.step(acts[k])
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for k in range(16):
                    sim.step(acts[k % 4])
        for _ in range(20):
            g.replay()
        torch.cuda.synchronize()
        st = sim.get_state()
        outs.append([x.clone() for x in st] + [sim.obs.clone(), sim.reward.clone(), sim.truncated.clone()] +
                    ([torch.from_numpy(sim.episode_stats())] if ar else []))
    def bits(x):        # NaN-proof bit comparison (a DYN drone has no ground: diverged envs hold inf/NaN in both runs alike)
        return x.contiguous().view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))
    for x, y in zip(*outs):
        assert torch.equal(bits(x), bits(y))
    fast.close(); slow.close()


@pytest.mark.parametrize("N,precision", [(1, "f64"), (2, "f32"), (5, "f64"), (64, "f32"), (64, "f64")])
def test_cuda_adjacency_matches_reference_loop(N, precision):
    """gpd_adjacency / BaseAviary._getAdjacencyMatrix against the restated reference loop (BaseAviary.py:658-675)."""
    from gpd_b200.envs import CtrlAviary
    from oracle import oracle as orc
    rng = np.random.default_rng(N)
    E = 37
    xyz = rng.uniform([-1, -1, 0.2], [1, 1, 1.5], size=(E, N, 3))
    for radius in (0.7, np.inf):
        env = CtrlAviary(num_envs=E, num_drones=N, neighbourhood_radius=radius, initial_xyzs=xyz, pyb_freq=240, ctrl_freq=48,
                         precision=precision)
        adj = env._getAdjacencyMatrix()
        assert adj.shape == (E, N, N)
        pos = env.pos.double().cpu().numpy()        # the positions the kernel saw (float32-rounded in f32 mode)
        want = np.stack([orc.adjacency_matrix(pos[e], radius) for e in range(E)])
        got = adj.double().cpu().numpy()
        if precision == "f64":
            assert np.array_equal(got, want)
        else:                                        # float32 distances: only pairs within rounding of the radius may differ
            d = np.linalg.norm(pos[:, :, None] - pos[:, None], axis=-1)
            assert np.array_equal(got[np.abs(d - radius) > 1e-5], want[np.abs(d - radius) > 1e-5])
        env.close()


def test_cuda_multihover_per_env_targets():
    """Per-env initial poses: every env is rewarded / terminated against ITS OWN targets INIT_XYZS[e] + [0,0,1/(i+1)]
    (MultiHoverAviary.py:71), checked against one single-env oracle per env."""
    from gpd_b200.envs import MultiHoverAviary
    rng = np.random.default_rng(8)
    E, N = 6, 2
    xyz = rng.uniform([-1, -1, 0.2], [1, 1, 1.5], size=(E, N, 3))
    env = MultiHoverAviary(num_envs=E, num_drones=N, initial_xyzs=xyz, precision="f64")
    assert env.TARGET_POS.shape == (E, N, 3)
    refs = []
    for e in range(E):
        kw = _kw("multihover", "rpm", N)
        kw["init_xyz"] = xyz[e]
        from oracle import oracle as orc
        refs.append(orc.OracleSim(load_drone_params(DroneModel.CF2X), 1, num_drones=N, env_kind="multihover", init_xyz=xyz[e],
                                  target_pos=xyz[e] + np.array([[0, 0, 1 / (i + 1)] for i in range(N)])))
    env.reset()
    for t in range(12):
        a = rng.uniform(-1, 1, (E, N, 4)).astype(np.float32)
        obs, rew, term, trunc, _ = env.step(torch.from_numpy(a).cuda())
        for e in range(E):
            _, r_ref, te, tr = refs[e].step(a[e:e + 1])
            assert abs(float(rew[e]) - r_ref[0]) <= 1e-9 * max(1.0, abs(r_ref[0])), (t, e)
            assert bool(term[e]) == bool(te[0]) and bool(trunc[e]) == bool(tr[0])
    env.close()


def test_cuda_episode_stats_through_an_nccl_communicator():
    """gpd_episode_stats(..., ncclComm_t): with a one-rank communicator the job-wide result equals the local one
    (exercises dlopen(libnccl), ncclCommInitRank, the all-gather and the device combine)."""
    kw = _kw()
    sim = make_sim(kw, 2048, "f32", auto_reset=True)
    rng = np.random.default_rng(0)
    for _ in range(40):
        sim.step(torch.from_numpy(rng.uniform(-1, 1, (2048, 1, 4)).astype(np.float32)).cuda())
    local = sim.episode_stats()
    assert local[0] > 0
    L = _lib.load()
    uid = C.create_string_buffer(128)
    _lib.check(L.gpd_nccl_unique_id(uid))
    comm = C.c_void_p()
    _lib.check(L.gpd_nccl_comm_init(uid.raw, 0, 1, 0, C.byref(comm)))
    job = sim.episode_stats(nccl_comm=comm)
    assert np.array_equal(job, local)
    _lib.check(L.gpd_nccl_comm_destroy(comm))
    sim.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_cuda_two_rank_nccl_stats_and_two_devices_in_one_process(tmp_path):
    """world_size 2 over NCCL: job-wide statistics from the in-library reduce equal the torch.distributed all-reduce of the
    per-rank vectors; and one process driving handles on two devices with a > 48 KB shared-memory layout (ADVICE r1)."""
    script = tmp_path / "two_rank.py"
    script.write_text('''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
import gpd_b200
from gpd_b200.distributed import NcclStatsComm, all_reduce_episode_stats
from gpd_b200.envs import HoverAviary
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
env = HoverAviary(num_envs=3000 + 500 * rank, device=local, auto_reset=True)
g = torch.Generator(device="cuda"); g.manual_seed(rank)
for _ in range(30):
    env.step(torch.rand((env.NUM_ENVS, 1, 4), generator=g, device="cuda") * 2 - 1)
mine = env._sim.episode_stats()
want = all_reduce_episode_stats(mine)
comm = NcclStatsComm(device=local)
got = env._sim.episode_stats(nccl_comm=comm.handle)
comm.close()
assert np.allclose(got, want, rtol=1e-12, atol=0), (got, want)
assert got[6] == 30 * (3000 + 3500)
dist.destroy_process_group()
print("rank", rank, "ok")
''' % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", "29533", str(script)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.count("ok") == 2, out.stdout[-1500:] + out.stderr[-3000:]
    # two devices, one process: MultiHover x2 at 30 Hz needs 224*14*16 = 50,176 B of dynamic shared memory per CTA
    from gpd_b200.envs import MultiHoverAviary
    envs = [MultiHoverAviary(num_envs=4096, num_drones=2, device=d, precision="f32") for d in (0, 1)]
    outs = []
    for d, env in enumerate(envs):
        a = torch.zeros((4096, 2, 4), device=f"cuda:{d}")
        with torch.cuda.device(d):
            for _ in range(3):
                o = env.step(a)[0]
            torch.cuda.synchronize()
        outs.append(o.cpu())
    assert torch.equal(outs[0], outs[1])
    for env in envs:
        env.close()


@pytest.mark.parametrize("act,flags,precision,freq,E,direct", [
    # multi-drone envs (MultiHover, in-order per-env sums through shared memory): N rides in the act string as "rpm*3"
    ("rpm*2", 0, "f64", 30, 300, 2), ("rpm*2", 3, "f64", 30, 257, 2), ("rpm*3", 1, "f64", 48, 101, 2), ("pid*2", 0, "f64", 48, 90, 2),
    ("rpm*5", 2, "f32", 30, 77, 2), ("vel*2", 0, "f64", 30, 64, 2),
    ("rpm", 0, "f64", 30, 1000, 2), ("rpm", 0, "f64", 48, 333, 2), ("rpm", 3, "f64", 30, 200, 2), ("vel", 0, "f64", 48, 777, 2),
    ("vel", 2, "f64", 48, 130, 2), ("rpm", 0, "f64", 240, 4096, 2), ("rpm", 0, "f32", 30, 1000, 2), ("rpm", 3, "f32", 30, 517, 2),
    ("vel", 0, "f32", 48, 300, 2),
    # what bypasses shared memory in the bulk kernel (GPD_BULK_DIRECT): 0 = nothing, 1 = the small per-env arrays
    ("rpm", 0, "f64", 30, 1000, 0), ("rpm", 3, "f64", 30, 200, 1), ("vel", 2, "f64", 48, 130, 0), ("rpm", 0, "f32", 30, 1000, 1),
    # actions narrower than a float4: the tile is loaded unshifted and every thread slides its own row in shared memory
    ("pid", 0, "f64", 48, 500, 2), ("pid", 3, "f64", 48, 131, 2), ("one_d_rpm", 0, "f64", 48, 257, 2), ("one_d_pid", 0, "f64", 48, 200, 2),
    ("one_d_rpm", 0, "f64", 240, 100, 2), ("pid", 0, "f32", 48, 300, 2)])
def test_cuda_bulk_copy_path_matches_the_per_thread_path(act, flags, precision, freq, E, direct, monkeypatch):
    """Single-drone RL envs run the bulk-copy data path (gpd_step_bulk.cuh) by default.  Against the
    per-thread / TMA-box kernel (GPD_BULK=0), FP64: identical bits in state, observation, reward, flags, terminal rows and
    episode statistics, with ragged last tiles, per-env initial poses, auto-reset, force models and the in-loop controller,
    a first step without a previous observation and a masked reset.  FP32 (FMA contraction is free to differ between two
    kernels): agreement to a few ulp over a short open-loop horizon; the ring part of the observation is always exact."""
    rng = np.random.default_rng(12)
    f64 = precision == "f64"
    act, _, n = act.partition("*")
    N = int(n or 1)
    kw = _kw("hover" if N == 1 else "multihover", act, N, freq, flags, model=DroneModel.CF2P if act == "vel" else DroneModel.CF2X)
    xyz = rng.uniform([-1, -1, 0.2], [1, 1, 1.5], size=(E, N, 3))
    rpy = rng.uniform(-0.2, 0.2, size=(E, N, 3))
    kw["init_xyz"], kw["init_rpy"] = xyz, rpy
    monkeypatch.setenv("GPD_BULK", "1")           # force the bulk path also where the default would not pick it (240 Hz rows)
    monkeypatch.setenv("GPD_BULK_DIRECT", str(direct))
    bulk = make_sim(kw, E, precision, auto_reset=f64)
    monkeypatch.delenv("GPD_BULK_DIRECT")
    monkeypatch.setenv("GPD_BULK", "0")
    ref = make_sim(kw, E, precision, auto_reset=f64)
    monkeypatch.delenv("GPD_BULK")

    def bits(x):
        return x.contiguous().view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))

    def close(u, v, tag):
        if f64 or not u.dtype.is_floating_point:
            assert torch.equal(bits(u), bits(v)), tag
        else:
            err = ((u.double() - v.double()).abs() / v.double().abs().clamp_min(1.0)).max().item()
            assert err <= 2e-5, (tag, err)

    def same(tag):
        for u, v in zip(bulk.get_state(), ref.get_state()):
            close(u, v, tag)
    # a first step with NO previous observation (all-zero ring), then the regular chain
    A = bulk.A
    a0 = torch.from_numpy(rng.uniform(-1, 1, (E, N, A)).astype(np.float32)).cuda()
    for sim in (bulk, ref):
        sim._have_prev = False
    for u, v in zip(bulk.step(a0)[:2], ref.step(a0)[:2]):
        close(u, v, "first step")
    same("first step")
    for t in range(40 if f64 else 8):
        a = torch.from_numpy(rng.uniform(-1, 1, (E, N, A)).astype(np.float32)).cuda()
        ob, oref = bulk.step(a), ref.step(a)
        for u, v in zip(ob[:2], oref[:2]):
            close(u, v, t)
        assert torch.equal(bits(ob[0][..., 12:]), bits(oref[0][..., 12:])), (t, "ring")
        if f64:
            assert torch.equal(ob[2], oref[2]) and torch.equal(ob[3], oref[3])
            assert torch.equal(bits(bulk.terminal_kin), bits(ref.terminal_kin)), t
        if t % 13 == 5:
            same(t)
        if t == 20:
            m = torch.from_numpy((rng.random(E) < 0.3).astype(np.uint8)).cuda()
            close(bulk.reset(m), ref.reset(m), "masked reset")
    same("end")
    if f64:
        sb, sr = bulk.episode_stats(), ref.episode_stats()
        # counts exactly; the float32 partial sums of the returns are grouped by warp, and the two kernels tile the envs differently
        assert np.array_equal(sb[[0, 2, 6, 7]], sr[[0, 2, 6, 7]]) and (sb[0] > 0 or freq == 240)
        assert np.allclose(sb[[1, 3]], sr[[1, 3]], rtol=1e-6, atol=0) and np.array_equal(sb[[4, 5]], sr[[4, 5]])
    bulk.close(); ref.close()



def test_oracle_matches_the_staged_reference_on_this_box():
    """The CPU arm of bench.py runs the unmodified upstream Python staged under oracle/_ref.  Where that copy exists, replay
    random configurations in it and in the oracle on the GPU machine itself: the checker of every parity test here is then
    pinned to the live upstream code, not only to the committed fixtures.  The upstream sources are not part of this
    repository (__graft_entry__.build() stages them from GPD_REFERENCE)."""
    import json
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref, "gym_pybullet_drones")):
        pytest.skip("needs the upstream gym-pybullet-drones sources, which this repository does not contain: build() "
                    "stages them into oracle/_ref when GPD_REFERENCE points at a checkout of them")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "fuzz_vs_reference.py"), "--ref", ref, "--seeds", "24"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert out.returncode == 0 and lines, out.stderr[-2000:] + out.stdout[-2000:]
    d = json.loads(lines[-1])
    assert d["cases"] == 24 and d["failures"] == []
    assert d["open_loop_worst"] <= 1e-10 and d["closed_loop_worst"] <= 1e-6


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_cuda_chained_stepping_across_eager_and_captured_launches(precision):
    """gpd_set_step_chaining on one stream handle that carries, in turn, eager steps, a CUDA-graph capture, replays of that
    graph, a reset and more eager steps: a step chains only behind a step kernel of the same capture (or of eager work), never
    behind the library's own reset, and the results equal unchained stepping bit for bit."""
    rng = np.random.default_rng(21)
    E = 20000
    kw = _kw()
    chained, plain = make_sim(kw, E, precision, auto_reset=True), make_sim(kw, E, precision, auto_reset=True)
    chained.set_step_chaining(True)
    acts = [torch.from_numpy(rng.uniform(-1, 1, (E, 1, 4)).astype(np.float32)).cuda() for _ in range(4)]
    side = torch.cuda.Stream()
    outs = []
    for sim in (chained, plain):
        sim.reset()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            for k in range(3):
                sim.step(acts[k % 4])                    # eager on the stream the capture will use
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for k in range(6):                       # even count: the observation ping-pong is back where it started
                    sim.step(acts[k % 4])
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            sim.step(acts[1])
            m = torch.from_numpy((rng.random(E) < 0.5).astype(np.uint8)).cuda() if sim is chained else m
            sim.reset(m)                                 # the library's own kernel breaks the chain
            sim.step(acts[2]); sim.step(acts[3])
        torch.cuda.synchronize()
        outs.append([x.clone() for x in sim.get_state()] + [sim.obs.clone(), sim.reward.clone(), torch.from_numpy(sim.episode_stats())])
    for x, y in zip(*outs):
        xi = x.contiguous().view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))
        yi = y.contiguous().view(xi.dtype)
        assert torch.equal(xi, yi)
    chained.close(); plain.close()


def test_cuda_default_tile_sizes():
    """gpd_create's measured layout defaults for the single-drone RL shapes (gpd_grid_size = number of tiles): 128-env tiles for
    lean FP32 sims of 37,888..262,144 envs (both ends included) and for FP64 / force-model sims, 64-env tiles otherwise (profiles/r02/sweep_b14/b16)."""
    L = _lib.load()
    def tiles(E, precision="f32", **over):
        sim = make_sim(_kw(**over), E, precision, auto_reset=True)
        g = L.gpd_grid_size(sim.h)
        sim.close()
        return g
    assert tiles(65536) == 512 and tiles(262144) == 2048 and tiles(37888) == 296
    assert tiles(16384) == 256 and tiles(37887) == 592 and tiles(600000) == 9375 and tiles(262145) == 4097
    assert tiles(65536, act="pid", freq=48, model=DroneModel.CF2P) == 1024        # 3-wide actions: 64-env tiles
    assert tiles(65536, "f64") == 512 and tiles(20000, "f64") == 157
    assert tiles(65536, flags=3) == 512                                            # force models: 128


@pytest.mark.parametrize("E,precision,act", [(56923, "f32", "rpm"), (65536, "f32", "rpm"), (60000, "f32", "pid"), (40000, "f64", "rpm")])
def test_cuda_two_tiles_per_cta_behind_another_handle(E, precision, act, monkeypatch):
    """The benchmark's launch pattern: several handles stepped in rotation on one stream, chained.  A launch behind a step of
    ANOTHER handle runs two tiles per CTA through one buffer (claims up front, a tile published under the next tile's loads;
    FP32, >= 444 tiles) — here with an odd, ragged tile count too.  Against the same rotation launched serially
    (GPD_TILE_DEP=0 GPD_PDL=0): identical bits in state, observation, reward, flags and statistics after 8 graph replays."""
    rng = np.random.default_rng(9)
    kw = _kw(act=act, freq=48 if act == "pid" else 30, model=DroneModel.CF2P if act == "pid" else DroneModel.CF2X)
    nsets = 3
    fast = [make_sim(kw, E, precision, auto_reset=True) for _ in range(nsets)]
    for s_ in fast:
        s_.set_step_chaining(True)
    monkeypatch.setenv("GPD_TILE_DEP", "0"); monkeypatch.setenv("GPD_PDL", "0")
    slow = [make_sim(kw, E, precision, auto_reset=True) for _ in range(nsets)]
    monkeypatch.delenv("GPD_TILE_DEP"); monkeypatch.delenv("GPD_PDL")
    A = fast[0].A
    acts = [torch.from_numpy(rng.uniform(-1, 1, (E, 1, A)).astype(np.float32)).cuda() for _ in range(5)]
    outs = []
    for sims in (fast, slow):
        for s_ in sims:
            s_.reset()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for k in range(4 * nsets):           # an even number of steps per handle: the ping-pong is back where it started
                    sims[k % nsets].step(acts[k % 5])
        for _ in range(8):
            g.replay()
        torch.cuda.synchronize()
        res = []
        for s_ in sims:
            res += [x.clone() for x in s_.get_state()] + [s_.obs.clone(), s_.reward.clone(), s_.truncated.clone(),
                                                            torch.from_numpy(s_.episode_stats())]
        outs.append(res)

    def bits(x):
        return x.contiguous().view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))
    for x, y in zip(*outs):
        assert torch.equal(bits(x), bits(y))
    for s_ in fast + slow:
        s_.close()
