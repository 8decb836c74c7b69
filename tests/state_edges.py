"""Seeded off-nominal states for the step kernels (tests/test_state_edges_cpu.py, tests/test_gpu_state_edges.py).

Every family is a function ``(rng, kw, E, precision) -> dict`` with
    state20 (E,N,20), rpy_rates (E,N,3), pid_state (E,N,9) float64; step_counter (E,) int32;
    actions (2,E,N,A) for two ctrl steps (float32; float64 values of the command for the Ctrl env);
    bands: names of the FP32 exemption bands the family may touch; groups: name -> env indices of one boundary.
It places E envs on, and on both sides of, one branch of the kernels (gpd_math.cuh, gpd_kernels.cuh, gpd_step_bulk.cuh).
For ``precision == "f32"`` the arrays are rounded to float32 before anything is derived from them (the kernel sees exactly
these values and so does the oracle), and boundary values are placed with float32 neighbours.  state20[7:10] is always the
oracle's Euler angles of the (rounded) quaternion: the reference keeps them in the state (BaseAviary.py:518) and the VEL
controller reads the yaw from there.
"""
import numpy as np

from helpers import default_targets
from gpd_b200.params import load_drone_params
from gpd_b200.utils.enums import DroneModel
from oracle import oracle as orc

A_WIDTH = {"rpm": 4, "one_d_rpm": 1, "pid": 3, "vel": 4, "one_d_pid": 1, "ctrl_rpm": 4, "ctrl_vel": 4}
SARG_T = 0.99999
SARG_T32 = float(np.float32(0.99999))

# (pyb_freq, ctrl_freq) and the kernel variant each shape reaches (gpd_api.cu picks the kernel; GPD_BULK=0 forces gpd::step_kernel)
SHAPES = {
    "hover30": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "hover48": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=240, ctrl_freq=48, physics_flags=0),
    "hover60_20": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=60, ctrl_freq=20, physics_flags=0),
    "hover240": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=240, ctrl_freq=240, physics_flags=0),
    "one_d_rpm": dict(env_kind="hover", action_type="one_d_rpm", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "gnd": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=1),
    "gnd_drag": dict(env_kind="hover", action_type="rpm", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=3),
    "pid": dict(env_kind="hover", action_type="pid", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "vel": dict(env_kind="hover", action_type="vel", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "one_d_pid": dict(env_kind="hover", action_type="one_d_pid", num_drones=1, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "multi3": dict(env_kind="multihover", action_type="rpm", num_drones=3, pyb_freq=240, ctrl_freq=30, physics_flags=0),
    "multi3_gd": dict(env_kind="multihover", action_type="rpm", num_drones=3, pyb_freq=240, ctrl_freq=30, physics_flags=3),
    "ctrl3_dw": dict(env_kind="ctrl", action_type="ctrl_rpm", num_drones=3, pyb_freq=240, ctrl_freq=48, physics_flags=7),
    "ctrl1": dict(env_kind="ctrl", action_type="ctrl_rpm", num_drones=1, pyb_freq=240, ctrl_freq=48, physics_flags=0),
}


def shape(name, **over):
    kw = dict(SHAPES[name], model=DroneModel.CF2X, init_xyz=None, init_rpy=None, episode_len_sec=8.0)
    kw.update(over)
    return kw


def max_counter(episode_len_sec, pyb_freq):
    """Largest step_counter with step_counter / PYB_FREQ <= EPISODE_LEN_SEC in Python float arithmetic (HoverAviary.py:114)."""
    k = int(np.floor(episode_len_sec * pyb_freq))
    while k > 0 and k / pyb_freq > episode_len_sec:
        k -= 1
    while (k + 1) / pyb_freq <= episode_len_sec:
        k += 1
    return k


# ---------------------------------------------------------------------------------------------------------------------
def shoemake(rng, n):
    """Uniform random unit quaternions (x, y, z, w)."""
    u1, u2, u3 = rng.random(n), rng.random(n), rng.random(n)
    a, b = np.sqrt(1 - u1), np.sqrt(u1)
    return np.stack([a * np.sin(2 * np.pi * u2), a * np.cos(2 * np.pi * u2), b * np.sin(2 * np.pi * u3),
                     b * np.cos(2 * np.pi * u3)], -1)


def quat(rpy):
    rpy = np.asarray(rpy, np.float64).reshape(-1, 3)
    return np.array([orc.quaternion_from_euler(r) for r in rpy])


def euler(q):
    q = np.asarray(q, np.float64).reshape(-1, 4)
    return np.array([orc.euler_from_quaternion(x) for x in q])


def sarg(q, dt=np.float64):
    """The argument of asin in quat_to_euler, formed in `dt` in the kernels' order: -2 * (x*z - w*y)."""
    q = np.asarray(q).astype(dt)
    x, y, z, w = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    return dt(-2) * (x * z - w * y)


def gimbal_quats(precision, offsets=(1e-15, 1e-9, 3e-6, 1e-5, 5e-5)):
    """Pure-pitch quaternions (with a yaw twist) whose sarg straddles +-0.99999 (and float32(0.99999) in FP32)."""
    out = []
    for thr in ((SARG_T32,) if precision == "f32" else (SARG_T,)):
        for off in offsets:
            for sgn in (-1, 1):
                s = thr * (1 + sgn * off)
                p = np.arcsin(min(s, 1.0))
                for pm in (1, -1):
                    out.append(quat([0.0, pm * p, 0.3 * sgn])[0])
    out.append(quat([0.0, np.pi / 2, 0.0])[0])
    out.append(quat([0.0, -np.pi / 2, 1.0])[0])
    return np.array(out)


def special_attitudes(precision):
    """roll = +-pi and neighbours, yaw = +-pi, roll = +-pi/2: fast_atan2f's x < 0 and |y| > |x| quadrants.  Roll = +-pi/2
    exactly only in FP64: in float32 the sign of atan2's x there (and with it the ground-effect gate) is a rounding residue."""
    rpy = []
    for r in (np.pi, -np.pi, np.pi - 1e-7, -np.pi + 1e-7, np.pi - 1e-3, -np.pi + 1e-3):
        rpy.append([r, 0.1, 0.2])
    for y in (np.pi, -np.pi, np.pi - 1e-6, -np.pi + 1e-6):
        rpy.append([0.05, -0.1, y])
    for r in ((np.pi / 2, -np.pi / 2) if precision == "f64" else ()) + (np.pi / 2 + 1e-3, -np.pi / 2 - 1e-3, np.pi / 2 - 1e-3):
        rpy.append([r, 0.2, -2.5])
    return quat(rpy)


def _hover_rpm(kw):
    return load_drone_params(kw["model"]).HOVER_RPM


def _balanced_action(kw, E, N):
    """Equal rotor speeds: zero torque (RPM action 0, HOVER_RPM for ctrl_rpm)."""
    A = A_WIDTH[kw["action_type"]]
    if kw["action_type"] == "ctrl_rpm":
        return np.full((2, E, N, A), _hover_rpm(kw))
    return np.zeros((2, E, N, A), np.float32)


def _random_action(rng, kw, E, N, scale=1.0):
    A = A_WIDTH[kw["action_type"]]
    if kw["action_type"] == "ctrl_rpm":
        return _hover_rpm(kw) * (1 + 0.05 * scale * rng.uniform(-1, 1, (2, E, N, A)))
    return (scale * rng.uniform(-1, 1, (2, E, N, A))).astype(np.float32)


def _positions(rng, kw, E, N):
    """Inside the Hover box; multi-drone envs on a height ladder whose gaps (0.15-0.35 m) stay clear of the downwash
    singularities (delta_z -> 0 and beta = 0 at 0.6875 m, DESIGN 3.6)."""
    xyz = np.stack([rng.uniform(-.8, .8, (E, N)), rng.uniform(-.8, .8, (E, N)), rng.uniform(0.3, 1.5, (E, N))], -1)
    if N > 1:
        z = np.array([0.2, 0.4, 0.55, 0.75, 0.9, 1.05])[None, :N] + rng.uniform(0, 0.01, (E, N))
        xyz[..., 2] = np.take_along_axis(z, np.argsort(rng.random((E, N)), axis=1), axis=1)
        xyz[..., :2] = rng.uniform(-.15, .15, (E, N, 2))
    return xyz


def assemble(kw, E, precision, pos, q, vel=None, rates=None, rpm_prev=None, pid_state=None, counter=None, actions=None,
             bands=(), groups=None):
    N = kw["num_drones"]
    z3 = np.zeros((E, N, 3))
    st = np.zeros((E, N, 20))
    st[..., 0:3] = pos
    st[..., 3:7] = q
    st[..., 10:13] = z3 if vel is None else vel
    if rpm_prev is not None:
        st[..., 16:20] = rpm_prev
    rr = z3.copy() if rates is None else np.array(rates, np.float64)
    ps = np.zeros((E, N, 9)) if pid_state is None else np.array(pid_state, np.float64)
    acts = np.asarray(actions)
    if precision == "f32":          # the kernel sees these float32 values; the oracle is handed exactly the same ones
        st, rr, ps = (x.astype(np.float32).astype(np.float64) for x in (st, rr, ps))
        if kw["env_kind"] == "ctrl":
            acts = acts.astype(np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        st[..., 7:10] = euler(st[..., 3:7]).reshape(E, N, 3)
    cnt = np.zeros(E, np.int32) if counter is None else np.asarray(counter, np.int32)
    return dict(state20=st, rpy_rates=rr, pid_state=ps, step_counter=cnt, actions=acts, bands=tuple(bands),
                groups=groups or {})


# ---------------------------------------------------------------------------------------------------------------------
THETAS = (0.1, 0.2 * (1 - 1e-5), 0.2 * (1 + 1e-5), 0.35, 0.5 * (1 - 1e-5), 0.5 * (1 + 1e-5), 0.6, 0.9, 1.6, 3.0)
TINY_RATES = (0.0, 5e-9, 1e-8, 2e-8)


def f1_rates(rng, kw, E, precision):
    """Body rates across the quaternion-update switches: t = |w|^2 (dt/2)^2 = theta^2 against 0.04 (lean_substep_f32) and
    0.25 (integrate_q<float>), the reference's |w| <= 1e-8 early return, then generic directions with random actions."""
    N = kw["num_drones"]
    dt = 1.0 / kw["pyb_freq"]
    pos = _positions(rng, kw, E, N)
    q = shoemake(rng, E * N).reshape(E, N, 4)
    rates = np.zeros((E, N, 3))
    acts = _balanced_action(kw, E, N)
    mags = [2 * th / dt for th in THETAS] + list(TINY_RATES)
    k = 0
    for m in mags:                                  # one principal axis each: zero torque and zero gyroscopic term
        for ax in range(3):
            if k < E:
                rates[k, :, ax] = m * (1 if (k % 2) else -1)
                k += 1
    # generic directions in the body x-y plane (Jx = Jy: no gyroscopic term, which at these rates makes the explicit
    # Euler update of the reference amplify any rounding), within 1 % of a switch: the rotor torques move |w| across it
    n_gen = E - k
    th = rng.choice([0.2, 0.5], n_gen) * (1 + rng.uniform(-0.01, 0.01, n_gen))
    phi = rng.uniform(0, 2 * np.pi, (n_gen, N))
    d = np.stack([np.cos(phi), np.sin(phi), np.zeros_like(phi)], -1)
    rates[k:] = d * (2 * th / dt)[:, None, None]
    acts[:, k:] = _random_action(rng, kw, n_gen, N)
    return assemble(kw, E, precision, pos, q, rates=rates, actions=acts, bands=("rpy", "flags"),
                    groups={"axis": np.arange(k), "generic": np.arange(k, E)})


def _attitudes(rng, E, precision, extra_gimbal=True):
    q = [special_attitudes(precision)]
    if extra_gimbal:
        q.append(gimbal_quats(precision))
    q = np.concatenate(q)
    n = E - len(q)
    rnd = shoemake(rng, (n + 1) // 2)
    rnd = np.concatenate([rnd, -rnd])[:n]
    return np.concatenate([q, rnd]), len(q)


def f2_attitudes(rng, kw, E, precision):
    """Any attitude: Shoemake quaternions (each also as -q), roll/yaw at +-pi, roll at +-pi/2, and pitch with sarg
    straddling the gimbal threshold.  The placed envs keep their attitude through the step (zero rates, equal rotors)."""
    N = kw["num_drones"]
    qa, n_fixed = _attitudes(rng, E * N, precision)
    q = qa.reshape(E, N, 4)
    rates = np.zeros((E, N, 3))
    acts = _balanced_action(kw, E, N)
    nf = (n_fixed + N - 1) // N                     # envs holding at least one placed attitude
    rates[nf:] = rng.uniform(-3, 3, (E - nf, N, 3))
    acts[:, nf:] = _random_action(rng, kw, E - nf, N)
    return assemble(kw, E, precision, _positions(rng, kw, E, N), q, rates=rates, actions=acts,
                    bands=("rpy", "flags"), groups={"fixed": np.arange(nf)})


NORMS = (0.5, 0.9, 0.99, 1.01, 1.1, 2.0)


def f3_quat_norm(rng, kw, E, precision):
    """|q| != 1 (the reference never renormalises, quirk 13): F2 attitudes scaled to NORMS, which also pushes |sarg| past 1
    where the gimbal branch has to catch it."""
    d = f2_attitudes(rng, kw, E, precision)
    N = kw["num_drones"]
    scale = np.asarray(NORMS)[np.arange(E * N) % len(NORMS)].reshape(E, N, 1)
    q = d["state20"][..., 3:7].reshape(-1, 4).copy()
    if precision == "f32":
        # a unit attitude at gimbal lock scaled below 1 leaves the gimbal branch with atan2(0, 0) for roll and yaw: the
        # reference's angles are then rounding residues, which float32 cannot reproduce
        lock = (np.abs(sarg(q)) > 0.999) & (scale.reshape(-1) < 1)
        q[lock] = shoemake(rng, int(lock.sum()))
    q = q * scale.reshape(-1, 1)
    placed = [v * quat([0.0, pm * np.arcsin(SARG_T * (1 + off) / v ** 2), 0.4])[0]      # v^2 sin(pitch) around 0.99999
              for v in NORMS if v > 1 for off in (-1e-4, 6e-6, 1e-4) for pm in (1, -1)]
    q[:len(placed)] = placed
    q = q.reshape(E, N, 4)
    st = d["state20"]
    return assemble(kw, E, precision, st[..., 0:3], q, rates=d["rpy_rates"], actions=d["actions"], bands=("rpy", "flags"),
                    groups={"norm": np.arange(E)})


def f4_ground(rng, kw, E, precision):
    """The in-step ground-effect gate (signs of the atan2/asin arguments) on any attitude, the rotor heights below, at and
    above GND_EFF_H_CLIP; large velocities with the previous RPM in state20[16:20] (drag of the first substep)."""
    N = kw["num_drones"]
    dp = load_drone_params(kw["model"])
    qa = np.concatenate([gimbal_quats(precision, offsets=(1e-4, 1e-3)), special_attitudes(precision),
                         quat([[0, 0, 0], [0.2, -0.1, 1.0], [-0.3, 0.2, -2.0]])])
    n = E * N - len(qa)
    rnd = shoemake(rng, n)
    q = np.concatenate([qa, rnd]).reshape(E, N, 4)
    pos = _positions(rng, kw, E, N)
    clip = dp.GND_EFF_H_CLIP
    low = np.array([0.0, 0.5 * clip, clip, clip * (1 + 1e-12), 1.5 * clip, 3 * clip, 0.1, 0.3])
    if N == 1:
        pos[..., 2] = low[np.arange(E) % len(low)][:, None]
    else:                                            # lowest drone near the ground, the others on the ladder above it
        pos[..., 2] = low[np.arange(E) % len(low)][:, None] + np.array([0.0, 0.15, 0.3, 0.45, 0.6, 0.75])[None, :N]
    vel = rng.uniform(-5, 5, (E, N, 3))
    rpm_prev = dp.HOVER_RPM * rng.uniform(0.5, 1.5, (E, N, 4))
    rates = rng.uniform(-2, 2, (E, N, 3))
    return assemble(kw, E, precision, pos, q, vel=vel, rates=rates, rpm_prev=rpm_prev,
                    actions=_random_action(rng, kw, E, N), bands=("rpy", "flags"), groups={"all": np.arange(E)})


def _nb(x, precision, k):
    """k-th neighbour of x in the precision's floating-point grid (k < 0: below)."""
    dt = np.float32 if precision == "f32" else np.float64
    v = dt(x)
    for _ in range(abs(k)):
        v = np.nextafter(v, dt(np.inf) if k > 0 else dt(-np.inf))
    return float(v)


EPISODE_LENS = (8.0, 7.3, 1 / 3, 5.000000000000001, 0.1 * 3)


def f5_episode_end(rng, kw, E, precision):
    """Hover / MultiHover flags at their thresholds: |x|, |y| at 1.5 (2.0) and one ulp beyond, z at 2.0 +- 1e-9, roll and
    pitch around 0.4, target distance at 1e-4 +- 1e-12, step_counter at max_counter - S, max_counter, max_counter + 1.
    Identity or fixed attitudes with zero rates and hover RPM: x, y and the attitude do not move during the step."""
    N = kw["num_drones"]
    S = kw["pyb_freq"] // kw["ctrl_freq"]
    lim = 1.5 if kw["env_kind"] == "hover" else 2.0
    tgt = default_targets(dict(kw, model=kw["model"]))
    mc = max_counter(kw["episode_len_sec"], kw["pyb_freq"])
    pos = np.broadcast_to(tgt + np.array([0.3, -0.2, -0.4]), (E, N, 3)).copy()
    rpy = np.zeros((E, N, 3))
    cnt = np.zeros(E, np.int64)
    groups = {}
    e = 0

    def take(name, n):
        nonlocal e
        idx = np.arange(e, e + n)
        groups[name] = idx
        e += n
        return idx
    vals = [_nb(s * lim, precision, k) for s in (1, -1) for k in (-1, 0, 1)]
    for ax in (0, 1):
        idx = take("xy%d" % ax, len(vals))
        pos[idx, -1, ax] = vals                      # the last drone of the env sits on the boundary
    zv = [2.0, 2.0 + 1e-9, 2.0 - 1e-9] if precision == "f64" else [2.0, _nb(2.0, precision, 1), _nb(2.0, precision, -1)]
    idx = take("z", len(zv))
    pos[idx, -1, 2] = zv
    # FP32: only offsets outside the 1e-5 flag band (inside it the kernel's float32 roll may fall either way)
    ang = [0.4 + s * d for s in (1, -1) for d in ((1e-15, 1e-12, 1e-9, 2e-5, 1e-4) if precision == "f64" else (2e-5, 1e-4))]
    for ax in (0, 1):
        idx = take("rp%d" % ax, 2 * len(ang))
        rpy[idx[:len(ang)], -1, ax] = ang
        rpy[idx[len(ang):], -1, ax] = -np.asarray(ang)
    if kw["env_kind"] == "hover":                   # distance to target (0, 0, 1): along z
        if precision == "f64":
            dz = [1e-4 + s * d for s in (1, -1) for d in (1e-12, 1e-13, 1e-9)]
            zz = [1.0 - x for x in dz]
        else:
            zz = [_nb(1 - 1e-4, precision, k) for k in (-2, -1, 0, 1, 2)]
        idx = take("dist", len(zz))
        pos[idx, 0, :2] = 0.0
        pos[idx, 0, 2] = zz
    else:                                           # sum of the drones' distances: all at their targets but one
        d = [1e-4 * (1 + s * f) for s in (1, -1) for f in ((1e-8, 1e-12) if precision == "f64" else (1e-3,))]
        idx = take("dist", len(d))
        pos[idx] = tgt
        pos[idx, -1, 2] = tgt[-1, 2] + np.asarray(d)
    idx = take("counter", 3 * 3)
    for j, c in enumerate((mc - S, mc, mc + 1)):
        cnt[idx[3 * j:3 * j + 3]] = c
    cnt[e:] = S * rng.integers(0, max(1, (mc - 2 * S) // S), E - e)
    assert e <= E, (e, E)
    q = quat(rpy.reshape(-1, 3)).reshape(E, N, 4)
    return assemble(kw, E, precision, pos, q, counter=cnt, actions=_balanced_action(kw, E, N), bands=("flags",),
                    groups=groups)


def f6_controller(rng, kw, E, precision):
    """DSLPID in the step: yaw and last_rpy across +-pi (rate_e is not wrapped, the torque saturates at +-3200),
    integrators at and beyond their clips, inverted drones (sthr <= 0), PID destinations at distance exactly 1, VEL actions
    with a zero direction or a negative speed fraction."""
    N = kw["num_drones"]
    A = A_WIDTH[kw["action_type"]]
    pos = _positions(rng, kw, E, N)
    rpy = rng.uniform(-0.2, 0.2, (E, N, 3))
    ps = np.zeros((E, N, 9))
    ps[..., 6:9] = rpy + rng.uniform(-0.01, 0.01, (E, N, 3))
    groups = {}
    k = E // 8
    yaw = np.concatenate([np.array([np.pi, -np.pi]), np.pi - np.geomspace(1e-3, 0.3, k - 2) * rng.choice([-1, 1], k - 2)])
    yaw = np.where(yaw > np.pi, yaw - 2 * np.pi, yaw)
    rpy[:k, :, 2] = yaw[:, None]
    ps[:k, :, 8] = -yaw[:, None] * rng.uniform(0.99, 1.0, (k, 1))      # last yaw on the other side of +-pi
    groups["yaw_wrap"] = np.arange(k)
    clips = np.array([[2, 2, .15, 1, 1, 1500], [2.5, -3, .2, 1.2, -1.5, 1600], [-2, -2, -.15, -1, -1, -1500],
                      [1.9, -1.9, .1, .9, -.9, 1000], [0.5, 0.5, 0.05, 0.3, 0.3, 100], [-2.5, 3, -.2, -1.2, 1.5, -1600]])
    idx = np.arange(k, 2 * k)
    ps[idx, :, 0:6] = clips[np.arange(k) % len(clips)][:, None, :]
    groups["clips"] = idx
    idx = np.arange(2 * k, 3 * k)
    rpy[idx, :, 0] = np.pi - rng.uniform(0, 0.5, (k, N))                # inverted: sthr <= 0
    groups["inverted"] = idx
    q = quat(rpy.reshape(-1, 3)).reshape(E, N, 4)
    vel = rng.uniform(-1, 1, (E, N, 3))
    rates = rng.uniform(-1, 1, (E, N, 3))
    acts = rng.uniform(-1, 1, (2, E, N, A)).astype(np.float32)
    if kw["action_type"] == "pid":                  # destinations at distance exactly 1 (and one ulp beyond)
        idx = np.arange(3 * k, 3 * k + 8)
        pos[idx] = np.array([0.25, -0.5, 0.5])
        for j, e in enumerate(idx):
            acts[:, e] = np.array([0.25, -0.5, 1.5], np.float32) if j % 2 == 0 else np.array(
                [0.25, -0.5, np.nextafter(np.float32(1.5), np.float32(2))], np.float32)
        groups["dist1"] = idx
    elif kw["action_type"] == "vel":
        idx = np.arange(3 * k, 4 * k)
        acts[:, idx[: k // 2], :, 0:3] = 0.0                            # zero direction
        acts[:, idx[k // 2:], :, 3] = -np.abs(acts[:, idx[k // 2:], :, 3])   # negative speed fraction
        groups["vel_edge"] = idx
    return assemble(kw, E, precision, pos, q, vel=vel, rates=rates, pid_state=ps, actions=acts, bands=("rpy", "flags", "yaw"),
                    groups=groups)


def f7_values(rng, kw, E, precision):
    """RPM actions of +-0.0, +-1, +-30 (negative RPM at -30: not clipped, drag changes sign), ctrl_rpm below 0 and above
    MAX_RPM, and one drone with a NaN and one with an Inf in its state."""
    N = kw["num_drones"]
    dp = load_drone_params(kw["model"])
    pos = _positions(rng, kw, E, N)
    q = shoemake(rng, E * N).reshape(E, N, 4) * np.sign(rng.uniform(-1, 1, (E, N, 1)))
    rates = rng.uniform(-2, 2, (E, N, 3))
    vel = rng.uniform(-1, 1, (E, N, 3))
    A = A_WIDTH[kw["action_type"]]
    if kw["action_type"] == "ctrl_rpm":
        vals = np.array([-1.0, -0.0, 0.0, dp.MAX_RPM, dp.MAX_RPM * 1.5, 1e9, dp.HOVER_RPM])
    else:
        vals = np.array([0.0, -0.0, 1.0, -1.0, 30.0, -30.0], np.float32)
    acts = vals[rng.integers(0, len(vals), (2, E, N, A))]
    if kw["action_type"] != "ctrl_rpm":
        acts = acts.astype(np.float32)
    rpm_prev = dp.HOVER_RPM * rng.uniform(-0.5, 1.5, (E, N, 4))
    nan_env, inf_env = E // 3, (2 * E) // 3
    pos[nan_env, 0, 0] = np.nan
    pos[inf_env, 0, 2] = np.inf
    return assemble(kw, E, precision, pos, q, vel=vel, rates=rates, rpm_prev=rpm_prev, actions=acts, bands=("rpy", "flags"),
                    groups={"nonfinite": np.array([nan_env, inf_env])})


FAMILIES = {"F1": f1_rates, "F2": f2_attitudes, "F3": f3_quat_norm, "F4": f4_ground, "F5": f5_episode_end,
            "F6": f6_controller, "F7": f7_values}


def oracle_sim(kw, E, init_xyz=None, init_rpy=None):
    from gpd_b200.params import default_pid_params
    dp = load_drone_params(kw["model"])
    pid = default_pid_params(DroneModel.CF2X) if kw["action_type"] in ("pid", "vel", "one_d_pid", "ctrl_vel") else None
    return orc.OracleSim(dp, E, num_drones=kw["num_drones"], env_kind=kw["env_kind"], action_type=kw["action_type"],
                         pyb_freq=kw["pyb_freq"], ctrl_freq=kw["ctrl_freq"], physics_flags=kw["physics_flags"],
                         pid_params=pid, init_xyz=init_xyz, init_rpy=init_rpy, target_pos=default_targets(kw),
                         episode_len_sec=kw["episode_len_sec"])


def inject_oracle(ref, fam):
    ref.state20[...] = fam["state20"]
    ref.rpy_rates[...] = fam["rpy_rates"]
    ref.pid_state[...] = fam["pid_state"]
    ref.step_counter[...] = fam["step_counter"]
