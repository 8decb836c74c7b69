"""Reference half of the planning-gradient tests (tests/test_gpu_plan_grad.py, tests/test_plan_grad_cpu.py): the LEAN
Physics.DYN control step (BaseAviary.py:831-889 with the RPM / ONE_D_RPM action map), the Hover / MultiHover reward and
flags (HoverAviary.py:68-117, MultiHoverAviary.py:84-130) and plan_ref.plan_returns' recurrence, restated in torch FP64
so that autograd differentiates them.

Two rules make the restatement's derivative the one gpd_plan_grad documents (include/gpd.h), while its values stay the
reference's:
  * the action map rpm = HOVER_RPM * (1 + 0.05 a) is evaluated in float32 as the reference does, with the derivative of
    the smooth map (0.05 in float32, times HOVER_RPM);
  * _integrateQ is differentiated as its smooth update cos(theta) I + (sin(theta)/|w|) Lambda(w), by its power series
    for small theta; where |w| <= 1e-8 the value is the reference's unchanged quaternion."""
import math

import numpy as np
import torch

from plan_ref import plan_returns
from state_edges import max_counter

C005 = float(np.float32(0.05))


class LeanRef:
    """One configuration: ``drone`` (gpd_b200.params.DroneParams), ``kw`` a state_edges-style shape dict (env_kind,
    action_type, num_drones, pyb_freq, ctrl_freq, episode_len_sec)."""

    def __init__(self, drone, kw):
        self.d = drone
        self.model = str(getattr(drone.model, "value", drone.model)).lower()
        self.multi = kw["env_kind"] == "multihover"
        self.one_d = kw["action_type"] == "one_d_rpm"
        self.S = kw["pyb_freq"] // kw["ctrl_freq"]
        self.dt = 1.0 / kw["pyb_freq"]
        self.max_counter = max_counter(kw["episode_len_sec"], kw["pyb_freq"])
        self.J = [float(drone.J[i][i]) for i in range(3)]
        self.JI = [float(drone.J_INV[i][i]) for i in range(3)]

    # ---- _preprocessAction and the rotor terms (BaseRLAviary.py:212-229, BaseAviary.py:838-851) ----
    def rpm(self, a):
        """a (..., A) float64 holding float32 values -> rpm (..., 4); the value is the float32 map's."""
        a32 = a.detach().float()
        u = torch.tensor(0.05, dtype=torch.float32, device=a.device) * a32
        u = (u + torch.tensor(1.0, dtype=torch.float32, device=a.device)).double()
        r = self.d.HOVER_RPM * (u + C005 * (a - a.detach()))
        return r[..., :1].expand(*r.shape[:-1], 4) if self.one_d else r

    def forcing(self, rpm):
        d = self.d
        f = rpm * rpm * d.KF
        zt = rpm * rpm * d.KM
        if self.model == "racer":
            zt = -zt
        f0, f1, f2, f3 = f.unbind(-1)
        T = f0 + ((f1 + f2) + f3)
        tz = -zt[..., 0] + zt[..., 1] - zt[..., 2] + zt[..., 3]
        if self.model == "cf2p":
            tx, ty = (f1 - f3) * d.L, (-f0 + f2) * d.L
        else:
            arm = d.L / math.sqrt(2)
            tx, ty = (f0 + f1 - f2 - f3) * arm, (-f0 + f1 + f2 - f3) * arm
        return T, torch.stack([tx, ty, tz], -1)

    # ---- one DYN substep (BaseAviary.py:831-874) ----
    def substep(self, p, q, v, w, T, tau):
        d, dt = self.d, self.dt
        x, y, z, qw = q.unbind(-1)
        s = 2.0 / (x * x + y * y + z * z + qw * qw)
        col = torch.stack([s * (x * z + qw * y), s * (y * z - qw * x), 1.0 - s * (x * x + y * y)], -1)
        F = col * T[..., None] - torch.tensor([0.0, 0.0, d.GRAVITY], dtype=p.dtype, device=p.device)
        J = torch.tensor(self.J, dtype=p.dtype, device=p.device)
        JI = torch.tensor(self.JI, dtype=p.dtype, device=p.device)
        w1 = w + dt * (JI * (tau - torch.cross(w, J * w, dim=-1)))
        v1 = v + dt * (F / d.M)
        p1 = p + dt * v1
        m = torch.stack([torch.stack([1.0 - s * (y * y + z * z), s * (x * y - qw * z), s * (x * z + qw * y)], -1),
                         torch.stack([s * (x * y + qw * z), 1.0 - s * (x * x + z * z), s * (y * z - qw * x)], -1),
                         torch.stack([s * (x * z - qw * y), s * (y * z + qw * x), col[..., 2]], -1)], -2)
        av = (m @ w1[..., None])[..., 0]
        return p1, self.integrate_q(q, w1), v1, w1, av

    def integrate_q(self, q, w):
        h = self.dt / 2
        n2 = (w * w).sum(-1)
        t = n2 * (h * h)
        small = t < 0.01
        ts = torch.where(small, torch.ones_like(t), t)
        th = torch.sqrt(ts)
        cs = torch.where(small, 1 + t * (-1 / 2 + t * (1 / 24 + t * (-1 / 720 + t / 40320))), torch.cos(th))
        sc = torch.where(small, h * (1 + t * (-1 / 6 + t * (1 / 120 + t * (-1 / 5040 + t / 362880)))),
                         h * torch.sin(th) / th)
        ap, aq, ar = (w * sc[..., None]).unbind(-1)
        x, y, z, qw = q.unbind(-1)
        q1 = torch.stack([cs * x + ar * y - aq * z + ap * qw, -ar * x + cs * y + ap * z + aq * qw,
                          aq * x - ap * y + cs * z + ar * qw, -ap * x - aq * y - ar * z + cs * qw], -1)
        still = (torch.sqrt(n2) <= 1e-8)[..., None]          # BaseAviary.py:879: the value is q itself
        return q1 + torch.where(still, q - q1, torch.zeros_like(q1)).detach()

    @staticmethod
    def euler(q):
        """pybullet getEulerFromQuaternion (roll, pitch, yaw)."""
        x, y, z, w = q.unbind(-1)
        sarg = -2 * (x * z - w * y)
        roll = torch.atan2(2 * (y * z + w * x), w * w - x * x - y * y + z * z)
        pitch = torch.asin(sarg.clamp(-1, 1))
        yaw = torch.atan2(2 * (x * y + w * z), w * w + x * x - y * y - z * z)
        lo, hi = sarg <= -0.99999, sarg >= 0.99999
        zero = torch.zeros_like(roll)
        roll = torch.where(lo | hi, zero, roll)
        pitch = torch.where(lo, zero - math.pi / 2, torch.where(hi, zero + math.pi / 2, pitch))
        yaw = torch.where(lo, 2 * torch.atan2(x, -y), torch.where(hi, 2 * torch.atan2(-x, y), yaw))
        return torch.stack([roll, pitch, yaw], -1)

    # ---- a control step and the plan ----
    def step(self, st, a, target):
        """st: dict p, q, v, w of shape (E, N, .); a (E, N, A) float64; target (E, N, 3).  Returns the next state (with
        rpy and ang_v), the (E,) reward and the terminated / truncated flags before the counter rule."""
        T, tau = self.forcing(self.rpm(a))
        p, q, v, w = st["p"], st["q"], st["v"], st["w"]
        for _ in range(self.S):
            p, q, v, w, av = self.substep(p, q, v, w, T, tau)
        rpy = self.euler(q)
        e = target - p
        dist = torch.sqrt((e * e).sum(-1))
        val = 2 - (dist * dist) ** 2
        r_i = torch.where(val > 0, val, torch.zeros_like(val))
        lim = 2.0 if self.multi else 1.5
        tr = ((p[..., 0].abs() > lim) | (p[..., 1].abs() > lim) | (p[..., 2] > 2.0) | (rpy[..., 0].abs() > .4) |
              (rpy[..., 1].abs() > .4)).any(-1)
        if self.multi:
            rew, term = r_i.sum(-1), dist.sum(-1) < 1e-4
        else:
            rew, term = r_i[..., 0], dist[..., 0] < 1e-4
        return dict(p=p, q=q, v=v, w=w, rpy=rpy, av=av), rew, term, tr

    def plan(self, st, counter, actions, target, gamma):
        """K steps of actions (K, E, N, A) (float64 holding float32 values, may require grad) from st / counter (E,) ->
        (returns (E,), done_step (E,), per-step states, rewards (K, E), terminated (K, E), truncated (K, E))."""
        cnt = counter.clone().long()
        rews, terms, truncs, states = [], [], [], []
        for k in range(actions.shape[0]):
            st, r, te, tr = self.step(st, actions[k], target)
            tr = tr | (cnt > self.max_counter)
            cnt = cnt + self.S
            states.append(st)
            rews.append(r)
            terms.append(te)
            truncs.append(tr)
        rew, term, trunc = torch.stack(rews), torch.stack(terms), torch.stack(truncs)
        G, done = plan_returns(rew, term | trunc, gamma)
        return G, done, states, rew, term, trunc


def start_state(state20, rpy_rates):
    """The restatement's state dict from exported state20 (E, N, 20) and rpy_rates (E, N, 3), float64 tensors."""
    return dict(p=state20[..., 0:3], q=state20[..., 3:7], v=state20[..., 10:13], w=rpy_rates)


def central_difference(G, a):
    """dG/da at a[0] from G at the actions a[0], a[0] + h, a[0] - h (float32).  The float32 action map rounds
    u = 1 + 0.05 a, so the two steps in u differ; the three-point formula on the steps it really took stays O(h^2)."""
    u = (np.float32(1) + np.float32(0.05) * np.asarray(a, np.float32)).astype(np.float64)
    d1, d2 = u[1] - u[0], u[0] - u[2]
    du = (d2 * d2 * (G[1] - G[0]) + d1 * d1 * (G[0] - G[2])) / (d1 * d2 * (d1 + d2))
    return du * C005
