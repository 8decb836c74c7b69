"""Batched ``BaseAviary``: the reference's ``reset()``/``step()`` contract on ``Physics.DYN``.

Mirrors reference ``envs/BaseAviary.py`` (constructor ``:25-40``, constants ``:74-128``, initial poses
``:194-207``, ``reset`` ``:220-255``, ``step`` ``:259-383``, ``_getDroneStateVector`` ``:541-561``)
with a leading batch axis: one instance simulates ``num_envs`` independent copies of the reference
environment on one GPU.  All arithmetic of the step runs in the fused CUDA kernel behind
``gpd_step`` (include/gpd.h); this class only owns buffers and metadata.

Differences from the reference, all forced by scope:
  * only ``Physics.DYN`` and the DYN-form composites (``Physics.DYN_GND`` ...) exist; the PyBullet
    solver modes raise ``ValueError``; ``gui``/``record``/RGB observations raise ``NotImplementedError``;
  * arrays carry the batch axis: obs ``(E, N, W)``, reward/terminated/truncated ``(E,)``;
  * ``step`` takes/returns CUDA tensors (zero-copy) or numpy arrays (host path, copies inside).
"""
from __future__ import annotations

import time

import numpy as np
import torch

from ..params import load_drone_params
from ..sim import BatchedSim
from ..utils.enums import PHYSICS_FLAGS, DroneModel, Physics


class BaseAviary:
    ENV_KIND = "ctrl"

    def __init__(self,
                 drone_model: DroneModel = DroneModel.CF2X,
                 num_drones: int = 1,
                 neighbourhood_radius: float = np.inf,
                 initial_xyzs=None,
                 initial_rpys=None,
                 physics: Physics = Physics.DYN,
                 pyb_freq: int = 240,
                 ctrl_freq: int = 240,
                 gui=False,
                 record=False,
                 obstacles=False,
                 user_debug_gui=True,
                 vision_attributes=False,
                 output_folder='results',
                 num_envs: int = 1,
                 device: int = 0,
                 precision: str = "f32",
                 auto_reset: bool = False,
                 threads_per_block: int = 0):
        #### Constants (BaseAviary.py:74-83) #######################
        self.G = 9.8
        self.RAD2DEG = 180 / np.pi
        self.DEG2RAD = np.pi / 180
        self.CTRL_FREQ = ctrl_freq
        self.PYB_FREQ = pyb_freq
        if self.PYB_FREQ % self.CTRL_FREQ != 0:
            raise ValueError('[ERROR] in BaseAviary.__init__(), pyb_freq is not divisible by env_freq.')
        self.PYB_STEPS_PER_CTRL = int(self.PYB_FREQ / self.CTRL_FREQ)
        self.CTRL_TIMESTEP = 1. / self.CTRL_FREQ
        self.PYB_TIMESTEP = 1. / self.PYB_FREQ
        self.NUM_DRONES = num_drones
        self.NUM_ENVS = int(num_envs)
        self.NEIGHBOURHOOD_RADIUS = neighbourhood_radius
        self.DRONE_MODEL = drone_model
        if gui or record or vision_attributes:
            raise NotImplementedError("GUI, video recording and vision observations need the PyBullet renderer: out of scope")
        if physics not in PHYSICS_FLAGS:
            raise ValueError(f"{physics} steps PyBullet's rigid-body solver, which is out of scope: use Physics.DYN "
                             "or a DYN-form composite (Physics.DYN_GND, DYN_DRAG, DYN_DW, DYN_GND_DRAG_DW)")
        self.GUI, self.RECORD = False, False
        self.PHYSICS = physics
        self.OBSTACLES = obstacles
        self.USER_DEBUG = user_debug_gui
        self.URDF = self.DRONE_MODEL.value + ".urdf"
        self.OUTPUT_FOLDER = output_folder
        #### Drone properties (BaseAviary.py:97-128) ###############
        p = load_drone_params(drone_model, self.G)
        self.PARAMS = p
        (self.M, self.L, self.THRUST2WEIGHT_RATIO, self.J, self.J_INV, self.KF, self.KM, self.COLLISION_H,
         self.COLLISION_R, self.COLLISION_Z_OFFSET, self.MAX_SPEED_KMH, self.GND_EFF_COEFF, self.PROP_RADIUS,
         self.DRAG_COEFF, self.DW_COEFF_1, self.DW_COEFF_2, self.DW_COEFF_3) = self._parseURDFParameters()
        self.GRAVITY = p.GRAVITY
        self.HOVER_RPM = p.HOVER_RPM
        self.MAX_RPM = p.MAX_RPM
        self.MAX_THRUST = p.MAX_THRUST
        self.MAX_XY_TORQUE = p.MAX_XY_TORQUE
        self.MAX_Z_TORQUE = p.MAX_Z_TORQUE
        self.GND_EFF_H_CLIP = p.GND_EFF_H_CLIP
        #### Initial poses (BaseAviary.py:194-207); (N,3) like the reference or (E,N,3) per env ####
        N, E = self.NUM_DRONES, self.NUM_ENVS
        if initial_xyzs is None:
            self.INIT_XYZS = np.vstack([np.array([x * 4 * self.L for x in range(N)]),
                                        np.array([y * 4 * self.L for y in range(N)]),
                                        np.ones(N) * (self.COLLISION_H / 2 - self.COLLISION_Z_OFFSET + .1)]
                                       ).transpose().reshape(N, 3)
        elif np.array(initial_xyzs).shape in ((N, 3), (E, N, 3)):
            self.INIT_XYZS = np.array(initial_xyzs, dtype=np.float64)
        else:
            raise ValueError("invalid initial_xyzs in BaseAviary.__init__(), try initial_xyzs.reshape(NUM_DRONES,3)")
        if initial_rpys is None:
            self.INIT_RPYS = np.zeros(self.INIT_XYZS.shape)
        elif np.array(initial_rpys).shape == self.INIT_XYZS.shape:
            self.INIT_RPYS = np.array(initial_rpys, dtype=np.float64)
        else:
            raise ValueError("invalid initial_rpys in BaseAviary.__init__(), try initial_rpys.reshape(NUM_DRONES,3)")
        #### Spaces and the device-side simulation ################
        self.action_space = self._actionSpace()
        self.observation_space = self._observationSpace()
        self._sim = BatchedSim(p, E, N, env_kind=self.ENV_KIND, action_type=self._actionCode(), pyb_freq=pyb_freq,
                               ctrl_freq=ctrl_freq, physics_flags=PHYSICS_FLAGS[physics], precision=precision,
                               device=device, auto_reset=auto_reset, target_pos=self._sharedTargets(),
                               episode_len_sec=getattr(self, "EPISODE_LEN_SEC", 8.0),
                               threads_per_block=threads_per_block)
        self._sim.set_init_poses(self.INIT_XYZS, self.INIT_RPYS)
        tp = self._targetPositions()
        if tp is not None and np.ndim(tp) == 3:          # per-env initial poses: every env has its own targets
            self._sim.set_targets(tp)
        self._sim.reset()
        self.RESET_TIME = time.time()
        self._host_out = None
        self._state_cache = None
        self._numpy_io = False      # the last step took numpy actions: reset() then answers in numpy too

    ################################################################################
    def reset(self, seed: int = None, options: dict = None, as_numpy: bool | None = None):
        """Resets every env (BaseAviary.py:220-255; ``seed`` is ignored there too).  Returns ``(obs, info)``.
        The observation is a numpy array when the env is being stepped with numpy actions (or ``as_numpy=True``), else a
        CUDA tensor.  Both kinds of step share ONE device observation chain, so the action ring survives the reset
        (BaseRLAviary.py:153-154) whichever way the env was stepped."""
        self.RESET_TIME = time.time()
        self._state_cache = None
        if as_numpy is None:
            as_numpy = self._numpy_io
        if as_numpy:
            return self._sim.reset_host(), self._computeInfo()
        return self._sim.reset(), self._computeInfo()

    def reset_envs(self, mask):
        """Resets only the envs with ``mask[e]`` set (device bool/uint8 tensor); returns the full observation."""
        self._state_cache = None
        return self._sim.reset(torch.as_tensor(mask))

    def step(self, action):
        """One control step of every env (BaseAviary.py:259-383).

        ``action``: CUDA tensor -> returns CUDA tensors (views of internal buffers, no copies);
        numpy array -> host path (H2D/D2H inside), returns numpy arrays.
        """
        self._state_cache = None
        if isinstance(action, np.ndarray):
            if self._host_out is None:
                self._host_out = self._sim.alloc_host_outputs(pinned=torch.cuda.is_available())
                self._host_flags = (self._host_out[2].view(np.bool_), self._host_out[3].view(np.bool_))
            self._numpy_io = True
            obs, rew = self._sim.step_host(action, self._host_out)[:2]
            return obs, rew, self._host_flags[0], self._host_flags[1], self._computeInfo()
        self._numpy_io = False
        obs, rew, term, trunc = self._sim.step(action)
        return obs, rew, term.view(torch.bool), trunc.view(torch.bool), self._computeInfo()

    def rollout(self, actions, return_traj: bool = False):
        """K control steps of a given action schedule in one launch: the same as ``for k: step(actions[k])`` when the
        intermediate observations are not read.  ``actions``: CUDA tensor (K, E, N, A).  Returns ``(obs, rewards,
        terminated, truncated, info)``: the observation after the last step, rewards / flags of shape (K, E) (bool flags);
        ``info["traj"]`` holds each step's kinematic part (K, E, N, 12) (the whole (K, E, N, 20) row for the Ctrl env)
        when ``return_traj``."""
        self._state_cache = None
        self._numpy_io = False
        out = self._sim.rollout(actions, traj=return_traj)
        obs, rew, term, trunc = out[:4]
        info = self._computeInfo()
        if return_traj:
            info = dict(info, traj=out[4])
        return obs, rew, term.view(torch.bool), trunc.view(torch.bool), info

    def plan(self, actions, gamma: float = 1.0, targets=None, reward: bool = False, final_kin: bool = False,
             out: dict | None = None) -> dict:
        """Scores S candidate schedules per env from its current state without advancing the env (MPPI, CEM, random
        shooting).  ``actions``: CUDA tensor (K, E, S, N, A).  Returns ``{"returns": (E, S), "done_step": (E, S)}``, plus
        ``reward`` (K, E, S) and ``final_kin`` (E, S, N, 12) when asked for; see ``BatchedSim.plan``.  The env, its
        observation and its episode statistics are left as they were."""
        return self._sim.plan(actions, gamma=gamma, targets=targets, reward=reward, final_kin=final_kin, out=out)

    def plan_grad(self, actions, gamma: float = 1.0, targets=None, out: dict | None = None) -> dict:
        """``plan``'s returns and done_step together with ``grad`` (K, E, S, N, A), the gradient of each candidate's
        return with respect to its actions (gradient-based shooting MPC), without advancing the env.  Physics.DYN with
        RPM or ONE_D_RPM actions only; see ``BatchedSim.plan_grad`` and ``BatchedSim.plan_return``."""
        return self._sim.plan_grad(actions, gamma=gamma, targets=targets, out=out)

    def render(self, mode='human', close=False):
        """Text output of env 0 (BaseAviary.py:387-412)."""
        st = self._state()[0][0].cpu().numpy()
        cnt = int(self._state()[3][0])
        print("[INFO] BaseAviary.render() --- it {:04d}".format(cnt),
              "--- wall-clock time {:.1f}s,".format(time.time() - self.RESET_TIME),
              "simulation time {:.1f}s@{:d}Hz".format(cnt * self.PYB_TIMESTEP, self.PYB_FREQ))
        for i in range(self.NUM_DRONES):
            print("[INFO] BaseAviary.render() --- drone {:d}".format(i),
                  "--- x {:+06.2f}, y {:+06.2f}, z {:+06.2f}".format(*st[i, 0:3]),
                  "--- velocity {:+06.2f}, {:+06.2f}, {:+06.2f}".format(*st[i, 10:13]),
                  "--- roll {:+06.2f}, pitch {:+06.2f}, yaw {:+06.2f}".format(*(st[i, 7:10] * self.RAD2DEG)),
                  "--- angular velocity {:+06.4f}, {:+06.4f}, {:+06.4f} --- ".format(*st[i, 13:16]))

    def close(self):
        self._sim.close()

    def getPyBulletClient(self):
        return -1   # there is no Bullet client behind this env

    def getDroneIds(self):
        return np.arange(1, self.NUM_DRONES + 1)

    ################################################################################
    def _state(self):
        if self._state_cache is None:
            self._state_cache = self._sim.get_state()
        return self._state_cache

    def _getDroneStateVector(self, nth_drone):
        """(E, 20) state of the n-th drone of every env (BaseAviary.py:541-561)."""
        return self._state()[0][:, nth_drone, :]

    pos = property(lambda self: self._state()[0][:, :, 0:3])
    quat = property(lambda self: self._state()[0][:, :, 3:7])
    rpy = property(lambda self: self._state()[0][:, :, 7:10])
    vel = property(lambda self: self._state()[0][:, :, 10:13])
    ang_v = property(lambda self: self._state()[0][:, :, 13:16])
    last_clipped_action = property(lambda self: self._state()[0][:, :, 16:20])
    rpy_rates = property(lambda self: self._state()[1])
    step_counter = property(lambda self: self._state()[3])

    def _parseURDFParameters(self):
        """Same 17-tuple as the reference (BaseAviary.py:982-1014)."""
        return self.PARAMS.urdf_tuple()

    def _getAdjacencyMatrix(self):
        """(E, N, N) adjacency (BaseAviary.py:658-675)."""
        return self._sim.adjacency(self.NEIGHBOURHOOD_RADIUS)       # gpd_adjacency: per-env position tile in shared memory

    def _calculateNextStep(self, current_position, destination, step_size=1):
        """Intermediate waypoint at most ``step_size`` from the current position (BaseAviary.py:1105-1147);
        batched over the leading axes: (..., 3) tensors."""
        cur = torch.as_tensor(current_position)
        dest = torch.as_tensor(destination, dtype=cur.dtype, device=cur.device)
        direction = dest - cur
        distance = torch.linalg.norm(direction, dim=-1, keepdim=True)
        nxt = cur + direction / distance.clamp_min(torch.finfo(cur.dtype).tiny) * step_size
        return torch.where(distance <= step_size, dest.expand_as(cur), nxt)

    def checkpoint(self):
        """Everything needed to resume bit-exactly: integrator state, controller state, counters and the current
        observation (which carries the action ring)."""
        st, rr, ps, cnt = self._sim.get_state()
        return {"state20": st.clone(), "rpy_rates": rr.clone(), "pid_state": ps.clone(), "step_counter": cnt.clone(),
                "obs": self._sim.obs.clone()}

    def restore(self, ckpt):
        sim = self._sim
        sim.set_state(ckpt["state20"], ckpt["rpy_rates"], ckpt["pid_state"], ckpt["step_counter"])
        sim.adopt_obs(ckpt["obs"])          # also marks a host mirror stale: it is rebuilt from this observation
        self._state_cache = None

    #### hooks of the subclasses (BaseAviary.py:1018-1101) ############################
    def _actionSpace(self):
        raise NotImplementedError

    def _observationSpace(self):
        raise NotImplementedError

    def _actionCode(self) -> str:
        raise NotImplementedError

    def _targetPositions(self):
        return None

    def _sharedTargets(self):
        """(N,3) targets for ``gpd_create`` (per-env targets, if any, are uploaded with ``gpd_set_targets``)."""
        tp = self._targetPositions()
        return None if tp is None else (tp if np.ndim(tp) == 2 else tp[0])

    def _computeInfo(self):
        return {"answer": 42}
