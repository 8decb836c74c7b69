"""``BatchedSim`` — thin host wrapper of one ``gpd_sim`` handle (``include/gpd.h``).

PyTorch is used only for device memory and streams: every I/O buffer is a caller-visible
CUDA tensor handed to the C ABI as a raw pointer (zero-copy).  The observation is kept in a
ping-pong pair because the RL observation carries the action ring (reference
``BaseRLAviary.py:317-318``): step k reads the history from the buffer step k-1 wrote.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from .params import DroneParams, PIDParams, default_pid_params
from .utils.enums import DroneModel


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _plan_inputs(sim, actions, targets):
    """The checks ``plan`` and ``plan_grad`` share: actions (K, E, S, N, A) in the action dtype on the device, targets."""
    if sim.is_ctrl:
        raise ValueError("the Ctrl env has no reward to plan on")
    if actions.dim() != 5 or tuple(actions.shape[1:2] + actions.shape[3:]) != (sim.E, sim.N, sim.A) or \
            actions.shape[0] < 1 or actions.shape[2] < 1:
        raise ValueError(f"actions must have shape (K, {sim.E}, S, {sim.N}, {sim.A}), got {tuple(actions.shape)}")
    K, S = int(actions.shape[0]), int(actions.shape[2])
    if actions.dtype != sim.act_dtype or not actions.is_cuda or not actions.is_contiguous():
        actions = actions.to(device=sim.device, dtype=sim.act_dtype).contiguous()
    if targets is not None and (tuple(targets.shape) != (sim.E, sim.N, 3) or targets.dtype != sim.real or
                                not targets.is_contiguous()):
        raise ValueError(f"targets must be a contiguous ({sim.E}, {sim.N}, 3) tensor of {sim.real}")
    return actions, K, S


def _plan_outputs(out, want, targets):
    """Output buffers of ``plan`` / ``plan_grad``: ``want`` maps each name to its (shape, dtype)."""
    for name, (shape, dt) in want.items():
        t = out.get(name)
        if t is None or tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"out[{name!r}] must be a contiguous {shape} tensor of {dt}")
    if not all(t.is_cuda for t in [out[n] for n in want] + ([] if targets is None else [targets])):
        raise ValueError("targets and the output buffers must be CUDA tensors")


class _PlanReturn(torch.autograd.Function):
    """``BatchedSim.plan_return``: forward ``gpd_plan_grad``'s returns, backward its gradient."""

    @staticmethod
    def forward(ctx, sim, actions, gamma, targets):
        res = sim.plan_grad(actions.detach(), gamma=gamma, targets=targets)
        ctx.save_for_backward(res["grad"])
        ctx.act_dtype = actions.dtype
        return res["returns"]

    @staticmethod
    def backward(ctx, grad_output):
        (grad,) = ctx.saved_tensors
        return None, (grad_output[None, :, :, None, None] * grad).to(ctx.act_dtype), None, None


class HostMirror:
    """Feature-major observation log in pinned host memory (``gpd_mirror_alloc``; layout in ``include/gpd.h``).

    ``log[row][col]``: row = observation feature, col = drone.  The observation of the current step is the strided view
    ``obs(e, n, j) = log[first_row + j][col0 + e*N + n]`` — shape ``(E, N, W)``, strides ``(4N, 4, 4*row_len)`` bytes, the
    transpose of a dense ``[W][D]`` block.  One mirror may serve several sims (env pools in lockstep) through different
    ``col0``.  The pinned block is released when the last numpy view of it is gone."""

    def __init__(self, W: int, A: int, row_len: int, slide_steps: int = 128):
        self.lib = _lib.load()
        self.W, self.A, self.row_len = int(W), int(A), int(row_len)
        self.rows = self.W + self.A * max(1, int(slide_steps))
        base = C.c_void_p()
        _lib.check(self.lib.gpd_mirror_alloc(self.rows, self.row_len, C.byref(base)))
        self.base = base
        self._buf = (C.c_float * (self.rows * self.row_len)).from_address(base.value)
        weakref.finalize(self._buf, self.lib.gpd_mirror_free, C.c_void_p(base.value))

    def view(self, first_row: int, E: int, N: int, col0: int = 0) -> np.ndarray:
        return np.ndarray((E, N, self.W), dtype=np.float32, buffer=self._buf,
                          offset=(int(first_row) * self.row_len + int(col0)) * 4,
                          strides=(4 * N, 4, 4 * self.row_len))


class BatchedSim:
    def __init__(self, drone: DroneParams, num_envs: int, num_drones: int = 1, env_kind: str = "hover",
                 action_type: str = "rpm", pyb_freq: int = 240, ctrl_freq: int = 30, physics_flags: int = 0,
                 precision: str = "f32", device: int = 0, auto_reset: bool = False, pid: PIDParams | None = None,
                 target_pos=None, episode_len_sec: float = 8.0, init_xyz=None, init_rpy=None,
                 threads_per_block: int = 0):
        self.lib = _lib.load()
        if precision not in ("f32", "f64"):
            raise ValueError("precision must be 'f32' or 'f64'")
        if pyb_freq % ctrl_freq != 0:
            raise ValueError('[ERROR] in BaseAviary.__init__(), pyb_freq is not divisible by env_freq.')
        self.E, self.N = int(num_envs), int(num_drones)
        self.env_kind, self.action_type = env_kind, action_type
        self.is_ctrl = env_kind == "ctrl"
        self.precision = precision
        self.real = torch.float64 if precision == "f64" else torch.float32
        self.np_real = np.float64 if precision == "f64" else np.float32
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        self.auto_reset = bool(auto_reset)
        self.physics_flags = int(physics_flags)
        cfg = _lib.ConfigC()
        cfg.device = self.device_index
        cfg.precision = _lib.GPD_F64 if precision == "f64" else _lib.GPD_F32
        cfg.num_envs, cfg.num_drones = self.E, self.N
        cfg.pyb_freq, cfg.ctrl_freq = int(pyb_freq), int(ctrl_freq)
        cfg.env_kind = _lib.ENV_CODES[env_kind]
        cfg.action_type = _lib.ACT_CODES[action_type]
        cfg.physics_flags = int(physics_flags)
        cfg.auto_reset = int(self.auto_reset)
        cfg.threads_per_block = int(threads_per_block)
        cfg.episode_len_sec = float(episode_len_sec)
        cfg.speed_limit = 0.03 * drone.MAX_SPEED_KMH * (1000 / 3600)       # BaseRLAviary.py:95
        cfg.drone = _lib.drone_params_c(drone)
        if pid is None and drone.model in (DroneModel.CF2X, DroneModel.CF2P):
            # in-env controllers are CF2X even for a CF2P env (BaseRLAviary.py:75-76); the pid.py-style rollout
            # passes the drone's own model explicitly
            pid = default_pid_params(DroneModel.CF2X)
        if pid is not None:
            cfg.pid = _lib.pid_params_c(pid)
        self._target = None
        if target_pos is not None:
            self._target = np.ascontiguousarray(np.asarray(target_pos, dtype=np.float64).reshape(self.N, 3))
            cfg.target_pos = self._target.ctypes.data_as(C.POINTER(C.c_double))
        h = C.c_void_p()
        _lib.check(self.lib.gpd_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.A = self.lib.gpd_action_width(h)
        self.W = self.lib.gpd_obs_width(h)
        self.S = self.lib.gpd_substeps(h)
        self.B = 0 if self.is_ctrl else ctrl_freq // 2
        self.act_dtype = self.real if self.is_ctrl else torch.float32
        self.obs_dtype = self.real if self.is_ctrl else torch.float32
        with torch.cuda.device(self.device):
            self.obs_buf = [torch.zeros((self.E, self.N, self.W), dtype=self.obs_dtype, device=self.device)
                            for _ in range(2)]
            self.reward = torch.zeros(self.E, dtype=self.real, device=self.device)
            self.terminated = torch.zeros(self.E, dtype=torch.uint8, device=self.device)
            self.truncated = torch.zeros(self.E, dtype=torch.uint8, device=self.device)
            self.terminal_kin = (torch.zeros((self.E, self.N, 12), dtype=torch.float32, device=self.device)
                                 if self.auto_reset and not self.is_ctrl else None)
        self._cur = 0
        self._have_prev = False
        self._mirror = None
        self._mirror_col0 = 0
        self._row = C.c_int64(0)
        # the step path re-uses these ctypes pointers (the buffers never move): eager stepping is host-bound at 65k envs
        self._p_obs = [_ptr(b) for b in self.obs_buf]
        self._p_out = (_ptr(self.reward), _ptr(self.terminated), _ptr(self.truncated), _ptr(self.terminal_kin))
        if init_xyz is not None or init_rpy is not None:
            self.set_init_poses(init_xyz, init_rpy)
            self.reset()

    # ------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_step_chaining(self, enable: bool = True):
        """Chained stepping (gpd_set_step_chaining, default off): back-to-back step() calls of one stream overlap across the
        kernel boundary, each tile waiting only for its own previous step.  Only valid when the actions of every step
        were complete before the PREVIOUS kernel of the stream was enqueued (a pre-computed action schedule, action repeat,
        independent env sets stepped in rotation) — never behind the policy kernel that computes them."""
        _lib.check(self.lib.gpd_set_step_chaining(self.h, int(bool(enable))))

    def set_targets(self, target_pos):
        """TARGET_POS (HoverAviary.py:51, MultiHoverAviary.py:71): (N,3) shared by every env or (E,N,3) per env."""
        t = np.ascontiguousarray(np.asarray(target_pos, dtype=np.float64))
        per_env = t.ndim == 3
        if t.shape != ((self.E, self.N, 3) if per_env else (self.N, 3)):
            raise ValueError("target_pos must have shape (N,3) or (E,N,3)")
        _lib.check(self.lib.gpd_set_targets(self.h, t.ctypes.data_as(C.POINTER(C.c_double)), int(per_env)))

    def set_init_poses(self, xyz, rpy):
        """initial_xyzs / initial_rpys (BaseAviary.py:194-207): (N,3) for all envs or (E,N,3) per env."""
        xyz = np.asarray(xyz, dtype=np.float64)
        rpy = np.zeros_like(xyz) if rpy is None else np.asarray(rpy, dtype=np.float64)
        per_env = xyz.ndim == 3
        shape = (self.E, self.N, 3) if per_env else (self.N, 3)
        if xyz.shape != shape or rpy.shape != shape:
            raise ValueError(f"initial poses must have shape {shape}")
        xyz, rpy = np.ascontiguousarray(xyz), np.ascontiguousarray(rpy)
        dp = C.POINTER(C.c_double)
        _lib.check(self.lib.gpd_set_init_poses(self.h, xyz.ctypes.data_as(dp), rpy.ctypes.data_as(dp), int(per_env)))

    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        """BaseAviary.reset for the masked envs (None = all); returns the observation of every env."""
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        nxt = self._cur ^ 1
        prev = self.obs_buf[self._cur] if self._have_prev else None
        _lib.check(self.lib.gpd_reset(self.h, _ptr(mask), _ptr(prev), _ptr(self.obs_buf[nxt]), self._stream()))
        self._cur, self._have_prev = nxt, True
        return self.obs_buf[nxt]

    def step(self, actions: torch.Tensor):
        """One BaseAviary.step on device tensors.  Returns views of internal buffers: the observation stays
        valid until the step after next (ping-pong); reward/terminated/truncated until the next step."""
        if actions.dtype != self.act_dtype or not actions.is_cuda or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=self.act_dtype).contiguous()
        if actions.numel() != self.E * self.N * self.A:
            raise ValueError(f"actions must have {self.E}x{self.N}x{self.A} elements, got {tuple(actions.shape)}")
        nxt = self._cur ^ 1
        rc = self.lib.gpd_step(self.h, C.c_void_p(actions.data_ptr()), self._p_obs[self._cur] if self._have_prev else None,
                               self._p_obs[nxt], *self._p_out, self._stream())
        if rc:
            _lib.check(rc)
        self._cur, self._have_prev = nxt, True
        return self.obs_buf[nxt], self.reward, self.terminated, self.truncated

    def step_into(self, actions: torch.Tensor, obs_prev: torch.Tensor, obs_out: torch.Tensor, reward: torch.Tensor,
                  terminated: torch.Tensor, truncated: torch.Tensor):
        """``gpd_step`` on caller-owned buffers (the C ABI's ownership model, SURVEY 8b): reads the action ring from
        ``obs_prev``, writes the new observation to ``obs_out`` and the per-env outputs in place.  A trajectory buffer
        ``obs[t] -> obs[t + 1]`` can thus be the observation chain itself (no per-step copies; ``rollout.py``).  The
        internal ping-pong buffers are not touched: call ``adopt_obs`` before going back to ``step``."""
        for t, dt in ((actions, self.act_dtype), (obs_prev, self.obs_dtype), (obs_out, self.obs_dtype), (reward, self.real),
                      (terminated, torch.uint8), (truncated, torch.uint8)):
            if t.dtype != dt or not t.is_cuda or not t.is_contiguous():
                raise ValueError("step_into needs contiguous CUDA tensors of the sim's dtypes")
        if obs_prev.numel() != self.E * self.N * self.W or obs_out.numel() != obs_prev.numel():
            raise ValueError("observation buffers must hold E x N x W elements")
        if reward.numel() != self.E or terminated.numel() != self.E or truncated.numel() != self.E:
            raise ValueError("reward / terminated / truncated must hold E elements")
        if actions.numel() != self.E * self.N * self.A:
            raise ValueError(f"actions must have {self.E}x{self.N}x{self.A} elements, got {tuple(actions.shape)}")
        _lib.check(self.lib.gpd_step(self.h, _ptr(actions), _ptr(obs_prev), _ptr(obs_out), _ptr(reward), _ptr(terminated),
                                     _ptr(truncated), self._p_out[3], self._stream()))

    def alloc_rollout_outputs(self, n_steps: int, traj: bool = False, terminal_kin: bool = False) -> dict:
        """Caller-owned per-step output buffers for ``rollout(..., out=...)``: reward / terminated / truncated (K, E), and
        ``traj`` / ``terminal_kin`` when asked for.  Reused across rollouts, a graph-captured planner loop allocates nothing."""
        K, E, N = int(n_steps), self.E, self.N
        kw = dict(device=self.device)
        out = {"reward": torch.zeros((K, E), dtype=self.real, **kw),
               "terminated": torch.zeros((K, E), dtype=torch.uint8, **kw),
               "truncated": torch.zeros((K, E), dtype=torch.uint8, **kw)}
        if traj:
            out["traj"] = (torch.zeros((K, E, N, 20), dtype=self.real, **kw) if self.is_ctrl
                           else torch.zeros((K, E, N, 12), dtype=torch.float32, **kw))
        if terminal_kin:
            out["terminal_kin"] = torch.zeros((K, E, N, 12), dtype=torch.float32, **kw)
        return out

    def rollout(self, actions: torch.Tensor, traj: bool = False, terminal_kin: bool = False, out: dict | None = None):
        """``gpd_rollout``: K = ``actions.shape[0]`` control steps of the schedule ``actions`` (K, E, N, A) in one launch, the
        same as K ``step`` calls whose intermediate observations are not read.  The final observation lands in the internal
        ping-pong, as with ``step``.  Returns ``(obs, rewards (K,E), terminated (K,E), truncated (K,E))``, then ``traj``
        ((K,E,N,12) kin rows, (K,E,N,20) for the Ctrl env) and ``terminal_kin`` ((K,E,N,12), written only where an env
        finished; auto-reset RL envs) when asked for.  ``out``: buffers from ``alloc_rollout_outputs``, written in place."""
        if actions.dtype != self.act_dtype or not actions.is_cuda or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=self.act_dtype).contiguous()
        per_step = self.E * self.N * self.A
        if actions.numel() == 0 or actions.numel() % per_step != 0:
            raise ValueError(f"actions must have shape (K, {self.E}, {self.N}, {self.A}), got {tuple(actions.shape)}")
        K = actions.numel() // per_step
        if out is None:
            out = self.alloc_rollout_outputs(K, traj, terminal_kin)
        for name in ("reward", "terminated", "truncated") + (("traj",) if traj else ()) + (("terminal_kin",) if terminal_kin else ()):
            t = out[name]
            if t.shape[0] != K or not t.is_cuda or not t.is_contiguous():
                raise ValueError(f"out[{name!r}] must be a contiguous CUDA tensor with K = {K} rows")
        tr = out["traj"] if traj else None
        tk = out["terminal_kin"] if terminal_kin else None
        nxt = self._cur ^ 1
        _lib.check(self.lib.gpd_rollout(self.h, int(K), _ptr(actions), self._p_obs[self._cur] if self._have_prev else None,
                                        self._p_obs[nxt], _ptr(out["reward"]), _ptr(out["terminated"]),
                                        _ptr(out["truncated"]), _ptr(tr), _ptr(tk), self._stream()))
        self._cur, self._have_prev = nxt, True
        res = (self.obs_buf[nxt], out["reward"], out["terminated"], out["truncated"])
        if traj:
            res += (tr,)
        if terminal_kin:
            res += (tk,)
        return res

    def alloc_plan_outputs(self, n_steps: int, n_samples: int, reward: bool = False, final_kin: bool = False) -> dict:
        """Caller-owned output buffers for ``plan(..., out=...)``: returns and done_step (E, S), and reward (K, E, S) /
        final_kin (E, S, N, 12) when asked for.  Reused across plans, a graph-captured planner loop allocates nothing."""
        K, S, E, N = int(n_steps), int(n_samples), self.E, self.N
        kw = dict(device=self.device)
        out = {"returns": torch.zeros((E, S), dtype=self.real, **kw),
               "done_step": torch.zeros((E, S), dtype=torch.int32, **kw)}
        if reward:
            out["reward"] = torch.zeros((K, E, S), dtype=self.real, **kw)
        if final_kin:
            out["final_kin"] = torch.zeros((E, S, N, 12), dtype=torch.float32, **kw)
        return out

    def plan(self, actions: torch.Tensor, gamma: float = 1.0, targets: torch.Tensor | None = None, reward: bool = False,
             final_kin: bool = False, out: dict | None = None) -> dict:
        """``gpd_plan``: scores S candidate schedules per env from its current state, without advancing the env.
        ``actions`` (K, E, S, N, A): sample s of env e runs K control steps of ``actions[:, e, s]`` on a copy of env e, with
        no auto-reset.  Returns a dict with ``returns`` (E, S) (discounted by ``gamma``, up to and including the step that
        ends the episode) and ``done_step`` (E, S) (that step, K if none), plus ``reward`` (K, E, S) and ``final_kin``
        (E, S, N, 12) (the kin part of the last step's observation) when asked for.  ``targets`` (E, N, 3): target
        positions for this plan only.  ``out``: buffers from ``alloc_plan_outputs``, written in place."""
        actions, K, S = _plan_inputs(self, actions, targets)
        if out is None:
            out = self.alloc_plan_outputs(K, S, reward, final_kin)
        want = {"returns": ((self.E, S), self.real), "done_step": ((self.E, S), torch.int32)}
        if reward:
            want["reward"] = ((K, self.E, S), self.real)
        if final_kin:
            want["final_kin"] = ((self.E, S, self.N, 12), torch.float32)
        _plan_outputs(out, want, targets)
        _lib.check(self.lib.gpd_plan(self.h, K, S, _ptr(actions), _ptr(targets), float(gamma), _ptr(out["returns"]),
                                     _ptr(out["done_step"]), _ptr(out.get("reward") if reward else None),
                                     _ptr(out.get("final_kin") if final_kin else None), self._stream()))
        return {name: out[name] for name in want}

    def plan_grad_tape_bytes(self, n_steps: int, n_samples: int) -> int:
        """Bytes of the workspace ``plan_grad`` needs for ``n_steps`` x ``n_samples`` copies of every env."""
        b = self.lib.gpd_plan_grad_tape_bytes(self.h, int(n_steps), int(n_samples))
        _lib.check(b if b < 0 else 0)
        return int(b)

    def alloc_plan_grad_outputs(self, n_steps: int, n_samples: int) -> dict:
        """Caller-owned buffers for ``plan_grad(..., out=...)``: returns and done_step (E, S), grad (K, E, S, N, A) and the
        tape (a uint8 workspace of ``plan_grad_tape_bytes`` bytes).  Reused across calls, a graph-captured planner
        allocates nothing."""
        K, S, E, N, A = int(n_steps), int(n_samples), self.E, self.N, self.A
        kw = dict(device=self.device)
        return {"returns": torch.zeros((E, S), dtype=self.real, **kw),
                "done_step": torch.zeros((E, S), dtype=torch.int32, **kw),
                "grad": torch.zeros((K, E, S, N, A), dtype=self.real, **kw),
                "tape": torch.empty(self.plan_grad_tape_bytes(K, S), dtype=torch.uint8, **kw)}

    def plan_grad(self, actions: torch.Tensor, gamma: float = 1.0, targets: torch.Tensor | None = None,
                  out: dict | None = None) -> dict:
        """``gpd_plan_grad``: ``plan``'s returns and done_step, and ``grad`` (K, E, S, N, A) in the handle's precision, the
        gradient of each copy's return with respect to its actions (flags and end step held constant, rows after the
        end step 0; include/gpd.h).  Physics.DYN with RPM or ONE_D_RPM actions on Hover / MultiHover only.  Arguments as
        for ``plan``; ``out``: buffers from ``alloc_plan_grad_outputs``, written in place."""
        if self.is_ctrl or self.action_type not in ("rpm", "one_d_rpm") or self.physics_flags != 0:
            raise ValueError("plan_grad differentiates Physics.DYN (physics_flags 0) with rpm / one_d_rpm actions on the "
                             "Hover and MultiHover envs only")
        actions, K, S = _plan_inputs(self, actions, targets)
        if out is None:
            out = self.alloc_plan_grad_outputs(K, S)
        want = {"returns": ((self.E, S), self.real), "done_step": ((self.E, S), torch.int32),
                "grad": ((K, self.E, S, self.N, self.A), self.real)}
        _plan_outputs(out, want, targets)
        tape = out.get("tape")
        need = self.plan_grad_tape_bytes(K, S)
        if tape is None or tape.dim() != 1 or tape.dtype != torch.uint8 or tape.numel() < need or not tape.is_cuda:
            raise ValueError(f"out['tape'] must be a CUDA uint8 tensor of at least {need} bytes")
        _lib.check(self.lib.gpd_plan_grad(self.h, K, S, _ptr(actions), _ptr(targets), float(gamma), _ptr(out["returns"]),
                                          _ptr(out["done_step"]), _ptr(out["grad"]), _ptr(tape), tape.numel(),
                                          self._stream()))
        return {name: out[name] for name in want}

    def plan_return(self, actions: torch.Tensor, gamma: float = 1.0, targets: torch.Tensor | None = None) -> torch.Tensor:
        """The (E, S) returns of ``plan_grad`` as a differentiable function of ``actions`` (K, E, S, N, A): its backward
        is ``grad_output[None, :, :, None, None] * grad``, cast to the actions' dtype, so torch optimisers and losses use
        the kernel's gradient directly."""
        return _PlanReturn.apply(self, actions, float(gamma), targets)

    def adopt_obs(self, obs: torch.Tensor):
        """Makes ``obs`` (the latest observation written by ``step_into``) the current internal observation."""
        self.obs_buf[self._cur].copy_(obs.reshape(self.obs_buf[self._cur].shape))
        self._have_prev = True
        # `obs` may be released by its owner; a host mirror is rebuilt from the adopted observation at its next use
        _lib.check(self.lib.gpd_note_latest_obs(self.h, self._p_obs[self._cur]))

    # host-buffer path: what a numpy call site (the reference's own step signature) sees
    def attach_mirror(self, mirror: HostMirror | None = None, col0: int = 0, slide_steps: int = 128):
        """Binds a host mirror (RL envs): numpy steps then return strided views of its pinned log and the device sends back
        only what it computed (kin, reward, flags).  ``mirror=None`` allocates a private one."""
        if self.is_ctrl:
            raise ValueError("the Ctrl observation has no action ring to mirror")
        if mirror is None:
            mirror = HostMirror(self.W, self.A, self.E * self.N, slide_steps)
        _lib.check(self.lib.gpd_mirror_attach(self.h, mirror.base, mirror.rows, mirror.row_len, int(col0)))
        self._mirror, self._mirror_col0 = mirror, int(col0)
        return mirror

    def _host_actions(self, actions):
        adt = self.np_real if self.is_ctrl else np.float32
        a = np.ascontiguousarray(actions, dtype=adt)
        if a.size != self.E * self.N * self.A:
            raise ValueError(f"actions must have {self.E}x{self.N}x{self.A} elements, got {a.shape}")
        return a

    def step_host_begin(self, actions: np.ndarray, out):
        """Enqueues one numpy-facing step on the current stream (mirror path) without waiting for it."""
        a = self._host_actions(actions)
        _, rew, term, trunc, tkin = out
        nxt = self._cur ^ 1
        _lib.check(self.lib.gpd_step_mirror_begin(
            self.h, C.c_void_p(a.ctypes.data), self._p_obs[self._cur] if self._have_prev else None, self._p_obs[nxt],
            C.c_void_p(rew.ctypes.data), C.c_void_p(term.ctypes.data), C.c_void_p(trunc.ctypes.data),
            None if tkin is None else C.c_void_p(tkin.ctypes.data), self._stream()))
        self._cur, self._have_prev = nxt, True
        self._pending_actions = a          # the library reads it until the step is complete

    def step_host_end(self) -> int:
        _lib.check(self.lib.gpd_step_mirror_end(self.h, C.byref(self._row), self._stream()))
        self._pending_actions = None
        return self._row.value

    def step_host(self, actions: np.ndarray, out=None):
        """One BaseAviary.step on numpy arrays.  RL envs: the host-mirror path (``gpd_step_mirror``) on the sim's own device
        observation chain — the returned observation is a strided view of the pinned log, valid until the next step.
        Ctrl env: ``gpd_step_host`` (every byte of its observation is device-computed)."""
        if out is None:
            out = self.alloc_host_outputs()
        if self.is_ctrl:
            a = self._host_actions(actions)
            obs, rew, term, trunc, tkin = out
            _lib.check(self.lib.gpd_step_host(self.h, C.c_void_p(a.ctypes.data), C.c_void_p(obs.ctypes.data),
                                              C.c_void_p(rew.ctypes.data), C.c_void_p(term.ctypes.data),
                                              C.c_void_p(trunc.ctypes.data), None, self._stream()))
            return out
        if self._mirror is None:
            self.attach_mirror()
        self.step_host_begin(actions, out)
        row = self.step_host_end()
        return (self._mirror.view(row, self.E, self.N, self._mirror_col0),) + tuple(out[1:])

    def reset_host(self, mask: np.ndarray | None = None, obs: np.ndarray | None = None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        if self.is_ctrl:
            if obs is None:
                obs = np.empty((self.E, self.N, self.W), dtype=self.np_real)
            _lib.check(self.lib.gpd_reset_host(self.h, None if m is None else C.c_void_p(m.ctypes.data),
                                               C.c_void_p(obs.ctypes.data), self._stream()))
            return obs
        if self._mirror is None:
            self.attach_mirror()
        nxt = self._cur ^ 1
        _lib.check(self.lib.gpd_reset_mirror(self.h, None if m is None else C.c_void_p(m.ctypes.data),
                                             self._p_obs[self._cur] if self._have_prev else None, self._p_obs[nxt],
                                             C.byref(self._row), self._stream()))
        self._cur, self._have_prev = nxt, True
        view = self._mirror.view(self._row.value, self.E, self.N, self._mirror_col0)
        if obs is not None:
            obs[...] = view
            return obs
        return view

    def alloc_host_outputs(self, pinned: bool = False, terminal_kin: bool | None = None):
        """Host result arrays ``(obs|None, reward, terminated, truncated, terminal_kin|None)``.  reward / terminated /
        truncated are carved out of ONE block laid out like the device staging, so they travel in a single device-to-host
        copy.  RL envs: ``obs`` is None (the observation is a view of the host mirror).  Ctrl env: a dense ``obs`` array
        heads the same block.  ``terminal_kin`` (12 floats per drone, needed only to rebuild SB3's terminal_observation)
        is transferred only when asked for (default: never for plain step(), always for the VecEnv adapter)."""
        odt = np.dtype(self.np_real if self.is_ctrl else np.float32)
        rdt = np.dtype(self.np_real)
        obs_b = self.E * self.N * self.W * odt.itemsize if self.is_ctrl else 0
        obs_pad = (obs_b + 15) & ~15                      # same padding as gpd_step_host's packed device block
        rew_b = self.E * rdt.itemsize
        total = obs_pad + rew_b + 2 * self.E
        if pinned:
            block = torch.empty(total, dtype=torch.uint8).pin_memory().numpy()
        else:
            block = np.empty(total, dtype=np.uint8)
        obs = block[:obs_b].view(odt).reshape(self.E, self.N, self.W) if self.is_ctrl else None
        rew = block[obs_pad:obs_pad + rew_b].view(rdt)
        term = block[obs_pad + rew_b:obs_pad + rew_b + self.E]
        trunc = block[obs_pad + rew_b + self.E:]
        tkin = None
        if terminal_kin is None:
            terminal_kin = False
        if terminal_kin and self.auto_reset and not self.is_ctrl:
            tkin = (torch.empty((self.E, self.N, 12), dtype=torch.float32).pin_memory().numpy() if pinned
                    else np.empty((self.E, self.N, 12), np.float32))
        self._host_block = block
        return (obs, rew, term, trunc, tkin)

    # ------------------------------------------------------------------
    def get_state(self):
        """state20 (E,N,20), rpy_rates (E,N,3), pid_state (E,N,9), step_counter (E,) — BaseAviary.py:541-561."""
        st = torch.empty((self.E, self.N, 20), dtype=self.real, device=self.device)
        rr = torch.empty((self.E, self.N, 3), dtype=self.real, device=self.device)
        ps = torch.empty((self.E, self.N, 9), dtype=self.real, device=self.device)
        cnt = torch.empty(self.E, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.gpd_get_state(self.h, _ptr(st), _ptr(rr), _ptr(ps), _ptr(cnt), self._stream()))
        return st, rr, ps, cnt

    def set_state(self, state20=None, rpy_rates=None, pid_state=None, step_counter=None):
        def prep(t, dt):
            return None if t is None else t.to(device=self.device, dtype=dt).contiguous()
        st, rr, ps = prep(state20, self.real), prep(rpy_rates, self.real), prep(pid_state, self.real)
        cnt = prep(step_counter, torch.int32)
        _lib.check(self.lib.gpd_set_state(self.h, _ptr(st), _ptr(rr), _ptr(ps), _ptr(cnt), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()   # the temporaries above must outlive the kernel

    def rollout_pid(self, n_ctrl_steps: int, waypoints: torch.Tensor, wp_counters: torch.Tensor, action: torch.Tensor):
        """examples/pid.py:127-147 loop in one launch (Ctrl env); updates wp_counters and action in place."""
        assert waypoints.dtype == self.real and action.dtype == self.real and wp_counters.dtype == torch.int32
        assert waypoints.is_cuda and action.is_cuda and wp_counters.is_cuda
        _lib.check(self.lib.gpd_rollout_pid(self.h, int(n_ctrl_steps), _ptr(waypoints.contiguous()),
                                            int(waypoints.shape[0]), _ptr(wp_counters), _ptr(action), self._stream()))

    def episode_stats(self, clear: bool = False, nccl_comm=None) -> np.ndarray:
        """This sim's episode statistics, or — with an ``ncclComm_t`` from ``distributed.NcclStatsComm`` — the job-wide
        ones, reduced inside the library (one all-gather)."""
        out = (C.c_double * 8)()
        _lib.check(self.lib.gpd_episode_stats(self.h, out, int(clear), nccl_comm, self._stream()))
        return np.array(list(out))

    def adjacency(self, radius: float) -> torch.Tensor:
        """(E, N, N) adjacency matrices from the current positions (BaseAviary.py:658-675)."""
        out = torch.empty((self.E, self.N, self.N), dtype=self.real, device=self.device)
        _lib.check(self.lib.gpd_adjacency(self.h, float(radius), _ptr(out), self._stream()))
        return out

    def count_nonfinite(self) -> int:
        """Drones whose integrator state holds a NaN/Inf (failure detection; off the step path)."""
        out = C.c_longlong(0)
        _lib.check(self.lib.gpd_count_nonfinite(self.h, C.byref(out), self._stream()))
        return int(out.value)

    @property
    def obs(self) -> torch.Tensor:
        return self.obs_buf[self._cur]

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.gpd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
