"""Windowed, teacher-forced oracle runs (tests/test_gpu_paths_vs_oracle.py, tests/test_paths_harness_cpu.py).

A checked GPU run must not read the state between its steps: `get_state` syncs a chained-state handle's tiles back into the
arrays and so changes the data path of the next step.  The runs are therefore compared at window ends only.  At each window
start the oracle is loaded from the GPU's exported state (state20 with the previous RPM in [16:20], rpy_rates, pid_state,
step counter) and the action ring of its latest observation; it then steps over the same actions, with the in-kernel
auto-reset restated by hand (`step_window`).  This module holds the oracle half, which needs no GPU.
"""
import numpy as np


def load_oracle(ref, state20, rpy_rates, pid_state, counter, obs):
    """Teacher-forces `ref` (an OracleSim) to an exported state; the ring comes from the observation's tail."""
    ref.state20[...] = state20
    ref.rpy_rates[...] = rpy_rates
    ref.pid_state[...] = pid_state
    ref.step_counter[...] = counter
    if not ref.is_ctrl:
        ref.ring[...] = np.asarray(obs, np.float32)[..., 12:].reshape(ref.ring.shape)


class Track:
    """What a window of oracle steps produced for one env set: last step's outputs, terminal kinematics of the envs that
    ended (latest end), FP32 exemption bands, and the episode statistics restated from the oracle's rewards."""

    def __init__(self, E, N, S):
        self.E, self.N, self.S = E, N, S
        self.ret = np.zeros(E)                  # float64 running return since each env's last reset
        self.tainted = np.zeros(E, bool)        # running return unknown (a flag decision inside a band)
        self.ep_len = np.zeros(E, np.int64)

    def start(self, counter):
        self.ep_len = np.asarray(counter, np.int64) // self.S
        self.n_ep = self.sum_len = self.steps = self.n_term = 0
        self.sum_ret, self.ret_ok = 0.0, True
        self.ended = np.zeros(self.E, bool)
        self.tkin = np.zeros((self.E, self.N, 12))
        self.ex_state = np.zeros((self.E, self.N), bool)
        self.ex_rpy = np.zeros((self.E, self.N), bool)
        self.ex_flag = np.zeros(self.E, bool)


def step_window(ref, tr, actions, auto_reset, nthreads=1, bands=None):
    """Steps `ref` over `actions` (a list of per-step action arrays), restating the in-kernel auto-reset and the statistics.
    `bands(ref, tr)` is called after every step, before the reset, to mark FP32 exemptions.  Returns the last step's
    (obs copy, reward, terminated, truncated)."""
    out = None
    for a in actions:
        o, r, te, trn = ref.step(a, nthreads=nthreads)
        r, te, trn = r.copy(), te.copy(), trn.copy()
        if bands is not None:
            bands(ref, tr)
        tr.steps += ref.E
        tr.ret += r
        tr.ep_len += 1
        if auto_reset and not ref.is_ctrl:
            done = (te | trn).astype(bool)
            if done.any():
                tr.tkin[done] = ref.obs[done][..., :12]
                tr.ended |= done
                tr.n_ep += int(done.sum())
                tr.n_term += int(te[done].astype(bool).sum())
                tr.sum_len += int(tr.ep_len[done].sum())
                tr.sum_ret += float(tr.ret[done].sum())
                tr.ret_ok &= not tr.tainted[done].any()
                tr.ret[done] = 0.0
                tr.tainted[done] = False
                tr.ep_len[done] = 0
                ref.reset(done.astype(np.uint8))
        out = (ref.obs.copy(), r, te, trn)
    return out
