"""The windowed, teacher-forced oracle of tests/test_gpu_paths_vs_oracle.py, checked without a GPU: an OracleSim loaded at
every window start from another one's arrays, with the action ring taken from its observation, must reproduce the other's
uninterrupted run bit for bit, through auto-resets, DSLPID state and multi-drone envs; and the episode statistics restated
window by window must equal those of the uninterrupted run."""
import numpy as np
import pytest

import state_edges as se
from paths_harness import Track, load_oracle, step_window

SHAPES = {
    "hover_rpm_short": (se.shape("hover30", episode_len_sec=0.3), 4),
    "hover_pid48": (se.shape("pid", ctrl_freq=48, episode_len_sec=0.2), 3),
    "one_d_rpm": (se.shape("one_d_rpm", episode_len_sec=0.2), 2),
    "multi3_gd": (se.shape("multi3_gd", episode_len_sec=0.4), 4),
    "ctrl3_dw": (se.shape("ctrl3_dw"), 4),
}


def _actions(rng, kw, E, A):
    N = kw["num_drones"]
    if kw["env_kind"] == "ctrl":
        from gpd_b200.params import load_drone_params
        return load_drone_params(kw["model"]).HOVER_RPM * (1 + 0.05 * rng.uniform(-1, 1, (E, N, A)))
    return rng.uniform(-1, 1, (E, N, A)).astype(np.float32)


@pytest.mark.parametrize("name", list(SHAPES))
def test_teacher_forced_windows_reproduce_an_uninterrupted_run(name):
    kw, win = SHAPES[name]
    E, windows = 97, 8
    rng = np.random.default_rng(3)
    S = kw["pyb_freq"] // kw["ctrl_freq"]
    N = kw["num_drones"]
    xyz = np.stack([rng.uniform(-.5, .5, (E, N)), rng.uniform(-.5, .5, (E, N)), rng.uniform(0.2, 1.2, (E, N))], -1)
    if kw["env_kind"] == "multihover":
        xyz[..., 2] += 0.3 * np.arange(N)
    rpy = rng.uniform(-.2, .2, (E, N, 3))
    full, forced = se.oracle_sim(kw, E, xyz, rpy), se.oracle_sim(kw, E, xyz, rpy)
    A = full.A
    auto = kw["env_kind"] != "ctrl"
    t_full, t_forced = Track(E, N, S), Track(E, N, S)
    t_full.start(full.step_counter)
    tot = dict(n_ep=0, sum_len=0, sum_ret=0.0, steps=0)
    ended_any = 0
    for w in range(windows):
        acts = [_actions(rng, kw, E, A) for _ in range(win)]
        # the other sim's exported arrays, as get_state returns them; the ring only through the observation
        load_oracle(forced, full.state20.copy(), full.rpy_rates.copy(), full.pid_state.copy(), full.step_counter.copy(),
                    full.obs.copy())
        if auto:
            assert np.array_equal(forced.ring, full.ring)
        t_forced.start(forced.step_counter)
        got = step_window(forced, t_forced, acts, auto)
        want = step_window(full, t_full, acts, auto)
        for x, y in zip(got, want):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8)), (name, w)
        for a, b in ((forced.state20, full.state20), (forced.rpy_rates, full.rpy_rates), (forced.pid_state, full.pid_state),
                     (forced.step_counter, full.step_counter), (forced.obs, full.obs)):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (name, w)
        if auto:
            assert np.array_equal(forced.ring, full.ring)
            assert np.array_equal(t_forced.tkin[t_forced.ended], t_full.tkin[t_forced.ended])
        for k in tot:
            tot[k] += getattr(t_forced, k)
        ended_any += int(t_forced.ended.sum())
    assert tot["steps"] == t_full.steps == E * win * windows
    assert tot["n_ep"] == t_full.n_ep and tot["sum_len"] == t_full.sum_len
    assert abs(tot["sum_ret"] - t_full.sum_ret) <= 1e-12 * max(abs(t_full.sum_ret), 1.0)     # summed per window
    if kw["action_type"] in ("pid", "one_d_pid"):
        assert np.abs(full.pid_state).max() > 0           # the controller state is carried across the windows
    if auto:
        assert t_full.n_ep > E and ended_any > 0          # auto-resets inside the windows, several per env
