"""-m gpu: chained state (GPD_STATE_IN_OBS).  Lean FP32 single-drone sims on the bulk kernel keep position and velocity only
in the latest observation row and rates / episode return in one packed vector; every other reader or writer of the state
syncs it back into the arrays first.  Handles with the mode on and off are driven through the same seeded sequence of
every path that touches the state, and must agree bit for bit (NaN / Inf included) in state, observation, reward, flags
and episode statistics after every event."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import state_edges as se
from helpers import default_targets
from gpd_b200.params import load_drone_params
from gpd_b200.sim import BatchedSim

pytestmark = pytest.mark.gpu

EP_LEN = 0.25           # 60 substeps: every env ends its first episode together (auto-reset bursts), later ones spread out


def bits(x):
    x = x.contiguous()
    return x.view(torch.int64 if x.element_size() == 8 else (torch.int32 if x.element_size() == 4 else torch.uint8))


def make(kw, E, on, monkeypatch):
    monkeypatch.setenv("GPD_STATE_IN_OBS", "1" if on else "0")
    s = BatchedSim(load_drone_params(kw["model"]), E, 1, "hover", kw["action_type"], kw["pyb_freq"], kw["ctrl_freq"], 0,
                   "f32", 0, auto_reset=True, target_pos=default_targets(kw), episode_len_sec=EP_LEN, threads_per_block=64)
    monkeypatch.delenv("GPD_STATE_IN_OBS")
    s.set_step_chaining(True)
    return s


class Pairs:
    """Env sets k = 0..n-1, each as a mode-on and a mode-off handle; an op is applied to both sides with the same inputs."""

    def __init__(self, kw, E, nsets, monkeypatch):
        self.on = [make(kw, E, True, monkeypatch) for _ in range(nsets)]
        self.off = [make(kw, E, False, monkeypatch) for _ in range(nsets)]
        self.E, self.A = E, self.on[0].A
        self.events = 0

    def sides(self):
        return (self.on, self.off)

    def compare(self, what, outs):
        """Step outputs only: no state read, so the next step of a chained handle still takes its state from the observation."""
        torch.cuda.synchronize()
        for x, y in zip(*outs):
            if isinstance(x, np.ndarray):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), what
            else:
                assert torch.equal(bits(x), bits(y)), what
        self.events += 1

    def check(self, what, outs=None):
        """Step outputs, then the exported state (which syncs a chained handle's tiles back into the arrays)."""
        if outs is not None:
            self.compare(what, outs)
        torch.cuda.synchronize()
        for k, (a, b) in enumerate(zip(self.on, self.off)):
            for x, y, name in zip(a.get_state(), b.get_state(), ("state20", "rpy_rates", "pid_state", "counter")):
                assert torch.equal(bits(x), bits(y)), f"{what}: set {k} {name}"
            assert torch.equal(bits(a.obs), bits(b.obs)), f"{what}: set {k} obs"
            assert np.array_equal(a.episode_stats(), b.episode_stats(), equal_nan=True), f"{what}: set {k} stats"
        self.events += 1

    def close(self):
        for s in self.on + self.off:
            s.close()


def rand_act(rng, E, A, scale=1.0):
    return torch.from_numpy(rng.uniform(-scale, scale, (E, 1, A)).astype(np.float32)).cuda()


@pytest.mark.parametrize("shape,E", [("hover30", 28453), ("one_d_rpm48", 5003)])
def test_state_chain_matches_arrays(shape, E, monkeypatch):
    """28,453 envs at 64 per tile = 445 tiles (two tiles per CTA behind another handle, a ragged last tile); ONE_D_RPM at
    48 Hz is the A = 1 path (unshifted tile, rows slid in shared memory)."""
    kw = se.shape("one_d_rpm", ctrl_freq=48) if shape == "one_d_rpm48" else se.shape("hover30")
    rng = np.random.default_rng(2024)
    P = Pairs(kw, E, 2, monkeypatch)
    E, A = P.E, P.A
    for side in P.sides():
        for s in side:
            s.reset()
    P.check("reset")

    # eager chained steps over the rotating sets, through the first auto-reset burst: three steps per set between state
    # reads, every output compared, so that most steps take their state from the observation chain
    for it in range(6):
        outs = ([], [])
        for rnd in range(3):
            acts = [rand_act(rng, E, A, 0.3) for _ in P.on]
            for j, side in enumerate(P.sides()):
                for k, s in enumerate(side):
                    o, r, te, tr = s.step(acts[k])
                    outs[j].extend([o.clone(), r.clone(), te.clone(), tr.clone()])
        if it % 2:
            P.check(f"eager steps {it}", outs)
        else:
            P.compare(f"eager steps {it}", outs)

    # CUDA graphs of the rotation (an even number of steps per set), replayed several times
    gacts = [rand_act(rng, E, A) for _ in range(5)]
    graphs = []
    for side in P.sides():
        side_stream = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.stream(side_stream):
            with torch.cuda.graph(g, stream=side_stream):
                for k in range(4 * len(side)):
                    side[k % len(side)].step(gacts[k % 5])
        graphs.append(g)
    for rep in range(3):
        for g in graphs:
            g.replay()
        P.check(f"graph replay {rep}")

    # get_state / set_state (rates only, then everything) between steps of a chained run
    rates = torch.from_numpy(rng.uniform(-3, 3, (E, 1, 3)).astype(np.float32)).cuda()
    for side in P.sides():
        side[0].step(rand_act(np.random.default_rng(5), E, A))
        side[1].step(rand_act(np.random.default_rng(6), E, A))
        side[0].get_state()
        side[1].set_state(rpy_rates=rates)
        side[0].step(rand_act(np.random.default_rng(7), E, A))
        side[1].step(rand_act(np.random.default_rng(8), E, A))
    P.check("set_state rates only")
    full = [x.clone() for x in P.on[0].get_state()]
    full[0][..., 10:13] *= -1
    for side in P.sides():
        side[0].set_state(*full)
        side[0].step(rand_act(np.random.default_rng(9), E, A))
    P.check("set_state full")

    # masked reset
    mask = torch.from_numpy(rng.random(E) < 0.4).cuda()
    for side in P.sides():
        for s in side:
            s.reset(mask)
        side[0].step(rand_act(np.random.default_rng(10), E, A))
    P.check("masked reset")

    # step_into over a trajectory buffer, then adopt_obs; then a foreign obs_prev (not the latest observation)
    T = 5
    tacts = [rand_act(rng, E, A) for _ in range(T)]
    trajs = []
    for side in P.sides():
        s = side[0]
        obs = torch.zeros((T + 1, E, 1, s.W), device="cuda")
        rew = torch.zeros((T, E), device="cuda")
        term = torch.zeros((T, E), dtype=torch.uint8, device="cuda")
        trunc = torch.zeros((T, E), dtype=torch.uint8, device="cuda")
        obs[0].copy_(s.obs)
        for t in range(T):
            s.step_into(tacts[t], obs[t], obs[t + 1], rew[t], term[t], trunc[t])
        s.adopt_obs(obs[T])
        trajs.append([obs, rew, term, trunc])
    P.check("step_into + adopt_obs", trajs)
    foreign = [], []
    fa = rand_act(rng, E, A)
    for j, side in enumerate(P.sides()):
        s = side[0]
        prev = torch.zeros((E, 1, s.W), device="cuda")
        prev[..., 12:] = s.obs[..., 12:]
        out = torch.empty_like(prev)
        rew = torch.zeros(E, device="cuda")
        fl = torch.zeros((2, E), dtype=torch.uint8, device="cuda")
        s.step_into(fa, prev, out, rew, fl[0], fl[1])
        s.adopt_obs(out)
        s.step(rand_act(np.random.default_rng(11), E, A))
        foreign[j].extend([out, rew, fl])
    P.check("foreign obs_prev", foreign)

    # host-mirror numpy steps, interleaved with device steps
    host = [], []
    hacts = [rng.uniform(-1, 1, (E, 1, A)).astype(np.float32) for _ in range(3)]
    for j, side in enumerate(P.sides()):
        s = side[1]
        for t in range(3):
            o, r, te, tr, _ = s.step_host(hacts[t])
            host[j].extend([np.ascontiguousarray(o).copy(), r.copy(), te.copy(), tr.copy()])
        s.step(rand_act(np.random.default_rng(12), E, A))
        o, r, te, tr, _ = s.step_host(hacts[0])
        host[j].extend([np.ascontiguousarray(o).copy(), r.copy()])
    P.check("host mirror", host)

    # adjacency and the non-finite count read the state too
    adj = [], []
    for j, side in enumerate(P.sides()):
        adj[j].append(side[0].adjacency(0.5))
        adj[j].append(torch.tensor([side[0].count_nonfinite()]))
        side[0].step(rand_act(np.random.default_rng(13), E, A))
    P.check("adjacency / nonfinite", adj)

    # off-nominal injected states: fast spins, any attitude, NaN / Inf drones, through chained steps
    kwf = dict(kw, episode_len_sec=EP_LEN)
    for fam_name in ("F1", "F2", "F7"):
        fam = se.FAMILIES[fam_name](np.random.default_rng(31), kwf, E, "f32")
        fa = [torch.from_numpy(np.ascontiguousarray(fam["actions"][k], np.float32)).cuda() for k in range(2)]
        st = torch.from_numpy(fam["state20"].astype(np.float32))
        rr = torch.from_numpy(fam["rpy_rates"].astype(np.float32))
        cnt = torch.from_numpy(fam["step_counter"])
        res = [], []
        for j, side in enumerate(P.sides()):
            side[0].set_state(st, rr, None, cnt)
            for k in range(2):
                side[0].step(fa[k])
                side[1].step(fa[k])
            res[j].extend([x.clone() for x in side[0].get_state()])
            for k in range(2):
                side[0].step(fa[k])
        P.check(f"family {fam_name}", res)
    assert P.events >= 20
    P.close()


def test_state_chain_observation_is_state(monkeypatch):
    """With the mode on, position and velocity of the next step come from the latest observation: an in-place edit of it
    is an edit of the env's state (include/gpd.h).  With the mode off the arrays stay authoritative."""
    kw = se.shape("hover30")
    E = 4096
    got = {}
    for on in (True, False):
        s = make(kw, E, on, monkeypatch)
        s.reset()
        s.step(torch.zeros((E, 1, 4), device="cuda"))
        s.obs[:, 0, 0] += 0.25          # kin[0] = x
        s.obs[:, 0, 7] = 1.5            # kin[7] = vy
        got[on] = s.get_state()[0].clone()
        s.close()
    assert torch.all(got[True][:, 0, 0] == got[False][:, 0, 0] + 0.25)
    assert torch.all(got[True][:, 0, 11] == 1.5)
    assert not torch.any(got[False][:, 0, 11] == 1.5)


def test_state_chain_mirror_step_behind_a_foreign_obs_prev(monkeypatch):
    """Host-mirror steps: chained steps, then a step whose obs_prev is not the latest observation (a step_into that was not
    adopted), which must sync the state before it runs."""
    kw = se.shape("hover30")
    E = 5003
    P = Pairs(kw, E, 1, monkeypatch)
    for side in P.sides():
        side[0].reset()
        side[0].attach_mirror()
    rng = np.random.default_rng(77)
    hacts = [rng.uniform(-1, 1, (E, 1, 4)).astype(np.float32) for _ in range(6)]
    dacts = rand_act(rng, E, 4)

    def host_steps(s, acts, res):
        for a in acts:
            o, r, te, tr, _ = s.step_host(a)
            res.extend([np.ascontiguousarray(o).copy(), r.copy(), te.copy(), tr.copy()])

    outs = [], []
    for j, side in enumerate(P.sides()):
        host_steps(side[0], hacts[:4], outs[j])
    P.compare("mirror steps", outs)
    outs = [], []
    for j, side in enumerate(P.sides()):
        s = side[0]
        out = torch.empty_like(s.obs)
        rew = torch.zeros(E, device="cuda")
        fl = torch.zeros((2, E), dtype=torch.uint8, device="cuda")
        s.step_into(dacts, s.obs, out, rew, fl[0], fl[1])     # not adopted: the next mirror step reads another obs_prev
        host_steps(s, hacts[4:], outs[j])
        outs[j].extend([out, rew, fl])
    P.check("mirror step behind a foreign obs_prev", outs)
    P.close()
