"""bench.py --dump-outputs: what the last timed step returned, as .npy files that two builds can compare output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("obs", "reward", "terminated", "truncated")


def test_dump_keeps_one_seeded_env_sample_within_64_mb(tmp_path):
    import bench
    rng = np.random.default_rng(3)
    E = 300_000                 # ~90 MB of step outputs
    out = {"obs": rng.random((E, 1, 72), dtype=np.float32), "reward": rng.random(E),
           "terminated": (rng.random(E) < 0.1).astype(np.uint8), "truncated": np.zeros(E, np.uint8)}
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted([n + ".npy" for n in NAMES] + ["env_index.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0)
    for n in NAMES:
        got = np.load(tmp_path / "a" / f"{n}.npy")
        assert got.dtype == (np.float64 if n == "reward" else np.float32)
        assert np.array_equal(got, out[n][idx.astype(np.int64)].astype(got.dtype))
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{n}.npy"))


def test_dump_is_refused_on_the_cpu_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr


@pytest.mark.gpu
def test_dump_is_reproducible_and_is_the_last_timed_step(tmp_path):
    """Same arguments, same outputs; one more timed step, other outputs.  Graph replay (one graph per window, or 32-step
    graphs replayed in cycles), direct launches and two streams step the sets through the same sequence, so they end on the
    same outputs.  With a tail graph (K = 37 = 32 + 5 in cycles mode) the dump is the tail's last step: the newest action in
    the observation's ring is the one the bench gave that step (action k % 4 of its seeded schedule, step k = 4)."""
    import torch
    E, nsets = 4096, 2

    def run(name, *args):
        d = tmp_path / name
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--warmup", "4", "--envs", str(E),
                              "--sets", str(nsets), "--no-extra", "--no-cpu", "--e2e-steps", "5", "--dump-outputs", str(d), *args],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        return {n: np.load(d / f"{n}.npy") for n in NAMES}

    def same(u, v):
        for n in NAMES:
            assert np.array_equal(u[n], v[n]), n
    a = run("a", "--steps", "7")
    assert a["obs"].shape == (E, 1, 72) and a["obs"].dtype == np.float32 and a["reward"].dtype == np.float32
    assert np.isfinite(a["obs"]).all() and a["obs"][..., 2].std() > 0
    same(a, run("b", "--steps", "7"))
    same(a, run("direct", "--steps", "7", "--launch", "direct"))
    same(a, run("streams", "--steps", "7", "--streams", "2"))
    assert not np.array_equal(a["obs"], run("more", "--steps", "8")["obs"])
    cycles = run("cycles", "--steps", "64", "--launch", "cycles")
    same(cycles, run("direct64", "--steps", "64", "--launch", "direct"))

    # the bench's action schedule: 2 * sets tensors from a generator seeded with the rank
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    acts = [(torch.rand((E, 1, 4), generator=g, device="cuda") * 2 - 1).cpu().numpy() for _ in range(2 * nsets)]

    def newest_action_is(out, k):
        live = (out["terminated"] == 0) & (out["truncated"] == 0)        # an auto-reset env shows its fresh observation
        assert live.sum() > E // 2
        return np.array_equal(out["obs"][live][:, 0, -4:], acts[k % (2 * nsets)][live][:, 0])
    assert newest_action_is(cycles, 31) and not newest_action_is(cycles, 4)
    tail = run("tail", "--steps", "37", "--launch", "cycles")
    assert newest_action_is(tail, 4) and not newest_action_is(tail, 31)
