"""bench.py --dump-outputs: what the last timed step returned, as .npy files that two builds can be compared on."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["agent_attr", "forest", "adjacency", "node_order", "edge_order", "valid_actions", "dist_target", "rewards", "dones"]


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d) if f.endswith(".npy")}


def test_dump_of_a_large_batch_is_a_seeded_sample_under_64_mb(tmp_path):
    import bench
    from flatland_marl_b200.batch import OBS_SHAPES
    E, N = 1024, 50                                                   # the headline batch: 124 MB of outputs
    g = torch.Generator().manual_seed(3)
    obs = {k: (torch.randn((E, N) + shp, generator=g) * 100).to(dt) for k, (shp, dt) in OBS_SHAPES.items()}
    rewards = torch.randint(-400, 1, (E, N), dtype=torch.int32, generator=g)
    dones = torch.randint(0, 2, (E, N + 1), dtype=torch.uint8, generator=g)
    obs["dist_target"] = obs["dist_target"].abs()
    obs["dist_target"][::3, ::7] = float("inf")                      # agents that cannot reach their target
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), (obs, rewards, dones))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 10**6
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == sorted(NAMES + ["env_index"])
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < E and (np.diff(idx) > 0).all()
    src = dict({k: v.numpy() for k, v in obs.items()}, rewards=rewards.numpy(), dones=dones.numpy())
    assert np.isinf(src["dist_target"][idx]).any()
    src["dist_target"] = np.where(np.isinf(src["dist_target"]), np.float32(-1), src["dist_target"])
    for k in NAMES:
        assert np.isfinite(a[k]).all(), k
        assert a[k].dtype == (np.float32 if src[k].dtype.kind == "f" else np.float64), k
        np.testing.assert_array_equal(a[k], src[k][idx], err_msg=k)
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "Test_00", "--envs", "6", "--steps", str(steps),
           "--warmup", "3", "--no-sweep", "--no-configs", "--no-cpu", "--no-policy", "--episodes", "0", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return _load(out)


@pytest.mark.gpu
def test_dump_is_the_same_for_the_same_arguments(tmp_path):
    a, b, c = _bench(tmp_path / "a", 5), _bench(tmp_path / "b", 5), _bench(tmp_path / "c", 6)
    assert sorted(a) == sorted(NAMES + ["env_index"])
    assert (a["env_index"] == np.arange(6)).all()
    assert a["forest"].shape == (6, 7, 31, 12) and a["dones"].shape == (6, 8)
    for k in NAMES:
        assert a[k].dtype in (np.float32, np.float64) and np.isfinite(a[k]).all(), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    # --steps sets the step whose outputs are written: one more timed step moves the trains
    assert not all((a[k] == c[k]).all() for k in ("agent_attr", "forest"))
