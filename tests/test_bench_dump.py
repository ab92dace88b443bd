"""bench.py --dump-outputs: what the last timed step computed, sampled within the size budget, identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from tests.helpers import REPO


def test_dump_samples_the_same_envs_of_every_array_within_the_budget(tmp_path):
    E, n = 5000, 30
    env_id = torch.arange(E, dtype=torch.float64)
    arrays = dict(obs=env_id[:, None, None].float().expand(E, 192, n).contiguous(),
                  p=env_id[:, None, None].expand(E, 2, n).contiguous(),
                  done=torch.zeros(E, 1, n, dtype=torch.bool),
                  nbr=env_id[:, None, None].int().expand(E, n, 6).contiguous(),
                  sensed=None)
    budget = 4 * 10**6
    bench.dump_outputs(str(tmp_path), "random", arrays, budget)
    files = sorted(os.listdir(tmp_path))
    assert files == ["random_done.npy", "random_nbr.npy", "random_obs.npy", "random_p.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= budget + 4 * 128       # + .npy headers
    got = {f[len("random_"):-4]: np.load(tmp_path / f) for f in files}
    assert got["p"].dtype == np.float64 and all(got[k].dtype == np.float32 for k in ("obs", "done", "nbr"))
    pick = got["p"][:, 0, 0]
    assert 100 < len(pick) < E and np.all(np.diff(pick) > 0)
    for k in ("obs", "nbr"):
        assert np.array_equal(got[k][:, 0, 0], pick)
    bench.dump_outputs(str(tmp_path / "again"), "random", arrays, budget)
    assert np.array_equal(np.load(tmp_path / "again" / "random_p.npy"), got["p"])


@pytest.mark.gpu
def test_two_runs_dump_identical_outputs_of_the_last_timed_step(tmp_path):
    lines = []
    for run, steps in (("a", 7), ("b", 7), ("c", 8)):
        r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "2", "--envs-per-gpu", "4096",
                            "--no-e2e", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path / run)],
                           cwd=REPO, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert [d["steps"] for d in lines] == [7, 7, 8] and lines[0]["regimes"]["random"]["ms_per_step"] > 0
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) == sorted(os.listdir(tmp_path / "c"))
    assert {f.split("_")[0] for f in files} == {"random", "converged"}
    assert "random_obs.npy" in files and "converged_a_prior.npy" in files
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and 0 < a.shape[0] < 4096       # a sample of the envs
        assert np.array_equal(a, b, equal_nan=True), f
    for regime in ("random", "converged"):
        obs, p = np.load(tmp_path / "a" / f"{regime}_obs.npy"), np.load(tmp_path / "a" / f"{regime}_p.npy")
        assert np.isfinite(obs).all() and obs.any() and np.isfinite(p).all()
        # one more timed step moves the state: the dump is the last timed step's, not an earlier one
        assert not np.array_equal(p, np.load(tmp_path / "c" / f"{regime}_p.npy"))
        assert not np.array_equal(obs, np.load(tmp_path / "c" / f"{regime}_obs.npy"))
