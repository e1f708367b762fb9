"""bench.py --dump-outputs: what one step returned, as float64 .npy files under the size cap, with a sample that is
the same from run to run.  Runs on stand-in results (no GPU needed)."""
import os

import numpy as np
import torch

import bench


def _step(B, nt):
    # every trajectory entry holds its problem's index: the dump must keep rows and indices together.
    # (an expanded view: the 1 GB block of a config-4 step is never materialised)
    traj = torch.arange(B, dtype=torch.float64).expand(10, nt, B)
    tf = 0.9 + torch.arange(B, dtype=torch.float64) * 1e-7
    return {"traj": traj, "tf": tf, "final_mass": 2600.0 + tf, "status": (torch.arange(B) % 3).to(torch.int32),
            "iterations": torch.full((B,), 23, dtype=torch.int32), "kkt": tf * 1e-11}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_of_a_config4_step_is_capped_and_reproducible(tmp_path):
    B, nt = 65536, 200
    raw = _step(B, nt)
    bench.dump_outputs(str(tmp_path / "a"), raw)
    bench.dump_outputs(str(tmp_path / "b"), raw)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert set(a) == {"tf", "final_mass", "status", "iterations", "kkt", "index", "traj", "traj_index"}
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64e6
    assert all(np.array_equal(a[k], b[k]) for k in a)
    # per-problem scalars: the whole batch; trajectories: a sorted sample without repeats, in the batch's order
    assert np.array_equal(a["index"], np.arange(B)) and np.array_equal(a["tf"], raw["tf"].numpy())
    assert np.array_equal(a["status"], raw["status"].numpy().astype(np.float64))
    n = a["traj_index"].size
    assert a["traj"].shape == (10, nt, n) and 1000 < n < B
    assert np.all(np.diff(a["traj_index"]) > 0)
    assert np.array_equal(a["traj"], np.broadcast_to(a["traj_index"], (10, nt, n)))


def test_dump_of_a_small_step_is_whole_and_offsets_a_shard(tmp_path):
    raw = _step(7, 5)
    bench.dump_outputs(str(tmp_path), raw, traj_offset=100)
    d = _load(tmp_path)
    assert np.array_equal(d["index"], np.arange(7)) and np.array_equal(d["traj_index"], 100 + np.arange(7))
    assert np.array_equal(d["traj"], raw["traj"].numpy())
    bench.dump_outputs(str(tmp_path / "no_traj"), dict(raw, traj=None))
    assert "traj" not in _load(tmp_path / "no_traj")
