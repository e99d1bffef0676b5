"""Host-side logic of bench.py (no GPU, no oracle compute): the workload table against SURVEY.md §8a / BASELINE.json, the
weak / strong batch split (train3d.py:495), and the reference arm's behaviour on ranks > 0 under torchrun."""
import os
import subprocess
import sys
from argparse import Namespace

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_config_table_matches_the_survey_token_counts_and_widths():
    # SURVEY.md §8a: tokens per sample 1296 / 5184 / 1936 / 2744 / 5832 and the per-layer widths
    want = {1: (1296, [1792, 1792], 256), 2: (5184, [1792, 1792, 896, 448], 256), 3: (1936, [2048, 2048, 2048], 256),
            4: (2744, [1024, 1024], 1024), 5: (5832, [1024, 1024, 1024], 2048)}
    for k, (n, dims, A) in want.items():
        c = bench.CONFIGS[k]
        tokens = 1
        for s in c["grid"]:
            tokens *= s
        assert tokens == n and c["dims"] == dims and c["attractors"] == A and c["modes"] == 4
        assert len(c["compress"]) == len(dims)
        assert bench.units_per_sample(c) == c["S"] ** (3 if c["kind"] == "3d" else 2)
    # the metric of the default line is BASELINE.json's: voxels/sec fwd+bwd Segtran3d BraTS 112^3 bs=4
    c = bench.CONFIGS[4]
    assert bench.metric_name(c).startswith("voxels/sec fwd+bwd Segtran3d BraTS 112^3 bs=4")
    assert bench.unit_name(c) == "voxels/s" and bench.unit_name(bench.CONFIGS[1]) == "pixels/s"


def test_weak_and_strong_batch_split():
    c = bench.CONFIGS[4]
    assert bench.local_batch(c, Namespace(scaling="weak"), 8) == 4          # per-GPU batch fixed
    assert bench.local_batch(c, Namespace(scaling="strong"), 2) == 2        # train3d.py:495: batch_size //= world_size
    assert bench.local_batch(c, Namespace(scaling="strong"), 4) == 1
    with pytest.raises(SystemExit):
        bench.local_batch(c, Namespace(scaling="strong"), 8)                # 4 samples do not split over 8 GPUs


def test_dump_outputs_writes_float32_and_samples_large_arrays_reproducibly(tmp_path):
    import numpy as np
    import torch
    n = bench.DUMP_MAX_ELEMS + 1000
    big = torch.arange(n, dtype=torch.float64)
    small = torch.randn(3, 4, dtype=torch.bfloat16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small, "loss": torch.tensor(1.5)})
    a = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in ("big", "small", "loss")}
    assert all(v.dtype == np.float32 for v in a.values())
    assert np.array_equal(a["small"], small.float().numpy()) and a["loss"].shape == () and float(a["loss"]) == 1.5
    # a sorted sample of positions drawn with a fixed seed: the same positions in every run, all in range
    assert a["big"].shape == (bench.DUMP_MAX_ELEMS,) and np.all(np.diff(a["big"]) >= 0) and a["big"][-1] < n
    assert len(np.unique(a["big"])) > bench.DUMP_MAX_ELEMS // 2
    assert np.array_equal(a["big"], np.load(str(tmp_path / "b" / "big.npy")))


def test_reference_arm_is_silent_on_other_ranks():
    """Under torchrun the driver starts `bench.py --impl reference` on every rank: only rank 0 works and prints."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    assert r.stdout.strip() == ""
