"""GPU: ``bench.py --dump-outputs`` writes the last timed step's outputs as float64 .npy files, and two runs with the
same arguments write identical files (the inputs are seeded), so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ITEMS = 9000          # more than bench.DUMP_ITEMS: the per-item arrays are the seeded sample


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--items", str(ITEMS), "--steps", "3", "--warmup", "1",
           "--no-cpu", "--no-e2e", "--no-secondary", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_are_repeatable(cuda, tmp_path):
    line = _bench(tmp_path / "a")
    _bench(tmp_path / "b")
    assert line["steps"] == 3
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"item_index.npy", "item_dice_coefficient.npy", "item_hausdorff_distance.npy", "dataset_confusion.npy"} <= set(names)
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float64 and np.array_equal(a, b, equal_nan=True), name
    idx = np.load(tmp_path / "a" / "item_index.npy")
    assert idx.shape == (8192,) and (np.diff(idx) > 0).all() and idx[-1] < ITEMS
    assert np.load(tmp_path / "a" / "item_dice_coefficient.npy").shape == (8192, 8)
    assert np.load(tmp_path / "a" / "dataset_n_items.npy") == ITEMS
    assert np.array_equal(np.load(tmp_path / "a" / "dataset_dice_coefficient.npy"), line["dataset_dice"])
