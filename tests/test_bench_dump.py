"""bench.py --dump-outputs: the arrays written are what the timed path returned, on the seeded workload; --steps sets the
number of timed steps.  The reference leg runs without a GPU, so it stands in for the path here."""
import json
import os
import subprocess
import sys

import numpy as np

import bench
import oracle_py as orc
from aardvark_b200 import abi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("status", "ed1", "ed2", "type_mask", "var_expected", "var_observed", "var_class", "totals", "solved_blocks")


def test_reference_leg_dumps_its_outputs_and_runs_the_steps_asked_for(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "chr20", "--scale", "0.002",
           "--steps", "7", "--warmup", "0", "--dump-outputs", str(tmp_path)]
    line = json.loads(subprocess.run(cmd, check=True, capture_output=True, text=True).stdout.splitlines()[-1])
    assert line["steps"] == 7
    ref, batch = synth.workload_chr20(scale=0.002, seed=20)
    out = orc.compare_batch(batch, [ref], abi.CompareCfg(50, 0, 0, 0), region_metrics=False)
    assert np.array_equal(np.load(tmp_path / "region_index.npy"), np.arange(batch.n_regions))
    assert np.array_equal(np.load(tmp_path / "variant_index.npy"), np.arange(batch.n_variants))
    for f in FIELDS:
        got = np.load(tmp_path / f"{f}.npy")
        assert got.dtype in (np.float32, np.float64), f
        want = getattr(out, f)
        n = batch.n_variants if f.startswith("var_") else batch.n_regions
        assert np.array_equal(got, want[:n] if want.ndim == 1 and want.size > 1 else want), f


def test_dump_samples_long_axes_the_same_way_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 8)
    n, nv = 100, 5
    arrays = {"status": np.arange(n, dtype=np.int32), "ed1": np.arange(n, dtype=np.uint32) * 3,
              "var_class": np.arange(nv, dtype=np.uint8), "totals": np.arange(6, dtype=np.uint64).reshape(2, 3)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, n, nv)
    ix = np.load(tmp_path / "a" / "region_index.npy")
    assert ix.size == 8 and np.all(np.diff(ix) > 0) and ix.max() < n
    assert np.array_equal(np.load(tmp_path / "a" / "status.npy"), ix)
    assert np.array_equal(np.load(tmp_path / "a" / "ed1.npy"), 3 * ix)
    assert np.array_equal(np.load(tmp_path / "a" / "var_class.npy"), np.arange(nv))
    assert np.array_equal(np.load(tmp_path / "a" / "totals.npy"), arrays["totals"])
    for f in ("region_index", "status", "ed1", "variant_index", "var_class", "totals"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{f}.npy"), np.load(tmp_path / "b" / f"{f}.npy"))
