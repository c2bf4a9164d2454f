"""bench.py --dump-outputs: what the timed path returned in its last step, written as .npy files, so that two builds
can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _util import ROOT
import bench
import vision_transformer_detector_b200 as vd


def _records(batch, seed=0):
    rng = np.random.default_rng(seed)
    return vd.DetectionRecords(rng.normal(size=(batch, 17, 6)).astype(np.float32), rng.normal(size=(batch, 17, 6)).astype(np.float32),
                               rng.integers(0, 80, (batch, 17)).astype(np.int32), rng.uniform(0, 1, (batch, 17)).astype(np.float32),
                               rng.integers(0, 2, (batch, 17)).astype(np.uint8), rng.integers(0, 608, (batch, 17, 4)).astype(np.int32))


def test_write_outputs_writes_every_record_field(tmp_path):
    rec = _records(5)
    shapes = bench.write_outputs(rec, str(tmp_path))
    assert shapes == {"logits": [5, 17, 6], "decoded": [5, 17, 6], "class_id": [5, 17], "class_conf": [5, 17], "keep": [5, 17],
                      "corners": [5, 17, 4]}
    for name in shapes:
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == (np.float32 if getattr(rec, name).dtype.kind == "f" else np.float64)
        assert np.array_equal(a, getattr(rec, name))
    import torch
    packed = torch.arange(34 * 13, dtype=torch.float32).reshape(34, 13)
    assert bench.write_outputs(packed, str(tmp_path / "packed")) == {"packed": [34, 13]}
    assert np.array_equal(np.load(tmp_path / "packed" / "packed.npy"), packed.numpy())


def test_write_outputs_samples_the_same_rows_under_the_limit(tmp_path):
    rec = _records(1000)
    limit = 200_000
    shapes = bench.write_outputs(rec, str(tmp_path / "a"), limit=limit)
    bench.write_outputs(rec, str(tmp_path / "b"), limit=limit)
    rows = np.load(tmp_path / "a" / "sample_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0)
    assert limit - 2000 < sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in shapes) <= limit
    for name in shapes:
        a = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{name}.npy"))                        # a fixed sample
        if name != "sample_rows":
            assert np.array_equal(a, getattr(rec, name)[rows])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit):
        bench.parse_args()


def _run_bench(out_dir, steps):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--batch-per-gpu", "4",
                        "--no-e2e", "--no-variants", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dumps_the_records_of_its_seeded_inputs(tmp_path):
    """Two runs with different --steps: the launches scale with the timed steps, and both dump the records that the
    model returns for the bench's seeded weights and images."""
    import torch
    two, three = _run_bench(tmp_path / "two", 2), _run_bench(tmp_path / "three", 3)
    assert (two["steps"], three["steps"]) == (2, 3)
    assert two["gpu_launches"] > 0 and two["gpu_launches"] * 3 == three["gpu_launches"] * 2
    cfg = vd.DetectorConfig()
    model = vd.VisionTransformerDetector(cfg, seed=None, compute_mode="bf16")
    model.set_weights(vd.random_weights(cfg, seed=1, spread=True))
    g = torch.Generator(device="cuda")
    g.manual_seed(1234)
    x = torch.rand((4, *cfg.input_shape), generator=g, device="cuda", dtype=torch.float32) * 2 - 1
    rec = model.detect(x, image_size=cfg.input_shape[:2])
    for name in ("logits", "decoded", "class_id", "class_conf", "keep", "corners"):
        want = getattr(rec, name).cpu().numpy()
        for run in ("two", "three"):
            assert np.array_equal(np.load(tmp_path / run / f"{name}.npy"), want), (run, name)
    model.close()
