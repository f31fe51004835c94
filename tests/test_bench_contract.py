"""CPU: the bench.py contract that can be checked without a GPU -- the reference arm prints ONE JSON line with the
required keys (it times the oracle port on the host cores), and our arm refuses to run without a B200 instead of
falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 0
    assert d["vs_baseline"] is None and d["value"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample_within_the_budget(tmp_path):
    import types

    import numpy as np
    import torch

    import bench
    n, H, W, lo = 5, 4, 6, 3
    ids = torch.arange(n * H * W, dtype=torch.int32).view(n, H, W) - 1
    wl = types.SimpleNamespace(H=H, W=W, n_local=n, lo=lo, ids_host=ids)
    res = {k: float(i) for i, k in enumerate(bench.PQ_FIELDS)}
    res["per_class"] = {7: {k: 1.0 for k in bench.CLASS_FIELDS}, 2: {k: 2.0 for k in bench.CLASS_FIELDS}}
    res["dvpq"] = {2: {"iou": np.full(19, 0.5), "tp": np.arange(19), "fn": np.zeros(19, np.int64),
                       "fp": np.ones(19, np.int64), "pq": 5.0, "pq_things": 1.0, "pq_stuff": 2.0, "n_windows": 4}}
    names = ("ids", "ids_frames", "pq", "pq_per_class", "dvpq_k2", "dvpq_k2_pq")
    dumps = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "cfg", wl, res, budget=2 * H * W * 4 + 1)   # room for two frames
        assert sorted(p.name for p in (tmp_path / d).iterdir()) == sorted(f"cfg_{k}.npy" for k in names)
        dumps.append({k: np.load(tmp_path / d / f"cfg_{k}.npy") for k in names})
    a = dumps[0]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    frames = a["ids_frames"].astype(np.int64)
    assert len(frames) == 2 and list(frames) == sorted(set(frames)) and all(lo <= f < lo + n for f in frames)
    assert np.array_equal(a["ids"], ids.numpy()[frames - lo].astype(np.float32))
    assert a["pq"].tolist() == list(range(len(bench.PQ_FIELDS)))
    assert a["pq_per_class"][:, 0].tolist() == [2, 7] and a["pq_per_class"].shape == (2, 1 + len(bench.CLASS_FIELDS))
    assert a["dvpq_k2"].shape == (4, 19) and a["dvpq_k2"][1].tolist() == list(range(19))
    assert a["dvpq_k2_pq"].tolist() == [5.0, 1.0, 2.0, 4.0]
    assert all(np.array_equal(a[k], dumps[1][k]) for k in names)   # the sample is fixed


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and r.stdout.strip() == ""  # no number, no fallback
