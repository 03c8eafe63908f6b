"""The bench line contract (driver prompt: metric/value/unit/..., e2e, gpu_launches, roofline, cpu_baseline), checked on
the committed lines of the final build: catches a key that gets dropped or renamed in bench.py."""
import glob
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}


def _latest(pattern):
    files = glob.glob(os.path.join(ROOT, "profiles", pattern))
    assert files, pattern
    return max(files, key=lambda f: tuple(int(x) for x in re.search(r"r(\d+)_v(\d+)_", f).groups()))


def test_single_gpu_line_has_every_contract_key():
    d = json.load(open(_latest("r[0-9]_v*_bench.json")))
    assert BASE | {"cpu_baseline"} <= set(d)
    assert d["metric"] == "separated utterance-sec/sec" and d["unit"] == "utt-s/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] != d["value"]                      # a real end-to-end number, not the device-timed one
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert d["roofline"]["bound"] in ("hbm", "tensor")
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-3
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["gpu_launches"] > 0 and d["warmup"] >= 3
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert abs(d["value"] - 256 * 1.0 / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6


def test_reference_arm_line():
    d = json.load(open(_latest("r[0-9]_v*_bench_reference_arm.json")))
    assert d["impl"] == "reference" and d["metric"] == "separated utterance-sec/sec"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]


def test_multi_gpu_line_is_whole_job_throughput():
    d = json.load(open(_latest("r[0-9]_v*_bench_n8.json")))
    assert BASE <= set(d) and d["n_gpus"] == 8 and d["config"]["global_batch"] == 8 * 256
    assert abs(d["value"] - 8 * 256 / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    # round 2: the headline IS the north-star data path (inputs scattered from rank 0, separated + masks gathered to it,
    # inside the timed region); the no-traffic variant and the transfer accounting ride beside it
    assert "scattered" in d["config"]["parallelism"] and "gathered" in d["config"]["parallelism"]
    assert {"ms_per_step", "value"} <= set(d["sharded_no_traffic"])
    sg = d["scatter_gather"]
    assert sg["gathered_equals_local_forward"] is True
    assert sg["bytes_out_of_rank0_per_step"] == 7 * d["e2e"]["h2d_bytes_per_step"]
    # on the wire back: both tensors, or masks only with `separated` rebuilt on the root (half of the bytes)
    per_rank = d["e2e"]["d2h_bytes_per_step"] // (2 if sg.get("wire") == "masks" else 1)
    assert sg["bytes_into_rank0_per_step"] == 7 * per_rank


def test_gather_wire_format_follows_the_traffic_through_the_root():
    import bench
    i_b, o_b, fwd = 69008384, 66318336, 0.53          # B=256 per rank: input / output bytes, ms per forward
    assert [bench.choose_wire(n, i_b, o_b, fwd) for n in (2, 4, 8)] == ["both", "both", "masks"]
    assert bench.choose_wire(8, i_b, o_b, fwd, "both") == "both" and bench.choose_wire(2, i_b, o_b, fwd, "masks") == "masks"
    assert bench.choose_wire(8, i_b, o_b, fwd, "auto") == "masks"
    with pytest.raises(SystemExit):
        bench.choose_wire(2, i_b, o_b, fwd, "bf16")


def test_dump_outputs_of_the_reference_arm_repeat_run_to_run(tmp_path):
    import subprocess
    import sys
    import numpy as np
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1",
                              "--steps", "1", "--warmup", "1", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 1
        runs.append({n: np.load(out / f"{n}.npy") for n in ("separated", "masks")})
    for n in ("separated", "masks"):
        assert runs[0][n].dtype == np.float32 and runs[0][n].shape == (8, 2, 257, 63), n
        assert np.array_equal(runs[0][n], runs[1][n]), n          # seeded inputs and weights: identical outputs
    assert runs[0]["masks"].min() >= 0.0 and runs[0]["masks"].max() <= 1.0
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert res.returncode != 0 and "--steps" in res.stderr


def test_dump_outputs_samples_whole_utterances_under_the_cap(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    a = torch.arange(10 * 2 * 3 * 4, dtype=torch.float64).view(10, 2, 3, 4)
    b = -a
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 1024 + 4 * 2 * a[0].numel() * 4)      # room for 4 of 10 utterances
    assert bench.dump_outputs(str(tmp_path), [("x", a), ("y", b)]) == 4
    x, y = np.load(tmp_path / "x.npy"), np.load(tmp_path / "y.npy")
    assert x.dtype == np.float32 and x.shape == (4, 2, 3, 4) and np.array_equal(y, -x)
    rows = [int(r[0, 0, 0]) // a[0].numel() for r in x]
    assert rows == sorted(set(rows)) and all(np.array_equal(x[i], a[r].numpy()) for i, r in enumerate(rows))
    monkeypatch.setattr(bench, "DUMP_BYTES", 10**6)
    assert bench.dump_outputs(str(tmp_path), [("x", a), ("y", b)]) == 10
    assert np.array_equal(np.load(tmp_path / "x.npy"), a.float().numpy())
