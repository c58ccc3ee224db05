"""CPU: the reference arm of bench.py prints the JSON contract (metric/unit/config, cpu_baseline, e2e zeros)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "msda_encoder", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["value"] > 0 and line["unit"] == "images/s" and "workload" in line["config"]


def test_workload_registry_and_defaults():
    sys.path.insert(0, ROOT)
    import bench_workloads as B
    assert B.DEFAULT_WORKLOAD == "pair_forward"
    assert set(B.WORKLOADS) >= {"pair_forward", "msda_encoder", "gdino_head"}
    assert set(B._CPU) >= set(B.WORKLOADS)
    p = B.measured_peaks()
    assert p["hbm_gbs"] > 1000 and p["bf16_tflops_sustained"] > 100


def test_dump_outputs_whole_and_sampled(tmp_path):
    """bench.py --dump-outputs: every tensor of a nested step result as <dotted name>.npy, float64 and integers as
    float64, other floats as float32; over the byte budget each array becomes the same seeded sample of distinct
    elements on every call, with its indices under sample_index/, all within the budget."""
    import glob
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    out = {"logits": torch.arange(1000, dtype=torch.bfloat16).reshape(10, 100),
           "aux": (torch.ones(3, dtype=torch.float64), torch.tensor([1, 2, (1 << 40) + 1])), "n": 4}
    m = bench.dump_outputs(out, str(tmp_path / "whole"))
    assert set(m) == {"logits", "aux.0", "aux.1"}
    a = np.load(tmp_path / "whole" / "logits.npy")
    assert a.dtype == np.float32 and a.shape == (10, 100) and np.array_equal(a, out["logits"].float().numpy())
    assert np.load(tmp_path / "whole" / "aux.0.npy").dtype == np.float64
    assert np.load(tmp_path / "whole" / "aux.1.npy").tolist() == [1, 2, (1 << 40) + 1]       # integers stay exact
    assert not (tmp_path / "whole" / "sample_index").exists()
    big = {"x": torch.randn(4096, generator=torch.Generator().manual_seed(0)), "y": torch.ones(1024, dtype=torch.float64),
           "tiny": torch.ones(1)}
    for d in ("s1", "s2"):
        bench.dump_outputs(big, str(tmp_path / d), budget=4096)
    assert bench.DUMP_BUDGET_BYTES == 64 * 10 ** 6
    x1, x2 = np.load(tmp_path / "s1" / "x.npy"), np.load(tmp_path / "s2" / "x.npy")
    ix = np.load(tmp_path / "s1" / "sample_index" / "x.npy")
    assert np.array_equal(x1, x2) and np.array_equal(x1, big["x"].numpy()[ix.astype(np.int64)])
    assert len(np.unique(ix)) == len(ix) and (np.diff(ix) > 0).all()                             # distinct, sorted
    assert np.load(tmp_path / "s1" / "tiny.npy").size == 1 and np.load(tmp_path / "s1" / "y.npy").dtype == np.float64
    written = sum(os.path.getsize(f) for f in glob.glob(str(tmp_path / "s1" / "**" / "*.npy"), recursive=True))
    assert written <= 4096
