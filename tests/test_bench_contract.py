"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm (the reference's own
CPU code from oracle/_ref) prints one JSON line with the agreed keys, and the GPU arm refuses to run on a CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libryg_ref.so")

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


@pytest.mark.skipif(not os.path.exists(REF_LIB), reason="oracle/_ref was not built (it needs the reference checkout)")
@pytest.mark.parametrize("workload", ["uniform_1GiB_word32", "zipf1.1_1GiB_alias32"])
def test_reference_arm_prints_the_contract_line(workload):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "2",
                          "--warmup", "1", "--size", str(4 << 20)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1                                           # ONE JSON line
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference" and d["gpu_launches"] == 0
    assert d["unit"] == "Gsymbols/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"] == workload
    assert d["steps"] == 2 and d["warmup"] == 1                    # the repetitions actually run, on the whole --size
    assert d["config"]["symbols_per_gpu"] == 4 << 20 and d["config"]["symbols_per_step"] == 4 << 20
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_gpu_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--size", str(1 << 20)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert "no CPU fallback" in out.stderr
    assert not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]      # and no number


def test_dump_outputs_writes_exact_seeded_samples(tmp_path):
    """--dump-outputs: byte arrays as float32, offsets as float64, both exact; an array too large for the per-array
    budget becomes the same seeded sample of distinct positions on every run and its file stays within the budget."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    big = torch.randint(0, 256, (bench.DUMP_BYTES // 4 + 1001,), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    outputs = {"blob": torch.arange(200, dtype=torch.uint8), "offsets": torch.tensor([0, 4096, (1 << 40) + 3]), "decoded": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outputs)
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in outputs}
    assert a["blob"].dtype == np.float32 and np.array_equal(a["blob"], np.arange(200))
    assert a["offsets"].dtype == np.float64 and a["offsets"].tolist() == [0, 4096, (1 << 40) + 3]
    assert a["decoded"].dtype == np.float32 and a["decoded"].size == bench.DUMP_BYTES // 4
    assert np.array_equal(a["decoded"], np.load(tmp_path / "b" / "decoded.npy"))
    positions = np.sort(np.random.default_rng(0).choice(big.numel(), a["decoded"].size, replace=False))
    assert np.unique(positions).size == positions.size and np.array_equal(a["decoded"], big.numpy()[positions])
    assert (tmp_path / "a" / "decoded.npy").stat().st_size <= bench.DUMP_BYTES + 128
