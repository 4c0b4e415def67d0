"""bench.py contract checks that need no GPU: the reference arm prints one well-formed JSON line from the CPU oracle port, and
the product arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "cpu_baseline", "e2e")


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True, timeout=900, env=e)


@pytest.mark.parametrize("workload", ["vit", "sae", "cfg5", "sae_fwd"])
def test_reference_arm_prints_one_json_line(workload):
    out = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--workload", workload)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["vs_baseline"] is None and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    assert (d["unit"], d["config"]["workload"][:3]) == (("images/s", "vit") if workload == "vit" else ("tokens/s", "sae"))


def test_reference_arm_nonzero_ranks_exit_quietly():
    out = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--gpus", "2", env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_output_dump_samples_the_same_positions_and_stays_under_budget(tmp_path):
    """--dump-outputs: float32 for floating point (bf16 included), float64 for integers, large arrays sampled at positions that do
    not change from run to run, and a refusal instead of writing more than OutputDump.BUDGET."""
    import numpy as np
    from bench import OutputDump
    g = torch.Generator().manual_seed(1)
    x, n = torch.randn(3_000_000, generator=g), torch.arange(12, dtype=torch.int32).reshape(3, 4)
    for run in ("a", "b"):
        dump = OutputDump(str(tmp_path / run))
        dump.add("big", x)
        dump.add("small", x[:10].bfloat16())
        dump.add("idx", n)
        dump.add("absent", None)
        dump.write()
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "idx.npy", "small.npy"] and files == sorted(os.listdir(tmp_path / "b"))
    big, idx, small = (np.load(tmp_path / "a" / f) for f in files)
    assert big.dtype == np.float32 and big.shape == (1 << 20,) and np.array_equal(big, np.load(tmp_path / "b" / "big.npy"))
    assert np.isin(big, x.numpy()).all()
    assert idx.dtype == np.float64 and np.array_equal(idx, n.numpy())
    assert small.dtype == np.float32 and small.shape == (10,)
    dump = OutputDump(str(tmp_path / "c"))
    for i in range(17):
        dump.add(f"a{i}", x)
    with pytest.raises(SystemExit):
        dump.write()
    assert not (tmp_path / "c").exists()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU refusal")
def test_product_arm_fails_loudly_without_a_gpu():
    out = _run("--steps", "1", "--warmup", "1")
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
