"""Parity helpers shared by the tests (SURVEY section 7 step 1)."""
import io
import lzma
import os

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    """tests/golden/<name>, or its LZMA-compressed form <name>.xz (golden/compact_golden.py)."""
    path = os.path.join(GOLDEN, name)
    if os.path.exists(path):
        return torch.load(path, weights_only=False)
    with open(path + ".xz", "rb") as f:
        return torch.load(io.BytesIO(lzma.decompress(f.read())), weights_only=False)


def rel_err(got: torch.Tensor, ref: torch.Tensor) -> float:
    """max |got - ref| relative to max |ref| of the tensor (the metric north_star's 1e-4 / 1e-2 refer to)."""
    got = got.detach().to("cpu", torch.float64)
    ref = ref.detach().to("cpu", torch.float64)
    denom = max(ref.abs().max().item(), 1e-30)
    return (got - ref).abs().max().item() / denom


def assert_close(got, ref, tol, what=""):
    assert tuple(got.shape) == tuple(ref.shape), f"{what}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    assert got.dtype == ref.dtype, f"{what}: dtype {got.dtype} != {ref.dtype}"
    e = rel_err(got, ref)
    assert e <= tol, f"{what}: rel err {e:.3e} > {tol:.1e}"
    return e
