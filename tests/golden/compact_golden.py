"""Shrink the SAE training fixtures written by make_golden_{sae,sae_bf16,gated,transcoder}.py to below 1 MB each.

    python tests/golden/compact_golden.py sae_tiny_b.pt [...]

Each named fixture is replaced by ``<name>.xz`` (LZMA-compressed torch.save output; tests/util.py:load_golden reads either form).
On the way, data no test reads is dropped and bit-identical tensors are stored once:
  * ``topk_val`` of every step (the tests compare the TopK indices and the reconstruction, not the raw values);
  * a final gradient equal to its raw gradient (no clipping, no projection on that parameter) shares the raw one's storage;
  * sae_tiny_b / sae_tiny_f: the parameter snapshot after step 2, and sae_tiny_f's gradients of step 3 (those of steps 0 and 5
    stay; every step keeps its losses, indices and reconstruction);
  * sae_bf16_v: the first 3 of the 4 steps of both trajectories (and the data they consume).
"""
import io
import lzma
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
DROP = {"sae_tiny_b.pt": ((2, "params_after"),), "sae_tiny_f.pt": ((2, "params_after"), (3, "raw_grads"), (3, "final_grads"))}
KEEP_STEPS = {"sae_bf16_v.pt": 3}


def _compact(obj, seen):
    if isinstance(obj, dict):
        return {k: _compact(v, seen) for k, v in obj.items() if k != "topk_val"}
    if isinstance(obj, list):
        return [_compact(v, seen) for v in obj]
    if isinstance(obj, torch.Tensor):
        key = (obj.dtype, tuple(obj.shape), obj.contiguous().view(torch.uint8).numpy().tobytes())
        return seen.setdefault(key, obj)
    return obj


def compact(name):
    path = os.path.join(HERE, name)
    gold = torch.load(path, weights_only=False)
    for step, key in DROP.get(name, ()):
        del gold["steps"][step][key]
    if name in KEEP_STEPS:
        n = KEEP_STEPS[name]
        gold.update(n_steps=n, steps=gold["steps"][:n], steps_fp32=gold["steps_fp32"][:n], data=gold["data"][:n * gold["batch"]].clone())
    buf = io.BytesIO()
    torch.save(_compact(gold, {}), buf)
    with open(path + ".xz", "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    os.remove(path)
    print("wrote", path + ".xz", os.path.getsize(path + ".xz"), "bytes")


if __name__ == "__main__":
    for name in sys.argv[1:]:
        compact(name)
