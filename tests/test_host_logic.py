"""CPU-side tests: hook runtime, cache container, config surface, C-ABI presence.  No kernel is launched."""
import ctypes
import re
import os

import pytest
import torch
import torch.nn as nn

from vit_prisma.configs.HookedViTConfig import HookedViTConfig
from vit_prisma.models.base_vit import HookedViT
from vit_prisma.prisma_tools.activation_cache import ActivationCache
from vit_prisma.prisma_tools.hook_point import HookPoint
from vit_prisma.prisma_tools.hooked_root_module import HookedRootModule
from vit_prisma.utils.prisma_utils import get_act_name
from tests.util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Toy(HookedRootModule):
    """HookPoints only -- lets the hook lifetime rules run without any arithmetic."""

    def __init__(self):
        super().__init__()
        self.hook_a = HookPoint()
        self.inner = nn.ModuleDict({"hook_b": HookPoint()})
        self.hook_c = HookPoint()
        self.setup()

    def forward(self, x):
        x = self.hook_a(x)
        x = self.inner["hook_b"](x)
        self.hook_c(x)            # observer: result ignored
        return x


class Counter:
    def __init__(self):
        self.count = 0

    def inc(self, *a, **k):
        self.count += 1


def test_setup_names_and_order():
    m = Toy()
    assert list(m.hook_dict) == ["hook_a", "inner.hook_b", "hook_c"]
    assert m.hook_dict["inner.hook_b"].name == "inner.hook_b"


def test_inert_fast_exit_and_replacement_semantics():
    m = Toy()
    x = torch.ones(3)
    assert m(x) is x                               # inert points return the very same tensor
    m.add_hook("hook_a", lambda t, hook: t + 1)    # non-None return replaces the activation
    m.add_hook("hook_c", lambda t, hook: t * 100)  # observer output is discarded by the model
    assert torch.equal(m(x), x + 1)
    m.reset_hooks()
    assert all(hp.is_inert for hp in m.hook_points())


def test_context_levels_and_exception_unwinding():
    m, c = Toy(), Counter()
    sel = lambda n: n == "hook_a"  # noqa: E731
    with m.hooks(fwd_hooks=[(sel, c.inc)]):
        with pytest.raises(ValueError):
            with m.hooks(fwd_hooks=[(sel, lambda t, hook: (_ for _ in ()).throw(ValueError("x")))]):
                assert len(m.hook_a.fwd_hooks) == 2
                m(torch.ones(1))
        assert len(m.hook_a.fwd_hooks) == 1 and m.context_level == 1
    assert len(m.hook_a.fwd_hooks) == 0 and m.context_level == 0 and c.count == 1


def test_perma_hooks_survive_reset_and_prepend_orders():
    m = Toy()
    order = []
    m.add_perma_hook("hook_a", lambda t, hook: order.append("perma"))
    m.add_hook("hook_a", lambda t, hook: order.append("late"))
    m.add_hook("hook_a", lambda t, hook: order.append("first"), prepend=True)
    m(torch.ones(1))
    assert order == ["first", "perma", "late"]
    m.reset_hooks()
    assert len(m.hook_a.fwd_hooks) == 1
    m.remove_all_hook_fns(including_permanent=True)
    assert len(m.hook_a.fwd_hooks) == 0


def test_run_with_cache_generic_path_filters_and_batch_dim():
    m = Toy()
    x = torch.arange(4.0).view(1, 4)
    out, cache = m.run_with_cache(x, names_filter=["hook_a", "hook_c"], remove_batch_dim=True)
    assert list(cache) == ["hook_a", "hook_c"] and cache["hook_a"].shape == (4,)
    out, cache = m.run_with_cache(x, names_filter="inner.hook_b")
    assert list(cache) == ["inner.hook_b"]
    out, cache = m.run_with_cache(x, names_filter=lambda n: n.startswith("hook_"))
    assert list(cache) == ["hook_a", "hook_c"]
    assert all(hp.is_inert for hp in m.hook_points())
    with pytest.raises(ValueError):
        m.hook_a.add_hook(lambda t, hook: t, dir="sideways")


def test_get_act_name_shorthand():
    assert get_act_name("k", 6, "a") == "blocks.6.attn.hook_k"
    assert get_act_name("pre", 2) == "blocks.2.mlp.hook_pre"
    assert get_act_name("embed") == "hook_embed"
    assert get_act_name("normalized", 27, "ln2") == "blocks.27.ln2.hook_normalized"
    assert get_act_name("k6") == "blocks.6.attn.hook_k"
    assert get_act_name("scale4ln1") == "blocks.4.ln1.hook_scale"
    assert get_act_name("pre5") == "blocks.5.mlp.hook_pre"
    assert get_act_name("scale") == "ln_final.hook_scale"
    assert get_act_name("blocks.3.hook_resid_post") == "blocks.3.hook_resid_post"
    assert get_act_name("attn", 1) == "blocks.1.attn.hook_pattern"


def test_activation_cache_container():
    class M:
        cfg = HookedViTConfig(n_layers=3, d_model=4, d_head=2, d_mlp=8)
    d = {"hook_embed": torch.zeros(1, 2, 4), "blocks.2.hook_resid_post": torch.ones(1, 2, 4), "blocks.0.attn.hook_q": torch.ones(1, 2, 2, 2)}
    c = ActivationCache(dict(d), M())
    assert c["embed"] is d["hook_embed"] and c["resid_post", -1] is d["blocks.2.hook_resid_post"] and c["q", 0] is d["blocks.0.attn.hook_q"]
    assert len(c) == 3 and list(c) == list(d) and list(c.keys()) == list(d)
    with pytest.raises(KeyError):
        c["blocks.9.hook_resid_post"]
    c.remove_batch_dim()
    assert c["embed"].shape == (2, 4) and not c.has_batch_dim


def test_config_positional_order_and_fields():
    cfg = HookedViTConfig(1, 8, 4, 16, return_type="logits")
    assert (cfg.n_layers, cfg.d_model, cfg.d_head, cfg.d_mlp) == (1, 8, 4, 16)
    assert cfg.n_heads == 4 and cfg.eps == 1e-6 and cfg.patch_size == 32 and cfg.image_size == 224 and cfg.n_classes == 10
    assert cfg.layer_norm_pre is False and cfg.normalize_output is False and cfg.dtype == torch.float32
    assert HookedViTConfig.from_dict({"n_layers": 2, "d_model": 4, "d_head": 2, "d_mlp": 8}).n_layers == 2
    assert cfg.n_tokens == 50


def test_weight_property_shapes_and_state_dict_layout():
    for conf in (HookedViTConfig(n_layers=3, d_head=32, d_model=64, d_mlp=128, n_heads=2, patch_size=4),
                 HookedViTConfig(n_layers=2, d_head=16, d_model=128, d_mlp=300, n_heads=8, patch_size=16)):
        m = HookedViT(conf)
        L, H, d, dh, M = conf.n_layers, conf.n_heads, conf.d_model, conf.d_head, conf.d_mlp
        for name in ("W_Q", "W_K", "W_V"):
            assert getattr(m, name).shape == (L, H, d, dh)
        assert m.W_O.shape == (L, H, dh, d) and m.W_in.shape == (L, d, M) and m.W_out.shape == (L, M, d)
        assert m.W_E.shape == (d, conf.n_channels, conf.patch_size, conf.patch_size) and m.W_H.shape == (d, conf.n_classes)
        for name in ("b_Q", "b_K", "b_V"):
            assert getattr(m, name).shape == (L, H, dh)
        assert m.b_O.shape == (L, d) and m.b_in.shape == (L, M) and m.b_out.shape == (L, d) and m.b_H.shape == (conf.n_classes,)
    gold = load_golden("vit_tiny_a_fp32.pt")
    m = HookedViT(HookedViTConfig(**gold["cfg"]))
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == gold["shapes"]
    assert len(m.hook_dict) == 2 * 23 + 10      # 23 hook points per block (6 conditional) + 10 model-level = 286 for ViT-B (SURVEY 8a2)


def test_conditional_hook_gates_on_cpu():
    m = HookedViT(HookedViTConfig(1, 8, 8, 8))
    with pytest.raises(AssertionError):
        m.add_hook("blocks.0.attn.hook_result", lambda t, hook: t)
    m.set_use_attn_result(True)
    m.add_hook("blocks.0.attn.hook_result", lambda t, hook: t)
    m.reset_hooks()


_REFUSAL = """
import pytest, torch
from vit_prisma.b200._lib import PrismaB200Error
from vit_prisma.configs.HookedViTConfig import HookedViTConfig
from vit_prisma.models.base_vit import HookedViT
assert not torch.cuda.is_available()
m = HookedViT(HookedViTConfig(1, 8, 8, 8))
with pytest.raises(PrismaB200Error, match="no CPU fallback"):
    m(torch.rand(1, 3, 224, 224))
with pytest.raises(PrismaB200Error):
    m.run_with_cache(torch.rand(1, 3, 224, 224))
print("refused")
"""


def test_product_path_refuses_cpu_tensors():
    """With no CUDA device visible, a call on host tensors raises instead of computing on the host.  (With one, a host-resident
    model is staged on the GPU instead, DESIGN.md section 1.)  Run in a child process that sees no device, so that the refusal is
    checked on machines with a GPU too."""
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "vit-prisma_b200"), env.get("PYTHONPATH", "")])
    out = subprocess.run([sys.executable, "-c", _REFUSAL], env=env, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("refused"), (out.stdout + out.stderr)[-3000:]


def test_c_abi_library_exports_every_declared_symbol():
    from vit_prisma.b200 import _lib as L
    from vit_prisma.b200 import p2p, sae_dense, sae_engine, sae_gated  # noqa: F401  (register the SAE / P2P entry points)
    header = open(os.path.join(ROOT, "include", "prisma_b200.h")).read()
    declared = set(re.findall(r"PB_API\s+[\w\s\*]+?\b(pb_\w+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(str(L.LIB_PATH))
    missing = [name for name in declared if not hasattr(lib, name)]
    assert not missing, f"declared in include/prisma_b200.h but not exported: {missing}"
    unbound = declared - set(L.SIGNATURES)
    assert not unbound, f"declared in the header but no ctypes signature: {unbound}"


def test_c_abi_struct_layouts_match_the_compiled_library():
    from vit_prisma.b200 import _lib as L
    from vit_prisma.b200 import p2p, sae_engine  # noqa: F401  (append PbSaeStep / PbP2PStep to ABI_STRUCTS)
    lib = ctypes.CDLL(str(L.LIB_PATH))
    lib.pb_abi_sizeof.restype = ctypes.c_int
    assert len(L.ABI_STRUCTS) == 10
    for idx, struct in enumerate(L.ABI_STRUCTS):
        if struct is None:      # device-side only struct
            assert lib.pb_abi_sizeof(idx) > 0
            continue
        assert lib.pb_abi_sizeof(idx) == ctypes.sizeof(struct), struct.__name__
    assert lib.pb_abi_sizeof(10_000) == -1


def test_product_synthetic_recipe_equals_the_oracle_recipe():
    """bench.py / smoke() build product models from vit_prisma.b200.synthetic; the CPU checker restates the same recipe in oracle/."""
    from oracle import vit_oracle
    from vit_prisma.b200 import synthetic
    assert synthetic.CLIP_B32 == vit_oracle.CLIP_B32 and synthetic.CLIP_L14 == vit_oracle.CLIP_L14
    tiny = dict(vit_oracle.CLIP_B32, n_layers=1, d_model=16, d_head=8, n_heads=2, d_mlp=32, patch_size=16, image_size=32, n_classes=5)
    shapes = vit_oracle.state_dict_shapes(tiny)
    a, b = synthetic.recipe_state_dict(shapes, 99), vit_oracle.recipe_state_dict(shapes, 99)
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)


def test_c_abi_header_is_plain_c(tmp_path):
    """include/prisma_b200.h is the drop-in boundary: it must compile as C99 (and as C++) with nothing but the standard headers --
    no torch, no CUDA headers, no C++-only constructs."""
    import shutil
    import subprocess
    src = tmp_path / "hdr.c"
    src.write_text('#include "prisma_b200.h"\nint main(void) { return (int)sizeof(PbGemm) == 0; }\n')
    inc = os.path.join(ROOT, "include")
    for cc, flags in (("gcc", ["-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror"]), ("g++", ["-x", "c++", "-std=c++11", "-Wall", "-Werror"])):
        if shutil.which(cc) is None:
            pytest.skip(f"{cc} not available")
        out = subprocess.run([cc, *flags, "-fsyntax-only", f"-I{inc}", str(src)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
