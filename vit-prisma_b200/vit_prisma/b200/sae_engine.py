"""TopK-SAE step engine: owns the device buffers of a training step and drives the six C-ABI calls.

    prep -> encoder GEMM (tcgen05 3xTF32 | exact FFMA) -> topk -> decode/loss -> backward -> adam

Stands in for ``StandardSparseAutoencoder.forward`` + ``loss.backward()`` + ``clip_grad_norm_`` +
``remove_gradient_parallel_to_decoder_directions`` + ``Adam.step`` of the reference
(sae/sae.py:557-645, sae/train_sae.py:278-411).  Nothing here synchronises with the host: the scalars
of a step (mse, grad norm, clip coefficient, l0) stay in an 8-float device buffer that callers read
only when they log.

Parameter storage: the encoder lives feature-major as ``W_encT [F, d]``; the module exposes
``W_enc`` as the transposed view ``W_encT.t()`` so state dicts keep the reference shape ``[d, F]``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from .ops import _need_cuda, _stream, cast as _cast


def ops_cast_f32(x: torch.Tensor) -> torch.Tensor:
    """Activations arrive in cfg.dtype (bf16 stores for reduced-precision configs); the step kernels read fp32."""
    return _cast(x.contiguous(), torch.float32)

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class PbSaeStep(C.Structure):
    _fields_ = (
        [(n, i32) for n in ("rows", "d", "F", "k", "norm_mode", "training", "step", "renorm_decoder")]
        + [(n, f32) for n in ("lr", "beta1", "beta2", "adam_eps", "max_grad_norm")]
        + [(n, vp) for n in (
            "x", "W_encT", "W_encT_lo", "W_dec", "b_enc", "b_dec",
            "sae_in", "mu", "sd", "xsum", "idx", "val", "feat_count", "sae_out", "g", "dval",
            "csc_off", "csc_cursor", "csc_entries", "gW_dec", "gW_encT", "gb_enc", "gb_dec", "gcol", "gbdec2",
            "fired", "scalars", "m_dec", "v_dec", "m_enc", "v_enc", "m_be", "v_be", "m_bd", "v_bd",
            "since_fired", "act_freq")]
        + [("global_rows", i32), ("dist", i32), ("work", vp), ("work_bytes", i64), ("enc_norm_max", vp), ("pre_zeroed", i32), ("W_encT_h", vp)]
    )


class PbSaeEncode(C.Structure):
    """Fused encoder -> TopK call (include/prisma_b200.h, csrc/sae_fused.cu)."""
    _fields_ = (
        [(n, i32) for n in ("rows", "d", "F", "k", "c_keep", "m_cand", "phases")] + [("err_coef", f32)]
        + [(n, vp) for n in ("sae_in", "W_encT", "b_enc", "enc_norm_max", "cand")] + [("cand_bytes", i64)]
        + [(n, vp) for n in ("idx", "val", "feat_count", "fb_count", "fb_rows", "fb_scratch")] + [("fb_scratch_bytes", i64)]
        + [(n, vp) for n in ("sae_in_h", "W_encT_h")]
    )


L.ABI_STRUCTS.append(PbSaeStep)
L.register_signatures({
    "pb_sae_prep": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
    "pb_sae_topk": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, i64, vp]),
    "pb_sae_scatter_acts": (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    "pb_sae_step_reset": (i32, [C.POINTER(PbSaeStep), vp, vp]),
    "pb_sae_decode": (i32, [C.POINTER(PbSaeStep), vp]),
    "pb_sae_backward": (i32, [C.POINTER(PbSaeStep), vp]),
    "pb_sae_adam": (i32, [C.POINTER(PbSaeStep), vp]),
    "pb_unit_norm_rows": (i32, [vp, vp, i32, i32, vp]),
    "pb_sae_mse": (i32, [vp, vp, vp, vp, i32, i32, vp]),
    "pb_sae_fused_workspace": (i32, [i32, i32, i32, C.POINTER(i64), C.POINTER(i64)]),
    "pb_sae_encode_topk_fused": (i32, [C.POINTER(PbSaeEncode), vp]),
    "pb_rownorm_max": (i32, [vp, i32, i32, vp, vp, vp]),
})

NORM_MODE = {"none": 0, None: 0, "layer_norm": 1, "constant_norm_rescale": 2}
SCALAR_NAMES = ("loss_sum", "gnorm_sq", "clip_coef", "mse", "l0", "pos_count", "grad_norm", "reserved")
TOPK_SEG = 256 * 96


def f16_ld(d: int) -> int:
    """Row stride (elements) of the fp16 operand shadows of the fused encoder: rows padded to 16 bytes."""
    return (d + 7) & ~7


def unit_norm_rows_(w: torch.Tensor, w_lo: Optional[torch.Tensor] = None) -> None:
    """In-place ``w /= ||w||_row`` on a contiguous [F, d] fp32 CUDA tensor (+ tf32 residual)."""
    _need_cuda(w)
    assert w.is_contiguous() and w.dtype == torch.float32
    L.check(L.get_lib().pb_unit_norm_rows(w.data_ptr(), None if w_lo is None else w_lo.data_ptr(), w.shape[0], w.shape[1], _stream()),
            "pb_unit_norm_rows")


def sae_prep(x2: torch.Tensor, b_dec: torch.Tensor, norm_mode: str):
    """(norm_in(x) - b_dec, mu [rows], std [rows]) for a contiguous fp32 [rows, d] CUDA tensor."""
    _need_cuda(x2, b_dec)
    rows, d = x2.shape
    sae_in = torch.empty_like(x2)
    mu = torch.empty(rows, device=x2.device)
    sd = torch.empty(rows, device=x2.device)
    L.check(L.get_lib().pb_sae_prep(x2.data_ptr(), b_dec.data_ptr(), sae_in.data_ptr(), None, None, mu.data_ptr(), sd.data_ptr(), None,
                                    rows, d, NORM_MODE[norm_mode], _stream()), "pb_sae_prep")
    return sae_in, mu, sd


def topk_support(hidden_pre2: torch.Tensor, k: int):
    """torch.topk(hidden_pre, k, -1) on the GPU: (idx int32 [rows,k], val [rows,k]) sorted by value descending."""
    _need_cuda(hidden_pre2)
    rows, F = hidden_pre2.shape
    idx = torch.empty(rows, k, dtype=torch.int32, device=hidden_pre2.device)
    val = torch.empty(rows, k, device=hidden_pre2.device)
    nseg = (F + TOPK_SEG - 1) // TOPK_SEG
    scratch = torch.empty(max(rows * nseg * k * 8, 16), dtype=torch.uint8, device=hidden_pre2.device) if F > TOPK_SEG else None
    L.check(L.get_lib().pb_sae_topk(hidden_pre2.data_ptr(), rows, F, k, idx.data_ptr(), val.data_ptr(), None,
                                    None if scratch is None else scratch.data_ptr(), 0 if scratch is None else scratch.numel(),
                                    _stream()), "pb_sae_topk")
    return idx, val


def topk_dense(x: torch.Tensor, k: int) -> torch.Tensor:
    """The TopK activation module's output: zeros_like(x).scatter_(-1, topk idx, relu(topk values))."""
    _need_cuda(x)
    lead, F = x.shape[:-1], x.shape[-1]
    x2 = x.reshape(-1, F).contiguous().float()
    idx, val = topk_support(x2, k)
    dense = torch.empty_like(x2)
    L.check(L.get_lib().pb_sae_scatter_acts(idx.data_ptr(), val.data_ptr(), dense.data_ptr(), x2.shape[0], k, F, 1, _stream()),
            "pb_sae_scatter_acts")
    return dense.view(*lead, F).to(x.dtype)


def sae_mse(x2: torch.Tensor, out2: torch.Tensor) -> torch.Tensor:
    """0-dim device tensor: mean((out - x)^2 / ||x - mean_batch(x)||) (sae.py:144-149)."""
    _need_cuda(x2, out2)
    rows, d = x2.shape
    xsum = torch.empty(d, device=x2.device)
    res = torch.empty(1, device=x2.device)
    L.check(L.get_lib().pb_sae_mse(x2.data_ptr(), out2.data_ptr(), xsum.data_ptr(), res.data_ptr(), rows, d, _stream()), "pb_sae_mse")
    return res[0]


class SaeStepEngine:
    """Buffers + launch sequence for one (d, F, k, rows) geometry.  ``train_step`` mutates the parameters in place."""
    is_data_parallel = False

    def __init__(self, W_encT: torch.Tensor, W_dec: torch.Tensor, b_enc: torch.Tensor, b_dec: torch.Tensor, k: int,
                 normalize_activations: str = "layer_norm", max_grad_norm: float = 1.0, betas=(0.9, 0.999), adam_eps: float = 1e-8,
                 gemm_impl: int = L.GEMM_AUTO, encoder: str = "auto", c_keep: int = 8, m_cand: Optional[int] = None):
        _need_cuda(W_encT, W_dec, b_enc, b_dec)
        for t in (W_encT, W_dec, b_enc, b_dec):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise L.PrismaB200Error("SaeStepEngine: parameters must be contiguous fp32 CUDA tensors")
        self.F, self.d = W_dec.shape
        assert W_encT.shape == (self.F, self.d) and b_enc.shape == (self.F,) and b_dec.shape == (self.d,)
        self.k = int(k)
        self.W_encT, self.W_dec, self.b_enc, self.b_dec = W_encT, W_dec, b_enc, b_dec
        self.norm_mode = NORM_MODE[normalize_activations]
        self.max_grad_norm = float(max_grad_norm or 0.0)
        self.betas, self.adam_eps = betas, adam_eps
        self.gemm_impl = gemm_impl
        dev = W_dec.device
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)  # noqa: E731
        # encoder route: "fused" = one-pass fp16 GEMM with a candidate epilogue + exact re-scoring (csrc/sae_fused.cu, no dense
        # hidden_pre); "dense" = fp32-grade GEMM -> hidden_pre -> k_topk.  "auto" picks fused whenever the geometry allows it and
        # the caller did not pin a GEMM implementation.
        fused_ok = self.d % 4 == 0 and self.d >= 32 and self.F % 128 == 0 and self.k <= 48 and self.F <= 131072
        if encoder == "auto":
            encoder = "fused" if (fused_ok and gemm_impl == L.GEMM_AUTO) else "dense"
        if encoder == "fused" and not fused_ok:
            raise L.PrismaB200Error(f"fused encoder->TopK needs d_in % 4 == 0, d_sae % 128 == 0, k <= 48 (d={self.d} F={self.F} k={self.k})")
        import os
        self.encoder, self.c_keep = encoder, int(os.environ.get("PRISMA_SAE_C_KEEP", c_keep))     # env overrides: tuning runs only
        self.m_cand = int(os.environ.get("PRISMA_SAE_M_CAND", 0)) or (int(m_cand) if m_cand else self.k + 8)   # first round; +16 per round while unproven
        self.enc_norm_max = z(2)                      # max ||w_f||, max ||w_f - f16(w_f)|| (error bound of the fused encoder)
        self.fb_count = z(2, dt=torch.int32)          # rows on the exact path, candidates re-scored (last fused encode)
        self.W_encT_lo = torch.empty_like(W_encT) if encoder == "dense" else None
        # fp16 shadow of W_encT read by the fused encoder's candidate GEMM; rewritten by every Adam step and by refresh_lo()
        self.W_encT_h = z(self.F, f16_ld(self.d), dt=torch.float16) if encoder == "fused" else None
        self.refresh_lo()
        # optimizer state (torch.optim.Adam: exp_avg / exp_avg_sq start at zero)
        self.m_dec, self.v_dec, self.m_enc, self.v_enc = z(self.F, self.d), z(self.F, self.d), z(self.F, self.d), z(self.F, self.d)
        self.m_be, self.v_be, self.m_bd, self.v_bd = z(self.F), z(self.F), z(self.d), z(self.d)
        # gradients
        self.gW_dec, self.gW_encT = torch.empty(self.F, self.d, device=dev), torch.empty(self.F, self.d, device=dev)
        self.gb_enc, self.gb_dec = z(self.F), z(self.d)
        self.gcol, self.gbdec2, self.xsum = z(self.d), z(self.d), z(self.d)
        self.feat_count, self.fired = z(self.F), z(self.F)
        self.csc_off, self.csc_cursor = z(self.F + 1, dt=torch.int32), z(self.F, dt=torch.int32)
        self.scalars = z(8)
        self.step_count = 0
        self._rows = -1

    def refresh_lo(self) -> None:
        """Recompute what the encoder kernels derive from W_enc (after an external write to the parameters): the tf32 residual
        plane of the dense 3xTF32 route; the fused route's fp16 shadow and the encoder-row norm maxima of its error bound."""
        if self.W_encT_lo is not None:
            from . import ops
            self.W_encT_lo.copy_(ops.split_tf32(self.W_encT))
        L.check(L.get_lib().pb_rownorm_max(self.W_encT.data_ptr(), self.F, self.d, self.enc_norm_max.data_ptr(),
                                           None if self.W_encT_h is None else self.W_encT_h.data_ptr(), _stream()), "pb_rownorm_max")

    def _ensure_rows(self, rows: int) -> None:
        if rows == self._rows:
            return
        dev, d, F, k = self.W_dec.device, self.d, self.F, self.k
        e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=dev)  # noqa: E731
        self.sae_in, self.g, self.sae_out = e(rows, d), e(rows, d), e(rows, d)
        self.mu, self.sd = e(rows), e(rows)
        if self.encoder == "fused":
            cb, sb = i64(0), i64(0)
            L.check(L.get_lib().pb_sae_fused_workspace(rows, F, self.c_keep, C.byref(cb), C.byref(sb)), "pb_sae_fused_workspace")
            self.cand = e(max(cb.value // 4, 4), dt=torch.int32)
            self.fb_rows = e(max(rows, 1), dt=torch.int32)
            self.fb_scratch = e(min(64, max(sb.value // (4 * F), 1)) * F)      # exact path: one d_sae row per resident CTA
            self.sae_in_h = torch.zeros(rows, f16_ld(d), dtype=torch.float16, device=dev)
            self.sae_in_lo = self.hidden_pre = None
        else:
            self.sae_in_lo, self.hidden_pre = e(rows, d), e(rows, F)
            self.sae_in_h = None
        self.idx, self.val, self.dval = e(rows, k, dt=torch.int32), e(rows, k), e(rows, k)
        self.csc_entries = e(rows * k, dt=torch.int32)
        self.work = e(8 + 4 * F + 8 * (rows * k // 32 + F + 1) + 64, dt=torch.uint8)   # hot-feature work lists (pb_sae_backward)
        nseg = (F + TOPK_SEG - 1) // TOPK_SEG
        self.topk_scratch = e(max(rows * nseg * k * 8, 16), dt=torch.uint8) if F > TOPK_SEG else None
        self._rows = rows

    def _desc(self, x: torch.Tensor, training: bool, lr: float = 0.0, since_fired=None, act_freq=None, want_out=True) -> PbSaeStep:
        s = PbSaeStep()
        s.rows, s.d, s.F, s.k = x.shape[0], self.d, self.F, self.k
        s.norm_mode, s.training, s.step, s.renorm_decoder = self.norm_mode, int(training), max(self.step_count, 1), 1
        s.lr, s.beta1, s.beta2, s.adam_eps, s.max_grad_norm = lr, self.betas[0], self.betas[1], self.adam_eps, self.max_grad_norm
        p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        s.x = p(x)
        s.W_encT, s.W_encT_lo, s.W_dec, s.b_enc, s.b_dec = p(self.W_encT), p(self.W_encT_lo), p(self.W_dec), p(self.b_enc), p(self.b_dec)
        s.sae_in, s.mu, s.sd, s.xsum = p(self.sae_in), p(self.mu), p(self.sd), p(self.xsum)
        s.idx, s.val, s.feat_count = p(self.idx), p(self.val), p(self.feat_count)
        s.sae_out, s.g, s.dval = (p(self.sae_out) if want_out else None), p(self.g), p(self.dval)
        s.csc_off, s.csc_cursor, s.csc_entries = p(self.csc_off), p(self.csc_cursor), p(self.csc_entries)
        s.gW_dec, s.gW_encT, s.gb_enc, s.gb_dec = p(self.gW_dec), p(self.gW_encT), p(self.gb_enc), p(self.gb_dec)
        s.gcol, s.gbdec2, s.fired, s.scalars = p(self.gcol), p(self.gbdec2), p(self.fired), p(self.scalars)
        s.m_dec, s.v_dec, s.m_enc, s.v_enc = p(self.m_dec), p(self.v_dec), p(self.m_enc), p(self.v_enc)
        s.m_be, s.v_be, s.m_bd, s.v_bd = p(self.m_be), p(self.v_be), p(self.m_bd), p(self.v_bd)
        s.since_fired, s.act_freq = p(since_fired), p(act_freq)
        s.work, s.work_bytes = p(self.work), self.work.numel()
        s.enc_norm_max = p(self.enc_norm_max)
        s.W_encT_h = p(self.W_encT_h)
        return s

    def _enc_desc(self, rows: int, phases: int = 0) -> PbSaeEncode:
        e = PbSaeEncode()
        e.rows, e.d, e.F, e.k, e.c_keep, e.m_cand, e.phases, e.err_coef = rows, self.d, self.F, self.k, self.c_keep, self.m_cand, phases, 0.0
        e.sae_in, e.W_encT, e.b_enc, e.enc_norm_max = self.sae_in.data_ptr(), self.W_encT.data_ptr(), self.b_enc.data_ptr(), self.enc_norm_max.data_ptr()
        e.cand, e.cand_bytes = self.cand.data_ptr(), self.cand.numel() * 4
        e.idx, e.val, e.feat_count = self.idx.data_ptr(), self.val.data_ptr(), self.feat_count.data_ptr()
        e.fb_count, e.fb_rows = self.fb_count.data_ptr(), self.fb_rows.data_ptr()
        e.fb_scratch, e.fb_scratch_bytes = self.fb_scratch.data_ptr(), self.fb_scratch.numel() * 4
        e.sae_in_h, e.W_encT_h = self.sae_in_h.data_ptr(), self.W_encT_h.data_ptr()
        return e

    # ------------------------------------------------------------------ pieces
    def _encoder_gemm(self, rows: int) -> None:
        """hidden_pre = sae_in @ W_enc + b_enc (sae.py:568) on the tcgen05 GEMM (3xTF32) or the exact FFMA kernel."""
        lib, st = L.get_lib(), _stream()
        use_tc = self.gemm_impl != L.GEMM_SIMT
        g = L.PbGemm()
        g.M, g.N, g.K, g.dtype, g.impl = rows, self.F, self.d, L.PB_F32, self.gemm_impl
        g.A, g.lda, g.B, g.ldb = self.sae_in.data_ptr(), self.d, self.W_encT.data_ptr(), self.d
        if use_tc:
            g.A_lo, g.B_lo = self.sae_in_lo.data_ptr(), self.W_encT_lo.data_ptr()
        g.bias, g.out0, g.ld0 = self.b_enc.data_ptr(), self.hidden_pre.data_ptr(), self.F
        L.check(lib.pb_gemm(C.byref(g), st), "pb_gemm(encoder)")

    def encode_topk(self, x: torch.Tensor, pre_zeroed: bool = False) -> None:
        """prep + encoder GEMM + topk; fills sae_in, mu, sd, xsum, hidden_pre, idx, val, feat_count.
        ``pre_zeroed``: the caller already ran ``pb_sae_step_reset`` (feat_count and fb_count are zero)."""
        lib, st = L.get_lib(), _stream()
        rows = x.shape[0]
        self._ensure_rows(rows)
        L.check(lib.pb_sae_prep(x.data_ptr(), self.b_dec.data_ptr(), self.sae_in.data_ptr(),
                                self.sae_in_lo.data_ptr() if (self.sae_in_lo is not None and self.gemm_impl != L.GEMM_SIMT) else None,
                                None if self.sae_in_h is None else self.sae_in_h.data_ptr(), self.mu.data_ptr(), self.sd.data_ptr(),
                                self.xsum.data_ptr(), rows, self.d, self.norm_mode, st), "pb_sae_prep")
        if not pre_zeroed:
            self.feat_count.zero_()
        if self.encoder == "fused":
            L.check(lib.pb_sae_encode_topk_fused(C.byref(self._enc_desc(rows, 8 if pre_zeroed else 0)), st), "pb_sae_encode_topk_fused")
            return
        self._encoder_gemm(rows)
        scratch = self.topk_scratch
        L.check(lib.pb_sae_topk(self.hidden_pre.data_ptr(), rows, self.F, self.k, self.idx.data_ptr(), self.val.data_ptr(),
                                self.feat_count.data_ptr(), None if scratch is None else scratch.data_ptr(),
                                0 if scratch is None else scratch.numel(), st), "pb_sae_topk")

    @torch.no_grad()
    def forward(self, x: torch.Tensor, want_out: bool = True):
        """Inference: encode -> topk -> decode -> mse.  Returns (sae_out | None, idx, val); scalars[3] = mse."""
        _need_cuda(x)
        x = ops_cast_f32(x)
        self.encode_topk(x)
        self.scalars.zero_()
        s = self._desc(x, training=False, want_out=want_out)
        L.check(L.get_lib().pb_sae_decode(C.byref(s), _stream()), "pb_sae_decode")
        return (self.sae_out if want_out else None), self.idx, self.val

    @torch.no_grad()
    def train_step(self, x: torch.Tensor, lr: float, since_fired: Optional[torch.Tensor] = None,
                   act_freq: Optional[torch.Tensor] = None, want_out: bool = False) -> torch.Tensor:
        """One optimizer step on batch ``x`` [rows, d].  Returns the 8-float device scalars buffer (no sync)."""
        _need_cuda(x)
        x = ops_cast_f32(x)
        lib, st = L.get_lib(), _stream()
        self._ensure_rows(x.shape[0])
        self.step_count += 1
        s = self._desc(x, training=True, lr=float(lr), since_fired=since_fired, act_freq=act_freq, want_out=want_out)
        s.pre_zeroed = 1
        L.check(lib.pb_sae_step_reset(C.byref(s), self.fb_count.data_ptr(), st), "pb_sae_step_reset")     # every accumulator of the step, one launch
        self.encode_topk(x, pre_zeroed=True)
        L.check(lib.pb_sae_decode(C.byref(s), st), "pb_sae_decode")
        L.check(lib.pb_sae_backward(C.byref(s), st), "pb_sae_backward")
        L.check(lib.pb_sae_adam(C.byref(s), st), "pb_sae_adam")
        return self.scalars

    # ------------------------------------------------------------------ instrumentation (bench.py / tools)
    def describe_encoder(self) -> str:
        if self.encoder == "fused":
            return (f"fused: one-pass fp16 tcgen05 GEMM (kind::f16) with top-{self.c_keep}-per-128-features epilogue -> exact fp32 re-scoring of "
                    f">= {self.m_cand} candidates per token -> exact top-{self.k} with a completeness proof (no dense hidden_pre)")
        return "tcgen05 3xTF32 GEMM -> dense hidden_pre -> exact k_topk" if self.gemm_impl != L.GEMM_SIMT else "exact FFMA GEMM -> k_topk"

    def fallback_rows(self) -> int:
        """Rows of the last fused encode that took the exact path (host read: synchronises)."""
        return int(self.fb_count[0].item()) if self.encoder == "fused" else 0

    def rescored_per_row(self, rows: int) -> float:
        """Mean number of candidates re-scored exactly per proven row in the last fused encode (host read: synchronises)."""
        fb, tot = self.fb_count.tolist()
        return tot / max(rows - fb, 1)

    def _optimizer_stages(self, s: PbSaeStep, x: torch.Tensor, lr: float, since_fired, act_freq):
        """(name, callable, info) of the stages after backward; the data-parallel engine replaces them with its peer-memory phases."""
        lib, st = L.get_lib(), _stream()
        return [("adam (clip + decoder-parallel-gradient removal + Adam + row renorm)", lambda: L.check(lib.pb_sae_adam(C.byref(s), st)),
                 dict(bytes=60 * self.d * self.F, ncu=r"k_sae_adam_rows"))]

    @torch.no_grad()
    def time_stages(self, x: torch.Tensor, lr: float, since_fired=None, act_freq=None, reps: int = 5) -> dict:
        """CUDA-event time of every stage of one training step, each replayed ``reps`` times back to back on the current stream
        (warm caches: shares of the step, not cold-start figures).  Mutates parameters / optimizer state like ``reps`` extra steps.
        Returns ``{stage: {"ms", "bytes" | "flops" (algorithmic, per launch), "ncu" (kernel-name regex for profiles/)}}``."""
        lib, st = L.get_lib(), _stream()
        x = ops_cast_f32(x)
        rows = x.shape[0]
        out = {}

        def timed(name, fn, **info):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            out[name] = dict(ms=a.elapsed_time(b) / reps, **info)

        for name, fn, info in self._encode_stages(x):
            timed(name, fn, **info)
        self.encode_topk(x)
        self.scalars.zero_()
        self.step_count += 1
        s = self._desc(x, training=True, lr=float(lr), since_fired=since_fired, act_freq=act_freq, want_out=False)
        self._prepare_timed_step(s, x)
        timed("decode (sparse decode + loss + d_hidden)", lambda: L.check(lib.pb_sae_decode(C.byref(s), st)),
              bytes=(12 * rows * self.d + 8 * rows * self.k), ncu=r"k_sae_decode")
        timed("backward (csc build + per-feature gradients + norm)", lambda: (self.scalars.zero_(), L.check(lib.pb_sae_backward(C.byref(s), st))),
              bytes=8 * self.d * self.F, ncu=r"k_sae_grads<")
        for name, fn, info in self._optimizer_stages(s, x, float(lr), since_fired, act_freq):
            timed(name, fn, **info)
        return out

    def _prepare_timed_step(self, s: PbSaeStep, x: torch.Tensor) -> None:
        pass

    def _encode_stages(self, x: torch.Tensor):
        rows = x.shape[0]
        if self.encoder == "fused":
            lib, st = L.get_lib(), _stream()
            self.encode_topk(x)
            flops = 2.0 * rows * self.d * self.F
            nkeys = (self.F // 128) * self.c_keep
            return [("encode + topk, fused (prep + fp16 candidate GEMM + select / exact re-score + exact path)", lambda: self.encode_topk(x),
                     dict(flops=flops, passes=1)),
                    ("candidate GEMM alone (one fp16 pass, top-c-per-segment epilogue)",
                     lambda: L.check(lib.pb_sae_encode_topk_fused(C.byref(self._enc_desc(rows, 1)), st)),
                     dict(flops=flops, passes=1, bytes=2 * self.d * self.F + 2 * rows * self.d + 4 * rows * nkeys, ncu=r"k_enc_cand")),
                    ("select + exact re-score alone", lambda: L.check(lib.pb_sae_encode_topk_fused(C.byref(self._enc_desc(rows, 2)), st)),
                     dict(bytes=4 * rows * nkeys + 4 * rows * self.d + 8 * rows * self.k, ncu=r"k_cand_select"))]
        return [("encode + topk (prep + encoder GEMM 3xTF32 + exact topk)", lambda: self.encode_topk(x),
                 dict(flops=2.0 * rows * self.d * self.F, passes=3, ncu=r"k_gemm_tc2<float")),
                ("encoder GEMM alone (hidden_pre = sae_in @ W_enc + b_enc)", lambda: self._encoder_gemm(rows),
                 dict(flops=2.0 * rows * self.d * self.F, passes=3, bytes=8 * self.d * self.F + 8 * rows * self.d + 4 * rows * self.F))]

    def dense_feature_acts(self) -> torch.Tensor:
        """feature_acts [rows, F] of the last encode (zeros.scatter_(idx, relu(val)))."""
        rows = self.idx.shape[0]
        dense = torch.empty(rows, self.F, device=self.W_dec.device)
        L.check(L.get_lib().pb_sae_scatter_acts(self.idx.data_ptr(), self.val.data_ptr(), dense.data_ptr(), rows, self.k, self.F, 1,
                                                _stream()), "pb_sae_scatter_acts")
        return dense

    def scalars_dict(self) -> dict:
        """Host read (synchronises): for logging / tests only."""
        vals = self.scalars.tolist()
        return dict(zip(SCALAR_NAMES, vals))

    # algorithmic HBM bytes of one training step (SURVEY section 8d): 80*d*F + 8*Bt*d
    def algorithmic_bytes(self, rows: int) -> int:
        return 80 * self.d * self.F + 8 * rows * self.d
