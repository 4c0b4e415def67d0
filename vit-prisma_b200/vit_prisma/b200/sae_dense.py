"""Dense-activation SAE training step (ReLU + L1) and the ghost-grad auxiliary loss, on the C-ABI kernels.

Stands in for ``StandardSparseAutoencoder.forward`` + ``VisionSAETrainer.train_step`` when ``activation_fn_str == "relu"``
(the reference's default; sae/sae.py:557-645, 810-839) and for ``_compute_ghost_residual_loss`` (sae/sae.py:151-179) with
either activation.  The six dense products of the reference graph run on ``pb_gemm`` (tcgen05, 3xTF32, K-major operands:
``pb_transpose`` supplies the transposed views autograd uses); ``csrc/sae_dense.cu`` holds the glue; clip / projection /
Adam / renorm / dead-feature counters are ``pb_sae_adam``, shared with the TopK pipeline.

Per step (tokens Bt, d = d_in, F = d_sae):
  prep -> hidden_pre, acts = relu(.) [GEMM + epilogue] -> stats -> out_n = acts @ W_dec + b_dec [GEMM] -> loss, g
  d_acts = g @ W_dec^T [GEMM] -> d_hid = (d_acts + l1/Bt) * [acts > 0]
  gW_dec = acts^T @ g [GEMM], gW_encT = d_hid^T @ sae_in [GEMM], gb_enc = colsum(d_hid), gb_dec = colsum(g) - gb_enc @ W_enc^T
  (+ ghost blocks on the dead features) -> grad norm / clip -> pb_sae_adam
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from . import ops
from .sae_engine import SaeStepEngine, _need_cuda, _stream

i32, i64, f32, vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p

L.register_signatures({
    "pb_transpose": (i32, [vp, vp, vp, i32, i32, vp]),
    "pb_colsum": (i32, [vp, vp, i32, i32, i32, vp]),
    "pb_gemv_rows": (i32, [vp, vp, vp, i32, i32, i32, vp]),
    "pb_sae_dense_stats": (i32, [vp, i32, i32, vp, vp, vp, vp]),
    "pb_sae_dense_loss": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]),
    "pb_sae_dense_dhid": (i32, [vp, vp, vp, f32, i64, vp]),
    "pb_sae_grad_finish": (i32, [vp, vp, vp, vp, i32, i32, vp, f32, i32, vp]),
    "pb_sae_ghost_gather": (i32, [vp, vp, i32, i32, i32, vp, i32, vp]),
    "pb_gather_rows": (i32, [vp, vp, i32, i32, i32, vp, vp]),
    "pb_scatter_add_rows": (i32, [vp, vp, i32, i32, vp, f32, vp]),
    "pb_mul_inplace": (i32, [vp, vp, i64, vp]),
    "pb_sae_ghost_rows": (i32, [vp, vp, vp, vp, vp, i32, i32, vp]),
})


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def transpose(x: torch.Tensor, want_lo: bool = True):
    """[rows, cols] fp32 -> ([cols, rows], its tf32 residual | None)."""
    _need_cuda(x)
    assert x.dim() == 2 and x.dtype == torch.float32 and x.is_contiguous()
    rows, cols = x.shape
    out = torch.empty(cols, rows, device=x.device)
    lo = torch.empty(cols, rows, device=x.device) if want_lo else None
    L.check(L.get_lib().pb_transpose(x.data_ptr(), out.data_ptr(), _p(lo), rows, cols, _stream()), "pb_transpose")
    return out, lo


def colsum(x: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    rows, cols = x.shape
    out = torch.empty(cols, device=x.device) if out is None else out
    L.check(L.get_lib().pb_colsum(x.data_ptr(), out.data_ptr(), rows, cols, int(accumulate), _stream()), "pb_colsum")
    return out


def gemv_rows(W: torch.Tensor, v: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    F, d = W.shape
    out = torch.empty(d, device=W.device) if out is None else out
    L.check(L.get_lib().pb_gemv_rows(W.data_ptr(), v.data_ptr(), out.data_ptr(), F, d, int(accumulate), _stream()), "pb_gemv_rows")
    return out


_GEMM_IMPL = [L.GEMM_AUTO]          # the engine's gemm_impl while one of its steps runs (GEMM_SIMT = exact-fp32 cross-check route)


class _gemm_impl:
    def __init__(self, impl: int):
        self.impl = impl

    def __enter__(self):
        _GEMM_IMPL.append(self.impl)

    def __exit__(self, *exc):
        _GEMM_IMPL.pop()


def gemm32(a: torch.Tensor, a_lo: Optional[torch.Tensor], b_nk: torch.Tensor, b_lo: Optional[torch.Tensor], bias=None, act=None,
           out0=None, out1=None, want_pre=True):
    """fp32-grade ``a @ b_nk.T``: 3xTF32 tensor-core GEMM when both operands come with their residual planes and the shape is
    TMA-legal, the exact FFMA kernel otherwise (pb_gemm's AUTO rule)."""
    impl = _GEMM_IMPL[-1]
    if impl == L.GEMM_SIMT:
        return ops.gemm(a, b_nk, bias, act=act, out0=out0, out1=out1, want_pre=want_pre, want_post=out1 is not None, impl=impl)
    if a_lo is None:
        a_lo = ops.split_tf32(a)
    if b_lo is None:
        b_lo = ops.split_tf32(b_nk)
    return ops.gemm(a, b_nk, bias, act=act, a_lo=a_lo, w_lo=b_lo, out0=out0, out1=out1, want_pre=want_pre, want_post=out1 is not None)


def ghost_loss_value(hidden_pre: torch.Tensor, W_dec: torch.Tensor, x2: torch.Tensor, sae_out2: torch.Tensor, mse: torch.Tensor,
                     dead_mask: torch.Tensor) -> torch.Tensor:
    """``_compute_ghost_residual_loss`` (sae/sae.py:151-179) as a 0-dim device tensor, for ``forward()``'s 7-tuple.
    hidden_pre [rows, F], x2 / sae_out2 [rows, d] fp32 contiguous; ``mse`` 0-dim device tensor; ``dead_mask`` [F] bool."""
    _need_cuda(hidden_pre, W_dec, x2, sae_out2)
    lib, st = L.get_lib(), _stream()
    rows, d = x2.shape
    F = hidden_pre.shape[1]
    dev = x2.device
    dead_idx = torch.nonzero(dead_mask).flatten().to(torch.int32)
    nd = int(dead_idx.numel())
    ndp = max(32, (nd + 31) // 32 * 32)
    sc = torch.zeros(8, device=dev)
    sc[0] = mse * float(rows * d)                                    # the row kernel reads mse as loss_sum / (rows * d)
    xsum = colsum(x2)
    resid = torch.empty_like(x2)
    dummy = torch.zeros(8, device=dev)
    L.check(lib.pb_sae_dense_loss(x2.data_ptr(), sae_out2.data_ptr(), None, None, xsum.data_ptr(), None, None, resid.data_ptr(),
                                  dummy.data_ptr(), rows, 0, d, 0, st), "pb_sae_dense_loss(resid)")
    E = torch.empty(rows, ndp, device=dev)
    L.check(lib.pb_sae_ghost_gather(hidden_pre.data_ptr(), _p(dead_idx), nd, rows, F, E.data_ptr(), ndp, st), "pb_sae_ghost_gather")
    WdD = torch.empty(ndp, d, device=dev)
    L.check(lib.pb_gather_rows(W_dec.data_ptr(), _p(dead_idx), nd, ndp, d, WdD.data_ptr(), st), "pb_gather_rows")
    WdDT, _ = transpose(WdD, want_lo=False)
    G0, _ = ops.gemm(E, WdDT, None, impl=L.GEMM_SIMT)             # exact fp32: see SaeDenseStepEngine._ghost_terms
    out = torch.zeros(1, device=dev)
    L.check(lib.pb_sae_ghost_rows(resid.data_ptr(), colsum(resid).data_ptr(), G0.data_ptr(), sc.data_ptr(), out.data_ptr(), rows, d, st),
            "pb_sae_ghost_rows")
    return out[0] / float(rows * d)


class SaeDenseStepEngine(SaeStepEngine):
    """``SaeStepEngine`` plus the dense (ReLU + L1) step and the ghost-grad terms.  ``k`` is unused on the dense path."""

    def __init__(self, *a, l1_coefficient: float = 0.0, **kw):
        kw["encoder"] = "dense"               # the dense / ghost terms read hidden_pre
        super().__init__(*a, **kw)
        self.l1_coefficient = float(l1_coefficient)
        self.aux = torch.zeros(4, device=self.W_dec.device)          # [l1_sum, ghost_sum, -, -]
        self._dummy_scalars = torch.zeros(8, device=self.W_dec.device)
        self._zero_idx = torch.zeros(1, dtype=torch.int32, device=self.W_dec.device)
        self.last_n_dead = 0

    # ------------------------------------------------------------------ ghost grads (either activation)
    def _ghost_terms(self, x: torch.Tensor, resid: torch.Tensor, dead_idx: torch.Tensor) -> None:
        """Adds d(ghost loss)/d(params) for the dead features ``dead_idx`` (int32, sorted, distinct) into the gradient arrays
        and the loss value into ``aux[1]``.  Needs hidden_pre, sae_in, scalars.loss_sum of this step; ``resid = x - sae_out``."""
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        nd = int(dead_idx.numel())
        self.last_n_dead = nd
        ndp = max(32, (nd + 31) // 32 * 32)                         # zero-padded block width (TMA-legal K / N)
        dev = x.device
        E = torch.empty(rows, ndp, device=dev)
        L.check(lib.pb_sae_ghost_gather(self.hidden_pre.data_ptr(), _p(dead_idx), nd, rows, F, E.data_ptr(), ndp, st), "pb_sae_ghost_gather")
        WdD = torch.empty(ndp, d, device=dev)
        L.check(lib.pb_gather_rows(self.W_dec.data_ptr(), _p(dead_idx), nd, ndp, d, WdD.data_ptr(), st), "pb_gather_rows")
        WdDT, _ = transpose(WdD, want_lo=False)
        # [rows, d] = exp(h_dead) @ W_dec[dead] (sae.py:165) on the exact-fp32 FFMA kernel: the ghost loss divides by
        # (G - r)^2 / rcn + 1e-6 element-wise, which amplifies round-off in G by ~1e3 (fp32 torch vs fp64: 6e-4 on the
        # gradients; with the 3xTF32 product here: 4e-2).  Every later ghost product is linear in dL/dG0 and stays on tcgen05.
        G0, _ = ops.gemm(E, WdDT, None, impl=L.GEMM_SIMT)
        rsum = colsum(resid)
        L.check(lib.pb_sae_ghost_rows(resid.data_ptr(), rsum.data_ptr(), G0.data_ptr(), self.scalars.data_ptr(), self.aux[1:].data_ptr(),
                                      rows, d, st), "pb_sae_ghost_rows")
        if nd == 0:
            return                                                    # loss value only: no parameter depends on it
        dG0 = G0
        dG0_lo = ops.split_tf32(dG0)
        dE, _ = gemm32(dG0, dG0_lo, WdD, None)                       # [rows, ndp]
        L.check(lib.pb_mul_inplace(dE.data_ptr(), E.data_ptr(), dE.numel(), st), "pb_mul_inplace")    # d h_dead = dE * exp(h)
        ET, ET_lo = transpose(E)
        dG0T, dG0T_lo = transpose(dG0)
        gWd_D, _ = gemm32(ET, ET_lo, dG0T, dG0T_lo)                  # [ndp, d] = E^T @ dG0
        dhT, dhT_lo = transpose(dE)
        sinT, sinT_lo = transpose(self.sae_in)
        gWe_D, _ = gemm32(dhT, dhT_lo, sinT, sinT_lo)                # [ndp, d] = d h_dead^T @ sae_in
        gbe_D = colsum(dE)                                           # [ndp]
        WeD = torch.empty(ndp, d, device=dev)
        L.check(lib.pb_gather_rows(self.W_encT.data_ptr(), _p(dead_idx), nd, ndp, d, WeD.data_ptr(), st), "pb_gather_rows")
        gbd = gemv_rows(WeD, gbe_D)                                  # sum over tokens of d h_dead @ W_enc[:, dead]^T
        sc = lib.pb_scatter_add_rows
        L.check(sc(self.gW_dec.data_ptr(), _p(dead_idx), nd, d, gWd_D.data_ptr(), 1.0, st), "pb_scatter_add_rows")
        L.check(sc(self.gW_encT.data_ptr(), _p(dead_idx), nd, d, gWe_D.data_ptr(), 1.0, st), "pb_scatter_add_rows")
        L.check(sc(self.gb_enc.data_ptr(), _p(dead_idx), nd, 1, gbe_D.data_ptr(), 1.0, st), "pb_scatter_add_rows")
        L.check(sc(self.gb_dec.data_ptr(), self._zero_idx.data_ptr(), 1, d, gbd.data_ptr(), -1.0, st), "pb_scatter_add_rows")

    def _resid_from_out(self, x: torch.Tensor) -> torch.Tensor:
        """x - sae_out from the TopK pipeline's sae_out buffer."""
        resid = torch.empty_like(x)
        self._dummy_scalars.zero_()
        L.check(L.get_lib().pb_sae_dense_loss(x.data_ptr(), self.sae_out.data_ptr(), None, None, self.xsum.data_ptr(), None, None,
                                              resid.data_ptr(), self._dummy_scalars.data_ptr(), x.shape[0], 0, self.d, 0, _stream()),
                "pb_sae_dense_loss(resid)")
        return resid

    def _finish(self, x: torch.Tensor, lr: float, since_fired, act_freq) -> torch.Tensor:
        lib, st = L.get_lib(), _stream()
        L.check(lib.pb_sae_grad_finish(self.gW_dec.data_ptr(), self.gW_encT.data_ptr(), self.gb_enc.data_ptr(), self.gb_dec.data_ptr(),
                                       self.F, self.d, self.scalars.data_ptr(), self.max_grad_norm, x.shape[0], st), "pb_sae_grad_finish")
        s = self._desc(x, training=True, lr=float(lr), since_fired=since_fired, act_freq=act_freq, want_out=False)
        L.check(lib.pb_sae_adam(C.byref(s), st), "pb_sae_adam")
        return self.scalars

    # ------------------------------------------------------------------ TopK + ghost grads
    def train_step_topk_ghost(self, x: torch.Tensor, lr: float, since_fired: torch.Tensor, act_freq, dead_feature_window: int) -> torch.Tensor:
        """TopK step with ``cfg.use_ghost_grads`` (train_sae.py:330-354): the sparse pipeline computes the main gradients, the
        ghost blocks are added before the norm / clip."""
        _need_cuda(x)
        x = x.contiguous().float()
        lib, st = L.get_lib(), _stream()
        dead_idx = torch.nonzero(since_fired > dead_feature_window).flatten().to(torch.int32)   # host sync, as the reference's mask indexing
        self.encode_topk(x)
        self.scalars.zero_(); self.aux.zero_()
        self.step_count += 1
        s = self._desc(x, training=True, lr=float(lr), since_fired=since_fired, act_freq=act_freq, want_out=True)
        s.dist = 1                                                    # local gradients only; norm / clip after the ghost blocks
        L.check(lib.pb_sae_decode(C.byref(s), st), "pb_sae_decode")
        L.check(lib.pb_sae_backward(C.byref(s), st), "pb_sae_backward")
        with _gemm_impl(self.gemm_impl):
            self._ghost_terms(x, self._resid_from_out(x), dead_idx)
        return self._finish(x, lr, since_fired, act_freq)

    # ------------------------------------------------------------------ dense ReLU + L1 (+ ghost grads)
    def train_step_dense(self, x: torch.Tensor, lr: float, since_fired: Optional[torch.Tensor] = None, act_freq=None,
                         use_ghost_grads: bool = False, dead_feature_window: int = 5000, want_out: bool = False) -> torch.Tensor:
        """One optimizer step with ``feature_acts = relu(hidden_pre)`` and ``loss = mse + l1_coefficient * mean_b ||acts||_1``."""
        with _gemm_impl(self.gemm_impl):
            return self._train_step_dense(x, lr, since_fired, act_freq, use_ghost_grads, dead_feature_window, want_out)

    def _train_step_dense(self, x, lr, since_fired, act_freq, use_ghost_grads, dead_feature_window, want_out) -> torch.Tensor:
        _need_cuda(x)
        x = x.contiguous().float()
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        self._ensure_rows(rows)
        dead_idx = None
        if use_ghost_grads:
            dead_idx = torch.nonzero(since_fired > dead_feature_window).flatten().to(torch.int32)
        L.check(lib.pb_sae_prep(x.data_ptr(), self.b_dec.data_ptr(), self.sae_in.data_ptr(), self.sae_in_lo.data_ptr(), None,
                                self.mu.data_ptr(),
                                self.sd.data_ptr(), self.xsum.data_ptr(), rows, d, self.norm_mode, st), "pb_sae_prep")
        self.scalars.zero_(); self.aux.zero_(); self.fired.zero_()
        self.step_count += 1
        # forward
        acts = torch.empty(rows, F, device=x.device)
        gemm32(self.sae_in, self.sae_in_lo, self.W_encT, self.W_encT_lo, self.b_enc, act="relu", out0=self.hidden_pre, out1=acts)
        L.check(lib.pb_sae_dense_stats(acts.data_ptr(), rows, F, self.fired.data_ptr(), self.aux.data_ptr(), self.scalars.data_ptr(), st),
                "pb_sae_dense_stats")
        acts_lo = ops.split_tf32(acts)
        WdT, WdT_lo = transpose(self.W_dec)                          # [d, F]: K-major B operand of the decoder product
        out_n, _ = gemm32(acts, acts_lo, WdT, WdT_lo, self.b_dec)
        resid = torch.empty_like(x) if use_ghost_grads else None
        L.check(lib.pb_sae_dense_loss(x.data_ptr(), out_n.data_ptr(), self.mu.data_ptr(), self.sd.data_ptr(), self.xsum.data_ptr(),
                                      self.sae_out.data_ptr() if want_out else None, self.g.data_ptr(), _p(resid), self.scalars.data_ptr(),
                                      rows, 0, d, self.norm_mode, st), "pb_sae_dense_loss")
        # backward
        g_lo = ops.split_tf32(self.g)
        d_hid, _ = gemm32(self.g, g_lo, self.W_dec, None)             # d_acts [rows, F] = g @ W_dec^T
        d_hid_lo = torch.empty_like(d_hid)
        L.check(lib.pb_sae_dense_dhid(d_hid.data_ptr(), acts.data_ptr(), d_hid_lo.data_ptr(), self.l1_coefficient / rows, d_hid.numel(), st),
                "pb_sae_dense_dhid")
        gT, gT_lo = transpose(self.g)                                # [d, rows]
        actsT, actsT_lo = transpose(acts)                            # [F, rows]
        gemm32(actsT, actsT_lo, gT, gT_lo, out0=self.gW_dec)         # gW_dec = acts^T @ g
        del actsT, actsT_lo
        dhT, dhT_lo = transpose(d_hid)
        sinT, sinT_lo = transpose(self.sae_in)
        gemm32(dhT, dhT_lo, sinT, sinT_lo, out0=self.gW_encT)        # gW_enc^T = d_hid^T @ sae_in
        colsum(d_hid, out=self.gb_enc)
        colsum(self.g, out=self.gb_dec)
        tmp = gemv_rows(self.W_encT, self.gb_enc)                    # sum_b d_sae_in = gb_enc @ W_enc^T
        L.check(lib.pb_scatter_add_rows(self.gb_dec.data_ptr(), self._zero_idx.data_ptr(), 1, d, tmp.data_ptr(), -1.0, st),
                "pb_scatter_add_rows")
        if use_ghost_grads:
            self._ghost_terms(x, resid, dead_idx)
        self.last_acts = acts
        return self._finish(x, lr, since_fired, act_freq)

    def loss_terms(self, rows: int) -> dict:
        """Host read (synchronises): mse, l1, ghost and their sum for logging / tests."""
        sc, aux = self.scalars.tolist(), self.aux.tolist()
        out = dict(mse=sc[3], l0=sc[4], grad_norm=sc[6], clip_coef=sc[2], l1=self.l1_coefficient * aux[0] / rows,
                   ghost=aux[1] / (rows * self.d))
        out["loss"] = out["mse"] + out["l1"] + out["ghost"]
        return out
