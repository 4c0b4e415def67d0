"""Gated SAE training step (``GatedSparseAutoencoder``, reference sae/sae.py:648-792 under ``VisionSAETrainer.train_step``).

    pi = sae_in @ W_enc + b_gate                      gate path              (:701)
    mag_pre = sae_in @ (W_enc * exp(r_mag)) + b_mag   magnitude path         (:705)   = (pi - b_gate) * exp(r_mag) + b_mag
    acts = [pi > 0] * relu(mag_pre)                                          (:707-709)
    loss = mse(decode(acts)) + l1 * mean_b sum_f relu(pi) ||W_dec[f]|| + mean_b ||relu(pi) @ W_dec + b_dec - sae_in||^2   (:726-744)

Because the magnitude path shares the encoder matrix, ONE encoder GEMM feeds both paths and one GEMM carries both paths'
gradient back to it (D = d_pi + d_mag * exp(r_mag)); the reference executes three encoder products forward.  The dense
products (encoder, two decoder products, their four transposed products) run on ``pb_gemm`` (3xTF32); the element-wise
pieces are ``pb_gated_*`` in csrc/sae_dense.cu; ``pb_sae_adam`` (W_dec projection + renorm, W_enc, b_gate in the b_enc slot,
b_dec, dead-feature counters) and ``pb_adam_vec`` (r_mag, b_mag) finish the step.  ``b_enc`` exists in the reference module but
never enters its graph (gradient ``None``, untouched by Adam): it is not an engine parameter.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from . import ops
from .sae_dense import _gemm_impl, _p, colsum, gemm32, gemv_rows, transpose
from .sae_engine import SaeStepEngine, _need_cuda, _stream

i32, i64, f32, vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p

L.register_signatures({
    "pb_gated_fwd": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]),
    "pb_gated_aux": (i32, [vp, vp, vp, vp, i32, i32, vp]),
    "pb_gated_bwd": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, vp, vp, i32, i32, vp]),
    "pb_row_norms": (i32, [vp, vp, i32, i32, vp]),
    "pb_gated_l1_rows": (i32, [vp, vp, vp, vp, f32, vp, i32, i32, vp]),
    "pb_sumsq": (i32, [vp, i64, vp, vp]),
    "pb_sae_clip_finish": (i32, [vp, f32, i32, i32, vp]),
    "pb_adam_vec": (i32, [vp, vp, vp, vp, i32, vp, f32, f32, f32, f32, i32, vp]),
})


class SaeGatedStepEngine(SaeStepEngine):
    """Parameters: W_encT [F,d] (feature-major view of W_enc), W_dec [F,d], b_gate, r_mag, b_mag [F], b_dec [d]."""

    def __init__(self, W_encT: torch.Tensor, W_dec: torch.Tensor, b_gate: torch.Tensor, r_mag: torch.Tensor, b_mag: torch.Tensor,
                 b_dec: torch.Tensor, l1_coefficient: float, **kw):
        kw["encoder"] = "dense"
        super().__init__(W_encT, W_dec, b_gate, b_dec, k=1, **kw)     # b_gate rides in the b_enc slot of pb_sae_adam
        _need_cuda(r_mag, b_mag)
        self.b_gate, self.r_mag, self.b_mag = b_gate, r_mag, b_mag
        self.l1_coefficient = float(l1_coefficient)
        dev = W_dec.device
        z = lambda n: torch.zeros(n, device=dev)  # noqa: E731
        self.m_r, self.v_r, self.m_bm, self.v_bm = z(self.F), z(self.F), z(self.F), z(self.F)
        self.gr_mag, self.gb_mag, self.dsum, self.piact_colsum, self.wnorm = z(self.F), z(self.F), z(self.F), z(self.F), z(self.F)
        self.aux = torch.zeros(4, device=dev)                          # [sum_f colsum(pi_act) ||W_dec[f]||, sum (via - sae_in)^2, -, -]
        self._zero_idx = torch.zeros(1, dtype=torch.int32, device=dev)

    # ------------------------------------------------------------------ forward pieces (shared by training and inference)
    def _forward(self, x: torch.Tensor, want_out: bool, training: bool):
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        self._ensure_rows(rows)
        L.check(lib.pb_sae_prep(x.data_ptr(), self.b_dec.data_ptr(), self.sae_in.data_ptr(), self.sae_in_lo.data_ptr(), None,
                                self.mu.data_ptr(),
                                self.sd.data_ptr(), self.xsum.data_ptr(), rows, d, self.norm_mode, st), "pb_sae_prep")
        self.scalars.zero_(); self.aux.zero_(); self.fired.zero_(); self.piact_colsum.zero_()
        gemm32(self.sae_in, self.sae_in_lo, self.W_encT, self.W_encT_lo, self.b_gate, out0=self.hidden_pre)        # pi
        dev = x.device
        acts, pi_act = torch.empty(rows, F, device=dev), torch.empty(rows, F, device=dev)
        acts_lo, pi_act_lo = torch.empty(rows, F, device=dev), torch.empty(rows, F, device=dev)
        L.check(lib.pb_gated_fwd(self.hidden_pre.data_ptr(), self.b_gate.data_ptr(), self.r_mag.data_ptr(), self.b_mag.data_ptr(),
                                 acts.data_ptr(), acts_lo.data_ptr(), pi_act.data_ptr(), pi_act_lo.data_ptr(), self.fired.data_ptr(),
                                 self.piact_colsum.data_ptr(), self.scalars.data_ptr(), rows, F, st), "pb_gated_fwd")
        WdT, WdT_lo = transpose(self.W_dec)                           # [d, F]: K-major B operand of both decoder products
        out_n, _ = gemm32(acts, acts_lo, WdT, WdT_lo, self.b_dec)
        via, _ = gemm32(pi_act, pi_act_lo, WdT, WdT_lo, self.b_dec)   # via-gate reconstruction (:786-787)
        L.check(lib.pb_sae_dense_loss(x.data_ptr(), out_n.data_ptr(), self.mu.data_ptr(), self.sd.data_ptr(), self.xsum.data_ptr(),
                                      self.sae_out.data_ptr() if want_out else None, self.g.data_ptr() if training else None, None,
                                      self.scalars.data_ptr(), rows, 0, d, self.norm_mode, st), "pb_sae_dense_loss")
        ga = torch.empty(rows, d, device=dev)
        L.check(lib.pb_gated_aux(via.data_ptr(), self.sae_in.data_ptr(), ga.data_ptr(), self.aux[1:].data_ptr(), rows, d, st), "pb_gated_aux")
        L.check(lib.pb_row_norms(self.W_dec.data_ptr(), self.wnorm.data_ptr(), F, d, st), "pb_row_norms")
        self.last_acts = acts
        return acts, acts_lo, pi_act, pi_act_lo, ga

    @torch.no_grad()
    def forward_losses(self, x: torch.Tensor, want_out: bool = True) -> torch.Tensor:
        """Inference / logging: fills sae_out, scalars (loss_sum, pos_count) and aux; returns feature_acts [rows, F]."""
        _need_cuda(x)
        x = x.contiguous().float()
        lib, st = L.get_lib(), _stream()
        with _gemm_impl(self.gemm_impl):
            acts, _, _, _, _ = self._forward(x, want_out, training=False)
        # l1 value without touching any gradient buffer: sum_f colsum(pi_act)[f] * ||W_dec[f]||
        scratch = torch.zeros(self.F, self.d, device=x.device) if not hasattr(self, "_l1_scratch") else self._l1_scratch
        self._l1_scratch = scratch
        L.check(lib.pb_gated_l1_rows(scratch.data_ptr(), self.W_dec.data_ptr(), self.piact_colsum.data_ptr(), self.wnorm.data_ptr(), 0.0,
                                     self.aux.data_ptr(), self.F, self.d, st), "pb_gated_l1_rows")
        L.check(lib.pb_sae_clip_finish(self.scalars.data_ptr(), 0.0, x.shape[0], self.d, st), "pb_sae_clip_finish")
        return acts

    # ------------------------------------------------------------------ one optimizer step
    def train_step_gated(self, x: torch.Tensor, lr: float, since_fired: Optional[torch.Tensor] = None, act_freq=None,
                         want_out: bool = False) -> torch.Tensor:
        _need_cuda(x)
        x = x.contiguous().float()
        with _gemm_impl(self.gemm_impl):
            return self._train_step(x, float(lr), since_fired, act_freq, want_out)

    def _train_step(self, x, lr, since_fired, act_freq, want_out) -> torch.Tensor:
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        self.step_count += 1
        acts, acts_lo, pi_act, pi_act_lo, ga = self._forward(x, want_out, training=True)
        l1_grad = self.l1_coefficient / rows
        Wd_lo = ops.split_tf32(self.W_dec)
        D, _ = gemm32(self.g, None, self.W_dec, Wd_lo)               # d_acts = g @ W_dec^T, becomes D in place
        d_pia, _ = gemm32(ga, None, self.W_dec, Wd_lo)
        D_lo = torch.empty_like(D)
        L.check(lib.pb_gated_bwd(D.data_ptr(), D_lo.data_ptr(), d_pia.data_ptr(), self.hidden_pre.data_ptr(), self.b_gate.data_ptr(),
                                 self.r_mag.data_ptr(), self.b_mag.data_ptr(), self.wnorm.data_ptr(), l1_grad, self.gb_enc.data_ptr(),
                                 self.gb_mag.data_ptr(), self.gr_mag.data_ptr(), self.dsum.data_ptr(), rows, F, st), "pb_gated_bwd")
        del d_pia
        # gW_dec = acts^T @ g + pi_act^T @ ga (+ L1 rows); the second product accumulates through the residual epilogue
        gT, gT_lo = transpose(self.g)
        gaT, gaT_lo = transpose(ga)
        actsT, actsT_lo = transpose(acts)
        first, _ = gemm32(actsT, actsT_lo, gT, gT_lo)
        del actsT, actsT_lo
        piT, piT_lo = transpose(pi_act)
        if self.gemm_impl == L.GEMM_SIMT:
            ops.gemm(piT, gaT, None, residual=first, out1=self.gW_dec, want_pre=False, impl=L.GEMM_SIMT)
        else:
            ops.gemm(piT, gaT, None, residual=first, out1=self.gW_dec, want_pre=False, a_lo=piT_lo, w_lo=gaT_lo)
        del piT, piT_lo, first
        L.check(lib.pb_gated_l1_rows(self.gW_dec.data_ptr(), self.W_dec.data_ptr(), self.piact_colsum.data_ptr(), self.wnorm.data_ptr(),
                                     l1_grad, self.aux.data_ptr(), F, d, st), "pb_gated_l1_rows")
        # gW_enc^T = D^T @ sae_in
        DT, DT_lo = transpose(D)
        sinT, sinT_lo = transpose(self.sae_in)
        gemm32(DT, DT_lo, sinT, sinT_lo, out0=self.gW_encT)
        # gb_dec = colsum(g) + 2 colsum(ga) - colsum(D) @ W_enc^T      (decoder bias twice, sae_in = xn - b_dec in the aux target and the encoder)
        colsum(self.g, out=self.gb_dec)
        sc = lib.pb_scatter_add_rows
        L.check(sc(self.gb_dec.data_ptr(), self._zero_idx.data_ptr(), 1, d, colsum(ga).data_ptr(), 2.0, st), "pb_scatter_add_rows")
        L.check(sc(self.gb_dec.data_ptr(), self._zero_idx.data_ptr(), 1, d, gemv_rows(self.W_encT, self.dsum).data_ptr(), -1.0, st),
                "pb_scatter_add_rows")
        # global norm over the six trained tensors -> clip coefficient
        self.scalars[1:2].zero_()
        acc = self.scalars[1:].data_ptr()
        for t in (self.gW_dec, self.gW_encT, self.gb_enc, self.gb_dec, self.gr_mag, self.gb_mag):
            L.check(lib.pb_sumsq(t.data_ptr(), t.numel(), acc, st), "pb_sumsq")
        L.check(lib.pb_sae_clip_finish(self.scalars.data_ptr(), self.max_grad_norm, rows, d, st), "pb_sae_clip_finish")
        s = self._desc(x, training=True, lr=lr, since_fired=since_fired, act_freq=act_freq, want_out=False)
        L.check(lib.pb_sae_adam(C.byref(s), st), "pb_sae_adam")
        for p, g, m, v in ((self.r_mag, self.gr_mag, self.m_r, self.v_r), (self.b_mag, self.gb_mag, self.m_bm, self.v_bm)):
            L.check(lib.pb_adam_vec(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), F, self.scalars.data_ptr(), lr, self.betas[0],
                                    self.betas[1], self.adam_eps, self.step_count, st), "pb_adam_vec")
        return self.scalars

    def loss_terms(self, rows: int) -> dict:
        """Host read (synchronises): mse, l1, aux reconstruction loss and their sum."""
        sc, aux = self.scalars.tolist(), self.aux.tolist()
        out = dict(mse=sc[3], l0=sc[4], grad_norm=sc[6], clip_coef=sc[2], l1=self.l1_coefficient * aux[0] / rows, aux=aux[1] / rows)
        out["loss"] = out["mse"] + out["l1"] + out["aux"]
        return out
