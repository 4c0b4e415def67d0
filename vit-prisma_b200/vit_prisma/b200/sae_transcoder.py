"""Transcoder training step and forward on the C-ABI kernels (reference sae/transcoder.py:6-116, trained by train_sae.py:278-411
with ``layer_acts[:, 0]`` as the input activation and ``layer_acts[:, 1]`` as the target).

    sae_in      = norm_in(x) - b_dec                                          (transcoder.py:33-39)
    hidden_pre  = sae_in @ W_enc + b_enc ; acts = relu(.) | TopK(.)           (:41-51)
    out_n       = acts @ W_dec + b_dec_out  [+ x @ W_skip^T]                   (:58-79: the skip term uses the RAW x)
    sae_out     = norm_out(out_n)   with the INPUT's row statistics           (:81)
    loss        = mean((sae_out - y)^2 / ||y - mean_batch(y)||) + l1           (:83, 93-103; l1 only for dense activations)

The dense products run on ``pb_gemm`` (3xTF32 tcgen05) exactly as in ``SaeDenseStepEngine``; this module adds the target-vs-input
split of the loss, the skip matrix (one more forward product through the residual epilogue, one more gradient product) and the
second decoder bias.  ``pb_sae_adam`` updates W_dec (clip, decoder-parallel-gradient removal, Adam, row renorm), W_enc, b_enc and
b_dec; ``pb_adam_vec`` updates W_skip and b_dec_out with the same clip coefficient.  Requires d_out == d_in (the reference default).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from . import ops
from .sae_dense import SaeDenseStepEngine, _gemm_impl, _p, colsum, gemm32, gemv_rows, transpose
from .sae_engine import _need_cuda, _stream, topk_dense

i32, f32, vp = C.c_int32, C.c_float, C.c_void_p
L.register_signatures({
    "pb_sumsq": (i32, [vp, C.c_int64, vp, vp]),
    "pb_sae_clip_finish": (i32, [vp, f32, i32, i32, vp]),
    "pb_adam_vec": (i32, [vp, vp, vp, vp, i32, vp, f32, f32, f32, f32, i32, vp]),
})


class SaeTranscoderStepEngine(SaeDenseStepEngine):
    """Parameters: W_encT [F, d] (feature-major view of W_enc), W_dec [F, d_out = d], b_enc [F], b_dec [d], b_dec_out [d],
    W_skip [d, d] or None."""

    def __init__(self, W_encT, W_dec, b_enc, b_dec, b_dec_out: torch.Tensor, W_skip: Optional[torch.Tensor], k: int, activation: str,
                 l1_coefficient: float = 0.0, **kw):
        super().__init__(W_encT, W_dec, b_enc, b_dec, k=max(int(k), 1), l1_coefficient=l1_coefficient, **kw)
        if W_dec.shape[1] != self.d:
            raise L.PrismaB200Error("B200 transcoder step: d_out must equal d_in")
        if activation not in ("relu", "topk"):
            raise NotImplementedError(f"B200 transcoder step: activation {activation!r} is not built (relu and topk are)")
        _need_cuda(b_dec_out, W_skip)
        self.activation, self.b_dec_out, self.W_skip = activation, b_dec_out, W_skip
        dev, d = W_dec.device, self.d
        z = lambda *s: torch.zeros(*s, device=dev)  # noqa: E731
        self.gb_dec_out, self.m_bo, self.v_bo = z(d), z(d), z(d)
        if W_skip is not None:
            self.gW_skip, self.m_sk, self.v_sk = z(d, d), z(d, d), z(d, d)
        self.ysum = z(d)

    # ------------------------------------------------------------------ forward pieces
    def _forward(self, x: torch.Tensor, y: Optional[torch.Tensor], want_out: bool, training: bool):
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        self._ensure_rows(rows)
        L.check(lib.pb_sae_prep(x.data_ptr(), self.b_dec.data_ptr(), self.sae_in.data_ptr(), self.sae_in_lo.data_ptr(), None,
                                self.mu.data_ptr(),
                                self.sd.data_ptr(), self.xsum.data_ptr(), rows, d, self.norm_mode, st), "pb_sae_prep")
        self.scalars.zero_(); self.aux.zero_(); self.fired.zero_()
        if self.activation == "relu":
            acts = torch.empty(rows, F, device=x.device)
            gemm32(self.sae_in, self.sae_in_lo, self.W_encT, self.W_encT_lo, self.b_enc, act="relu", out0=self.hidden_pre, out1=acts)
        else:
            gemm32(self.sae_in, self.sae_in_lo, self.W_encT, self.W_encT_lo, self.b_enc, out0=self.hidden_pre)
            acts = topk_dense(self.hidden_pre, self.k)                       # zeros.scatter_(topk idx, relu(topk values))
        L.check(lib.pb_sae_dense_stats(acts.data_ptr(), rows, F, self.fired.data_ptr(), self.aux.data_ptr(), self.scalars.data_ptr(), st),
                "pb_sae_dense_stats")
        WdT, WdT_lo = transpose(self.W_dec)
        out_n, _ = gemm32(acts, None, WdT, WdT_lo, self.b_dec_out)
        if self.W_skip is not None:                                           # + x @ W_skip^T: W_skip [d_out, d_in] is already K-major
            x_lo = ops.split_tf32(x)
            if self.gemm_impl == L.GEMM_SIMT:
                _, out_n = ops.gemm(x, self.W_skip, None, residual=out_n, want_pre=False, impl=L.GEMM_SIMT)
            else:
                _, out_n = ops.gemm(x, self.W_skip, None, residual=out_n, want_pre=False, a_lo=x_lo, w_lo=ops.split_tf32(self.W_skip))
        if y is not None:                                                      # loss against the TARGET activation, centred on its batch mean
            colsum(y, out=self.ysum)
            L.check(lib.pb_sae_dense_loss(y.data_ptr(), out_n.data_ptr(), self.mu.data_ptr(), self.sd.data_ptr(), self.ysum.data_ptr(),
                                          self.sae_out.data_ptr() if want_out else None, self.g.data_ptr() if training else None, None,
                                          self.scalars.data_ptr(), rows, 0, d, self.norm_mode, st), "pb_sae_dense_loss")
        elif want_out:                                                         # inference without a target: sae_out only
            dummy = torch.zeros(8, device=x.device)
            L.check(lib.pb_sae_dense_loss(x.data_ptr(), out_n.data_ptr(), self.mu.data_ptr(), self.sd.data_ptr(), self.xsum.data_ptr(),
                                          self.sae_out.data_ptr(), None, None, dummy.data_ptr(), rows, 0, d, self.norm_mode, st),
                    "pb_sae_dense_loss")
        self.last_acts = acts
        return acts

    @torch.no_grad()
    def forward_losses(self, x: torch.Tensor, y: Optional[torch.Tensor], want_out: bool = True) -> torch.Tensor:
        """Inference / logging: fills sae_out and (with a target) scalars.mse / l0 and aux[0] = sum |acts|; returns feature_acts."""
        _need_cuda(x, y)
        x = x.contiguous().float()
        y = None if y is None else y.contiguous().float()
        with _gemm_impl(self.gemm_impl):
            acts = self._forward(x, y, want_out, training=False)
        L.check(L.get_lib().pb_sae_clip_finish(self.scalars.data_ptr(), 0.0, x.shape[0], self.d, _stream()), "pb_sae_clip_finish")
        return acts

    # ------------------------------------------------------------------ one optimizer step
    @torch.no_grad()
    def train_step_transcoder(self, x: torch.Tensor, y: torch.Tensor, lr: float, since_fired: Optional[torch.Tensor] = None,
                              act_freq: Optional[torch.Tensor] = None, want_out: bool = False) -> torch.Tensor:
        _need_cuda(x, y)
        x, y = x.contiguous().float(), y.contiguous().float()
        with _gemm_impl(self.gemm_impl):
            return self._train_step_tc(x, y, float(lr), since_fired, act_freq, want_out)

    def _train_step_tc(self, x, y, lr, since_fired, act_freq, want_out) -> torch.Tensor:
        lib, st = L.get_lib(), _stream()
        rows, d, F = x.shape[0], self.d, self.F
        self.step_count += 1
        acts = self._forward(x, y, want_out, training=True)
        l1_grad = (self.l1_coefficient / rows) if self.activation != "topk" else 0.0       # TopK: no sparsity term (transcoder.py:96-100)
        d_hid, _ = gemm32(self.g, None, self.W_dec, None)                    # d_acts = g @ W_dec^T
        d_hid_lo = torch.empty_like(d_hid)
        L.check(lib.pb_sae_dense_dhid(d_hid.data_ptr(), acts.data_ptr(), d_hid_lo.data_ptr(), l1_grad, d_hid.numel(), st), "pb_sae_dense_dhid")
        gT, gT_lo = transpose(self.g)                                        # [d, rows]
        actsT, actsT_lo = transpose(acts)
        gemm32(actsT, actsT_lo, gT, gT_lo, out0=self.gW_dec)                 # gW_dec = acts^T @ g
        del actsT, actsT_lo
        dhT, dhT_lo = transpose(d_hid)
        sinT, sinT_lo = transpose(self.sae_in)
        gemm32(dhT, dhT_lo, sinT, sinT_lo, out0=self.gW_encT)                # gW_enc^T = d_hid^T @ sae_in
        colsum(d_hid, out=self.gb_enc)
        colsum(self.g, out=self.gb_dec_out)                                   # b_dec_out enters the output only
        tmp = gemv_rows(self.W_encT, self.gb_enc)                             # b_dec enters through sae_in = norm(x) - b_dec only
        self.gb_dec.zero_()
        L.check(lib.pb_scatter_add_rows(self.gb_dec.data_ptr(), self._zero_idx.data_ptr(), 1, d, tmp.data_ptr(), -1.0, st), "pb_scatter_add_rows")
        grads = [self.gW_dec, self.gW_encT, self.gb_enc, self.gb_dec, self.gb_dec_out]
        if self.W_skip is not None:
            xT, xT_lo = transpose(x)                                         # [d, rows]
            gemm32(gT, gT_lo, xT, xT_lo, out0=self.gW_skip)                  # gW_skip = g^T @ x   ([d_out, d_in], out += x @ W_skip^T)
            grads.append(self.gW_skip)
        self.scalars[1:2].zero_()
        acc = self.scalars[1:].data_ptr()
        for t in grads:
            L.check(lib.pb_sumsq(t.data_ptr(), t.numel(), acc, st), "pb_sumsq")
        L.check(lib.pb_sae_clip_finish(self.scalars.data_ptr(), self.max_grad_norm, rows, d, st), "pb_sae_clip_finish")
        s = self._desc(x, training=True, lr=lr, since_fired=since_fired, act_freq=act_freq, want_out=False)
        L.check(lib.pb_sae_adam(C.byref(s), st), "pb_sae_adam")
        extra = [(self.b_dec_out, self.gb_dec_out, self.m_bo, self.v_bo)]
        if self.W_skip is not None:
            extra.append((self.W_skip, self.gW_skip, self.m_sk, self.v_sk))
        for p, g, m, v in extra:
            L.check(lib.pb_adam_vec(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), self.scalars.data_ptr(), lr, self.betas[0],
                                    self.betas[1], self.adam_eps, self.step_count, st), "pb_adam_vec")
        return self.scalars

    def loss_terms(self, rows: int) -> dict:
        sc, aux = self.scalars.tolist(), self.aux.tolist()
        l1 = self.l1_coefficient * aux[0] / rows if self.activation != "topk" else 0.0
        return dict(mse=sc[3], l0=sc[4], grad_norm=sc[6], clip_coef=sc[2], l1=l1, loss=sc[3] + l1)
