"""fp16 candidate pass of the fused SAE encoder (csrc/sae_fused.cu): the operand conversion, the error bound with its fp32
accumulation term, the grouped top-C epilogue, and the fp16 shadows the GPU kernels keep (DESIGN.md sections 3 and 4).

The CPU tests restate the decision logic in numpy; the GPU tests check the kernels against float64."""
import math

import numpy as np
import pytest
import torch

from oracle.fused_topk_model import SEG, f2ord, ord2f

F16_MAX, F16_MIN_NORMAL = 65504.0, 2.0 ** -14
TAU_REL = 2.0 ** -13                                      # the bound's |tau_k| term (fp32 rounding of the bias add and of tau itself)


# ---------------------------------------------------------------------------- numpy model
def f16_cand(x: np.ndarray) -> np.ndarray:
    """common.cuh f16_cand: round to nearest fp16, saturate to +-65504, flush results below 2^-14 to zero (as float64)."""
    x = np.asarray(x, dtype=np.float32)
    with np.errstate(over="ignore"):
        h = x.astype(np.float16).astype(np.float64)
    h = np.clip(h, -F16_MAX, F16_MAX)
    h[np.abs(h) < F16_MIN_NORMAL] = 0.0
    return h


def error_bound(a: np.ndarray, W: np.ndarray, coef: float = 1.05) -> float:
    """E without the |tau| term: coef (||a - h(a)|| max||w|| + ||a|| max||w - h(w)|| + d 2^-22 ||a|| max||w||)."""
    a64, W64 = a.astype(np.float64), W.astype(np.float64)
    a_n, a_lo = np.linalg.norm(a64), np.linalg.norm(a64 - f16_cand(a))
    w_n, w_lo = np.linalg.norm(W64, axis=1).max(), np.linalg.norm(W64 - f16_cand(W), axis=1).max()
    return coef * (a_lo * w_n + a_n * w_lo + a.shape[-1] * 2.0 ** -22 * a_n * w_n)


def _trunc_f32(v: np.ndarray) -> np.ndarray:
    """float64 -> the fp32 value next to it towards zero."""
    f = v.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(v)
    f[over] = np.nextafter(f[over], np.float32(0))
    return f


def tensor_core_model(a: np.ndarray, W: np.ndarray) -> np.ndarray:
    """Worst-case model of the kind::f16 product: exact fp16 x fp16 products, summed one by one in fp32 with every sum truncated
    towards zero (the bound allows one such rounding per addition)."""
    ha, hW = f16_cand(a), f16_cand(W)
    acc = np.zeros(W.shape[0], dtype=np.float32)
    for i in range(W.shape[1]):
        acc = _trunc_f32(acc.astype(np.float64) + hW[:, i] * ha[i])
    return acc


def grouped_topc(seg_keys: np.ndarray, c: int) -> np.ndarray:
    """enc_cand_epilogue's selection on one segment's 128 distinct keys: groups of 4 sorted, rank r -> a list of c // r slots kept
    by insertion, the lists merged by insertion into the rank-1 list."""
    lists = [[np.iinfo(np.int64).min] * (c // r) for r in (1, 2, 3, 4)]

    def insert(s, x):
        for i in range(len(s) - 1):
            s[i], x = max(s[i], x), min(s[i], x)
        s[-1] = max(s[-1], x)

    for g in range(0, len(seg_keys), 4):
        grp = sorted(seg_keys[g:g + 4].tolist(), reverse=True)
        for r in range(4):
            insert(lists[r], grp[r])
    for s in lists[1:]:
        for x in s:
            insert(lists[0], x)
    return np.array(lists[0])


def select_row_f16(a, W, b, k, c_keep=8, m_cand=None, coef=1.05, max_cand=128, extend=16, slots=512):
    """k_cand_select on the keys of the fp16 candidate pass (tensor_core_model), as in oracle.fused_topk_model.select_row."""
    F = W.shape[0]
    m_cand = k + 8 if m_cand is None else m_cand
    exact = W.astype(np.float64) @ a.astype(np.float64) + b.astype(np.float64)
    approx = tensor_core_model(a, W) + b.astype(np.float32)
    keys = (f2ord(approx) & np.int32(~127)) | (np.arange(F, dtype=np.int32) & 127)
    keys = -np.sort(-keys.reshape(F // SEG, SEG).astype(np.int64), axis=1)[:, :c_keep]
    flat = keys.reshape(-1)
    pos = np.arange(flat.size)
    order = np.lexsort((pos, -flat))
    G = min(flat.size, slots)
    sorted_keys, sorted_pos = flat[order], pos[order]
    u_below = sorted_keys[G] if flat.size > G else None
    feat_of = (sorted_pos // c_keep) * SEG + (sorted_keys & 127)
    E0 = error_bound(a, W, coef)
    Gs = min(G, max_cand)
    m_cur = min(m_cand, Gs)
    while True:
        cand = feat_of[:m_cur]
        vals = exact[cand]
        top = sorted(range(m_cur), key=lambda j: (-vals[j], cand[j]))[:k]
        tau_k = vals[top[-1]]
        last = keys[:, c_keep - 1]
        sat = last[last >= sorted_keys[m_cur - 1]]
        u = sorted_keys[m_cur] if m_cur < G else u_below
        if sat.size:
            u = sat.max() if u is None else max(u, sat.max())
        u_val = -np.inf if u is None else float(ord2f(np.int32((int(u) & ~127) | 127)))
        proven = m_cur >= k and (u_val + E0 + abs(tau_k) * TAU_REL < tau_k)
        if proven or m_cur >= Gs:
            break
        m_cur = min(m_cur + extend, Gs)
    idx = np.array([cand[j] for j in top]) if proven else np.array(sorted(range(F), key=lambda f: (-exact[f], f))[:k])
    return dict(idx=idx, proven=bool(proven))


# ---------------------------------------------------------------------------- CPU
def test_f16_conversion_rounds_saturates_and_flushes():
    x = np.array([1.0, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 7e4, -1e30, 2.0 ** -15, -2.0 ** -14, 2.0 ** -14 * (1 - 2.0 ** -12)],
                 dtype=np.float32)
    h = f16_cand(x)
    assert h[0] == 1.0 and h[1] == 1.0 and h[2] == 1.0 + 2.0 ** -9                      # ties to even
    assert h[3] == F16_MAX and h[4] == -F16_MAX                                          # satfinite, not inf
    assert h[5] == 0.0 and h[6] == -2.0 ** -14 and h[7] == 2.0 ** -14                    # flush below the smallest normal
    rng = np.random.default_rng(0)
    v = rng.standard_normal(100_000).astype(np.float32) * 10.0
    rel = np.abs(v.astype(np.float64) - f16_cand(v)) / np.abs(v)
    assert rel[np.abs(v) >= F16_MIN_NORMAL].max() <= 2.0 ** -11                         # half an ulp of an 11-bit significand


@pytest.mark.parametrize("case", ["random", "representable", "near_overflow", "near_flush", "mixed_scale"])
def test_bound_covers_the_fp16_product(case):
    rng = np.random.default_rng(len(case))
    d, F = 256, 64
    a = rng.standard_normal(d).astype(np.float32)
    W = (rng.standard_normal((F, d)) / math.sqrt(d)).astype(np.float32)
    if case == "representable":                            # operand terms vanish: only the accumulation term is left
        a, W = f16_cand(a).astype(np.float32), f16_cand(W).astype(np.float32)
        a[: d // 2] *= 1024.0                              # products of very different sizes: the fp32 sums lose low bits
    elif case == "near_overflow":
        a *= np.float32(2.0e4)
        a[3] = np.float32(65519.0)                         # rounds to 65504
        a[7] = np.float32(-7e4)                            # saturates: large residual
    elif case == "near_flush":
        a *= np.float32(2.0 ** -13)                        # many entries flush to zero
        W *= np.float32(2.0 ** -3)
    elif case == "mixed_scale":
        W[::3] *= np.float32(100.0)
    exact = W.astype(np.float64) @ a.astype(np.float64)
    got = tensor_core_model(a, W).astype(np.float64)
    E = error_bound(a, W, coef=1.0)
    assert np.abs(got - exact).max() <= E, (case, np.abs(got - exact).max(), E)
    if case == "representable":
        assert np.abs(got - exact).max() > 0.0             # the accumulation error is real, and the new term covers it


def test_proven_rows_equal_the_exact_topk():
    rng = np.random.default_rng(5)
    d, F, k = 64, 2048, 16
    W = (rng.standard_normal((F, d)) / math.sqrt(d)).astype(np.float32)
    b = (0.01 * rng.standard_normal(F)).astype(np.float32)
    n_proven = 0
    for r in range(12):
        a = (rng.standard_normal(d) * 2.0).astype(np.float32)
        if r == 11:
            a[0] = np.float32(1e5)                          # saturated operand: the bound must fail
        res = select_row_f16(a, W, b, k)
        exact = W.astype(np.float64) @ a.astype(np.float64) + b.astype(np.float64)
        ref = sorted(range(F), key=lambda f: (-exact[f], f))[:k]
        assert res["idx"].tolist() == ref
        n_proven += res["proven"]
        if r == 11:
            assert not res["proven"]
    assert n_proven >= 9


@pytest.mark.parametrize("c", [4, 6, 8])
def test_grouped_network_keeps_the_segment_topc(c):
    rng = np.random.default_rng(c)
    for trial in range(300):
        vals = rng.standard_normal(SEG).astype(np.float32)
        if trial % 3 == 1:                                 # winners clustered in a few groups of 4
            vals[rng.integers(0, 32) * 4 + np.arange(4)] += 10.0
            vals[rng.integers(0, 32) * 4 + np.arange(4)] += 10.0
        if trial % 3 == 2:                                 # many equal values: keys differ only in the column bits
            vals = np.round(vals)
        keys = ((f2ord(vals) & np.int32(~127)) | np.arange(SEG, dtype=np.int32)).astype(np.int64)
        np.testing.assert_array_equal(grouped_topc(keys, c), np.sort(keys)[::-1][:c])


# ---------------------------------------------------------------------------- GPU
def _engine(d, F, k, seed, norm="layer_norm"):
    from vit_prisma.b200.sae_engine import SaeStepEngine
    g = torch.Generator().manual_seed(seed)
    W_encT = torch.randn(F, d, generator=g) / math.sqrt(d)
    W_dec = torch.randn(F, d, generator=g)
    W_dec /= W_dec.norm(dim=1, keepdim=True)
    b_enc = 0.01 * torch.randn(F, generator=g)
    eng = SaeStepEngine(W_encT.cuda(), W_dec.cuda(), b_enc.cuda(), torch.zeros(d).cuda(), k=k, normalize_activations=norm, encoder="fused")
    return eng, g


def _f16_cand_torch(x: torch.Tensor) -> torch.Tensor:
    h = x.half().float().clamp(-F16_MAX, F16_MAX)
    h[h.abs() < F16_MIN_NORMAL] = 0.0
    return h.half()


def _ord2f(k: torch.Tensor) -> torch.Tensor:
    return (k ^ ((k >> 31) & 0x7FFFFFFF)).view(torch.float32)


@pytest.mark.gpu
def test_candidate_pass_keys_within_bound_at_bench_size():
    """phases = 1 at 4096 x 768 x 24576: every stored key lies within E_row of the float64 pre-activation (plus its 128-ulp bucket),
    which checks the accumulation term on the tensor core itself; each segment keeps the float64 top-C up to near-ties."""
    import ctypes as C
    from vit_prisma.b200 import _lib as L
    from vit_prisma.b200.ops import _stream
    rows, d, F, k, c = 4096, 768, 24576, 32, 8
    eng, g = _engine(d, F, k, seed=11)
    x = (torch.randn(rows, d, generator=g) * 2.0 + torch.randn(d, generator=g)).cuda()
    eng.encode_topk(x)
    L.check(L.get_lib().pb_sae_encode_topk_fused(C.byref(eng._enc_desc(rows, 1)), _stream()), "phase 1")
    torch.cuda.synchronize()
    nseg = F // SEG
    sample = torch.arange(0, rows, 8, device="cuda")                      # 512 rows
    a = eng.sae_in[sample].double()
    W = eng.W_encT.double()
    exact = a @ W.t() + eng.b_enc.double()                                 # [512, F]
    a_n, a_lo = a.norm(dim=1), (a - _f16_cand_torch(eng.sae_in[sample]).double()).norm(dim=1)
    w_n, w_lo = W.norm(dim=1).max(), (W - _f16_cand_torch(eng.W_encT).double()).norm(dim=1).max()
    E = (a_lo * w_n + a_n * w_lo + d * 2.0 ** -22 * a_n * w_n)[:, None, None]   # [512, 1, 1]
    keys = eng.cand.view(rows, nseg, -1)[sample][:, :, :c]                 # [512, nseg, c]
    cols = torch.arange(nseg, device="cuda")[None, :, None] * SEG + (keys & 127).long()
    v = torch.gather(exact, 1, cols.view(len(sample), -1)).view_as(keys.double())
    lo, hi = _ord2f(keys & ~127).double(), _ord2f(keys | 127).double()
    slack = E + TAU_REL * v.abs()
    assert bool(((v >= lo - slack) & (v <= hi + slack)).all()), "a candidate key lies outside its error bound"
    # kept sets vs the float64 top-C of every segment
    seg = exact.view(len(sample), nseg, SEG)
    top = seg.topk(c, dim=2)
    cth = top.values[:, :, -1:]
    kept = torch.zeros_like(seg, dtype=torch.bool).scatter_(2, (keys & 127).long(), True)
    ref = torch.zeros_like(seg, dtype=torch.bool).scatter_(2, top.indices, True)
    diff = kept ^ ref
    near = (seg - cth).abs() <= 2 * E + 2 * (hi[:, :, :1] - lo[:, :, :1]).abs() + TAU_REL * seg.abs()
    assert bool((~diff | near).all()), "a segment dropped a feature that is clearly in its top-C"


@pytest.mark.gpu
def test_fp16_shadow_follows_w_enc():
    d, F, k, rows = 128, 4096, 16, 512
    eng, g = _engine(d, F, k, seed=3)

    def check():
        torch.cuda.synchronize()
        ref = _f16_cand_torch(eng.W_encT)
        assert torch.equal(eng.W_encT_h[:, :d].view(torch.int16), ref.view(torch.int16))

    check()
    x = (torch.randn(4 * rows, d, generator=g) * 2.0).cuda()
    for i in range(4):
        eng.train_step(x[i * rows:(i + 1) * rows], lr=1e-3)
    check()
    with torch.no_grad():                                   # an outside write, then the refresh every caller runs after one
        eng.W_encT[::7] *= 3.0
        eng.W_encT[5, :4] = torch.tensor([1e5, -7e4, 1e-9, 3e-5])
    eng.refresh_lo()
    check()
    w = eng.W_encT.double()
    torch.testing.assert_close(eng.enc_norm_max[0].double(), w.norm(dim=1).max(), rtol=1e-5, atol=0)
    torch.testing.assert_close(eng.enc_norm_max[1].double(), (w - _f16_cand_torch(eng.W_encT).double()).norm(dim=1).max(), rtol=1e-4, atol=0)


@pytest.mark.gpu
def test_row_beyond_fp16_range_takes_the_exact_path():
    d, F, k, rows = 128, 4096, 16, 64
    eng, g = _engine(d, F, k, seed=7, norm="none")
    x = torch.randn(rows, d, generator=g)
    x[5, 3] = 1e5                                           # saturates in the fp16 shadow of sae_in
    eng.encode_topk(x.cuda())
    torch.cuda.synchronize()
    assert eng.fallback_rows() >= 1
    hp = x.double() @ eng.W_encT.double().cpu().t() + eng.b_enc.double().cpu()
    ref = torch.topk(hp, k, dim=1)
    assert torch.equal(eng.idx.cpu().long(), ref.indices)
