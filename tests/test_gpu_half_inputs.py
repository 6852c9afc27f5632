"""bf16 / fp16 q, k, v on the exponent-sign path: every result equals the same call on the exactly widened fp32
tensors - masks, indices, codes and exponents bit for bit, outputs equal to the fp32 output rounded to the
16-bit type - with the same kernel launches (no conversion pass).  Also the CPU-side dtype validation."""
import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import fused_qkv_views, make_qkv, mx_specs

HALF = [torch.bfloat16, torch.float16]
HALF_IDS = ["bf16", "fp16"]


def _m():
    import mx_quantization_b200 as m
    return m


# ---------------------------------------------------------------------------------------------- CPU: validation
def test_dtype_codes_and_mixed_dtypes_cpu():
    from mx_quantization_b200 import _lib, ops
    assert ops.DTYPE_CODES == {torch.float32: _lib.MXP_DT_F32, torch.bfloat16: _lib.MXP_DT_BF16,
                               torch.float16: _lib.MXP_DT_F16}
    with pytest.raises(ValueError, match="float64"):
        ops._dtype_code(torch.float64, "q")
    a, b = torch.zeros(1, 1, 4, 32), torch.zeros(1, 1, 4, 32, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="share one dtype"):
        ops._same_dtype(("q", a), ("k", b))
    assert ops._same_dtype(("q", b), ("k", b.clone())) == torch.bfloat16


# ---------------------------------------------------------------------------------------------- GPU
def _quant_input(kind, hd, dt):
    q, k, v = make_qkv(2, 3, 70, hd, seed=5, kind=kind)
    if kind == "edges":
        q[0, 1, 2, :] = -1e-42                 # below half of bf16's smallest subnormal: -0 in bf16 and fp16
        q[1, 0, 3, :32] = 0.0
    qv, kv, vv = fused_qkv_views(q.to(dt), k.to(dt), v.to(dt))
    return qv


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("hd", [64, 72, 128])
@pytest.mark.parametrize("kind", ["randn", "lognormal", "edges"])
def test_quantizer_matches_fp32(dt, hd, kind):
    m = _m()
    xh = _quant_input(kind, hd, dt).cuda()
    assert xh.stride(-1) == 1 and not xh.is_contiguous()
    for bf in (32, 16):
        sp = mx_specs(bf)
        c16, e16, s16 = m.quantize_mxint8(xh, sp, with_signs=True)
        c32, e32, s32 = m.quantize_mxint8(xh.float(), sp, with_signs=True)
        assert torch.equal(c16, c32) and torch.equal(e16, e32) and torch.equal(s16, s32)
        oc, oe = O.quantize_mxint8(xh.float().cpu(), bfloat=bf)
        assert torch.equal(c16.cpu(), oc) and torch.equal(e16.cpu(), oe)


SEL = [  # B, H, Nq, Nk, hd, top_k, bfloat, flush, kind
    (2, 3, 197, 197, 64, 30, 32, False, "randn"),
    (1, 2, 256, 256, 72, 154, 16, False, "randn"),
    (1, 2, 256, 256, 72, 40, 32, True, "edges"),
    (2, 2, 130, 77, 64, 20, 32, False, "randn"),
    (1, 2, 300, 300, 64, 60, 32, False, "randn"),
    (1, 2, 1024, 1024, 64, 128, 32, False, "randn"),
    (1, 1, 4096, 4096, 72, 512, 16, False, "randn"),
    (1, 2, 1536, 1536, 64, 200, 32, False, "lognormal"),
    (1, 2, 2304, 2304, 128, 300, 32, False, "lognormal"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("shape", SEL, ids=lambda s: "x".join(str(x) for x in s[:6]) + f"_b{s[6]}_{s[8]}")
def test_selection_matches_fp32(dt, shape):
    m = _m()
    B, H, Nq, Nk, hd, top_k, bf, flush, kind = shape
    q, k, _ = make_qkv(B, H, Nq, hd, seed=11, kind=kind, Nk=Nk)
    qh, kh = q.to(dt).cuda(), k.to(dt).cuda()
    sp = mx_specs(bf, flush)
    r16 = m.predict_topk(qh, kh, sp, top_k, return_idx=True)
    n16 = m.last_launch_count()
    r32 = m.predict_topk(qh.float(), kh.float(), sp, top_k, return_idx=True)
    n32 = m.last_launch_count()
    assert torch.equal(r16["mask"], r32["mask"]) and torch.equal(r16["idx"], r32["idx"])
    assert n16 == n32
    if Nk <= 256 and kind == "randn" and not flush:
        qc, qe = O.quantize_mxint8(qh.float().cpu(), bfloat=bf)
        kc, ke = O.quantize_mxint8(kh.float().cpu(), bfloat=bf)
        want = O.canonical_topk(O.pred_scores_integer(qc, qe, kc, ke), top_k)
        assert torch.equal(r16["idx"].cpu().long(), torch.sort(want, dim=-1).values.long())   # idx: ascending keys


WHOLE = [  # B, H, Nq, Nk, hd, top_k, bfloat, fused mode, with key bias
    (6, 12, 197, 197, 64, 30, 32, 1, False),       # fused launch (>= 64 heads), cost-follows-k epilogue
    (2, 2, 256, 256, 72, 154, 16, 2, False),       # fused launch forced, dense epilogue
    (2, 3, 197, 197, 64, 30, 32, 0, False),        # three kernels, dense epilogue
    (1, 3, 197, 197, 64, 30, 32, 1, False),        # cost-follows-k attention kernel, few heads
    (2, 4, 256, 120, 72, 30, 16, 1, True),         # PixArt cross-attention with the text mask
    (1, 2, 1024, 1024, 64, 128, 32, 1, False),     # long sequence
    (1, 2, 4096, 4096, 72, 512, 16, 1, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("shape", WHOLE, ids=lambda s: "x".join(str(x) for x in s[:6]) + f"_b{s[6]}_f{s[7]}" +
                         ("_bias" if s[8] else ""))
def test_pruned_attention_matches_fp32(dt, shape):
    m = _m()
    B, H, Nq, Nk, hd, top_k, bf, mode, biased = shape
    q, k, v = make_qkv(B, H, Nq, hd, seed=3, Nk=Nk)
    qh, kh, vh = (x.to(dt).cuda() for x in (q, k, v))
    q32, k32, v32 = qh.float(), kh.float(), vh.float()
    sp = mx_specs(bf)
    kb = None
    if biased:
        kb = torch.zeros(B, 1, 1, Nk)
        kb[:, :, :, Nk - 40:] = -10000.0
        kb = kb.cuda()
    m.set_fused_path(mode)
    try:
        out32, mask32 = m.pruned_attention(q32, k32, v32, sp, top_k, return_mask=True, key_bias=kb)
        n32 = m.last_launch_count()
        out16, mask16 = m.pruned_attention(qh, kh, vh, sp, top_k, return_mask=True, key_bias=kb)
        n16 = m.last_launch_count()
        assert out16.dtype == dt
        assert torch.equal(mask16, mask32)
        assert n16 == n32
        assert torch.equal(out16, out32.to(dt))
        # an fp32 out= buffer gets the fp32 result
        o32 = torch.empty(B, H, Nq, hd, device="cuda")
        m.pruned_attention(qh, kh, vh, sp, top_k, out=o32, key_bias=kb)
        assert torch.equal(o32, out32)
        # a permuted (B, Nq, H, hd) 16-bit output view
        buf = torch.full((B, Nq, H, hd), float("nan"), dtype=dt, device="cuda")
        m.pruned_attention(qh, kh, vh, sp, top_k, out=buf.permute(0, 2, 1, 3), key_bias=kb)
        assert torch.equal(buf.permute(0, 2, 1, 3), out32.to(dt))
    finally:
        m.set_fused_path(1)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_fused_qkv_views_and_sparse_attention(dt):
    m = _m()
    q, k, v = make_qkv(2, 4, 197, 64, seed=8)
    qv, kv, vv = fused_qkv_views(q.to(dt).cuda(), k.to(dt).cuda(), v.to(dt).cuda())
    sp = mx_specs()
    out16 = m.pruned_attention(qv, kv, vv, sp, 30)
    out32 = m.pruned_attention(qv.float(), kv.float(), vv.float(), sp, 30)
    assert torch.equal(out16, out32.to(dt))
    r = m.predict_topk(qv.float(), kv.float(), sp, 30, return_codes=True)
    args = (r["q_codes"], r["q_exps"], r["k_codes"], r["k_exps"])
    s16 = m.sparse_attention(*args, vv, r["mask"], sp)
    s32 = m.sparse_attention(*args, vv.float(), r["mask"], sp)
    assert s16.dtype == dt and torch.equal(s16, s32.to(dt))
    f32 = m.sparse_attention(*args, vv, r["mask"], sp, out=torch.empty_like(s32))
    assert torch.equal(f32, s32)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_rejections_leave_no_cuda_error(dt):
    m = _m()
    q, k, v = (x.to(dt).cuda() for x in make_qkv(1, 2, 64, 64, seed=1))
    sp = mx_specs()
    with pytest.raises(ValueError):
        m.pruned_attention(q, k.float(), v, sp, 8)                     # mixed dtypes
    with pytest.raises(ValueError):
        m.pruned_attention(q, k, v, sp, 8, pred_mode="partial_Q")
    with pytest.raises(ValueError):
        m.pruned_attention(q, k, v, sp, 8, pred_mode="ELSA", orthogonal_matrix=torch.eye(64))
    q36, k36, v36 = (x.to(dt).cuda() for x in make_qkv(1, 2, 64, 36, seed=1))
    with pytest.raises(ValueError):
        m.pruned_attention(q36, k36, v36, sp, 8)                       # head_dim outside the tensor-core domain
    big = torch.zeros(1, 2, 64, 68, dtype=dt, device="cuda")
    with pytest.raises(ValueError):
        m.pruned_attention(big[..., :64], big[..., :64], big[..., :64], sp, 8)   # row stride 68: not a multiple of 8
    d = torch.zeros(1, 2, 64, 64, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        m.pruned_attention(d, d, d, sp, 8)
    with pytest.raises(ValueError):
        m.predict_topk(q, k, sp, 8, pred_mode="partial_K")
    torch.cuda.synchronize()
    # a valid call still runs and no error is pending
    out = m.pruned_attention(q, k, v, sp, 8)
    torch.cuda.synchronize()
    assert out.dtype == dt and torch.isfinite(out.float()).all()
