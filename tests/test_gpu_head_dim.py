"""Every entry point at every head_dim the C ABI accepts, against the CPU oracle, with guard-banded outputs.

What changes from one head_dim to the next is the tail ``hd % 32``: the partial last MX block of a row, and with it
store widths, chunk counts and padding.  The sweeps cover

  H4  every multiple of 4 in [4, 128]    (quantizer, CUDA-core predictor, CUDA-core attention)
  H8  every multiple of 8 in [32, 128]   (tensor-core predictor and attention, 16-bit inputs)

Each output lives inside a larger buffer of canary bytes; after the call every byte outside the output must still hold
the canary, so a store that strays past a row or past the end of the output fails the test even where it changes no
value the test reads back.
"""
import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import (Guarded, assert_out_close, canonical_idx_from_mask, make_qkv, mx_specs, select_guarded,
                           unpack_mask)

pytestmark = pytest.mark.gpu

H4 = list(range(4, 129, 4))
H8 = list(range(32, 129, 8))
OUT_TOL = 1e-3
# the rankings of tests/test_gpu_parity.py::MODES
MODES = ["partial_Q", "partial_K", "MXINT4", "two_step_leading_ones", "true_ex", "exact"]


@pytest.fixture(scope="module")
def mxq():
    import mx_quantization_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


def _out_view(shape, dtype):
    """A guarded ``out=`` view with a padded row stride: hd + 4 floats for fp32, hd + 8 elements for 16-bit."""
    return Guarded(shape, dtype, row_pad=4 if dtype == torch.float32 else 8)


def _paths(mxq, predict="tcgen05", attention="tcgen05", fused=1):
    """Set the process-wide path switches; returns the function that restores the defaults."""
    mxq.set_predict_path(predict)
    mxq.set_attention_path(attention)
    mxq.set_fused_path(fused)

    def restore():
        mxq.set_predict_path("tcgen05")
        mxq.set_attention_path("tcgen05")
        mxq.set_fused_path(True)
    return restore


def _words(t):
    return t.cpu().to(torch.int64) & 0xFFFFFFFF


# ---- 1. quantizer ----------------------------------------------------------------------------------------------------
def _quantize_guarded(x, bfloat, flush):
    """mxp_quantize_mxint8_dt with codes, exps and sign words written into guarded buffers."""
    from mx_quantization_b200 import _lib, ops
    lib = _lib.load()
    B, H, N, hd = x.shape
    nb = (hd + 31) // 32
    codes, exps = Guarded((B, H, N, hd), torch.int8), Guarded((B, H, N, nb), torch.int8)
    signs = Guarded((B, H, N, nb), torch.int32)
    p = ops._ptr
    rc = lib.mxp_quantize_mxint8_dt(p(x), ops.DTYPE_CODES[x.dtype], *x.stride()[:3], B, H, N, hd, bfloat, int(flush),
                                    p(codes.t), p(exps.t), p(signs.t), ops._stream())
    _lib.check(rc, "mxp_quantize_mxint8_dt")
    for name, g in (("codes", codes), ("exps", exps), ("signs", signs)):
        g.assert_intact(name)
    return codes.t.cpu(), exps.t.cpu(), _words(signs.t)


def _exp_sign_guarded(x, bfloat, flush):
    from mx_quantization_b200 import _lib, ops
    B, H, N, hd = x.shape
    out = Guarded((B, H, N, hd), torch.float32)
    p = ops._ptr
    rc = _lib.load().mxp_exp_sign_approx(p(x), *x.stride()[:3], B, H, N, hd, bfloat, int(flush), p(out.t), ops._stream())
    _lib.check(rc, "mxp_exp_sign_approx")
    out.assert_intact("approx")
    return out.t.cpu()


def _check_quantizer(codes, exps, signs, x, bfloat, flush):
    oc, oe = O.quantize_mxint8(x, 32, bfloat, flush)
    bad = (codes != oc).reshape(-1, x.shape[-1])
    assert not bool(bad.any()), (f"codes differ in {int(bad.any(-1).sum())} of {bad.shape[0]} rows; "
                                 f"first bad positions {bad.nonzero()[:4, 1].tolist()}")
    assert torch.equal(exps, oe)
    assert torch.equal(signs, O.sign_words(oc))
    return oc, oe


@pytest.mark.parametrize("hd", H4)
def test_quantizer_fp32(mxq, hd):
    """2 x 3 heads of 70 rows: rows cross warp and CTA boundaries of both quantizer kernels."""
    q, k, _ = make_qkv(2, 3, 70, hd, seed=hd, kind="edges")
    for bfloat in (32, 16):
        for x in (q, k):
            xc = x.cuda()
            oc, oe = _check_quantizer(*_quantize_guarded(xc, bfloat, False), x, bfloat, False)
            assert torch.equal(_exp_sign_guarded(xc, bfloat, False), O.exponent_based_sign(oc, oe))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("hd", list(range(8, 129, 8)))
def test_quantizer_16bit(mxq, hd, dtype):
    """16-bit x: the oracle on the widened tensor, and the fp32 call on it, bit for bit."""
    q, k, _ = make_qkv(2, 3, 70, hd, seed=100 + hd, kind="edges")
    for bfloat in (32, 16):
        for x in (q, k):
            xw = x.to(dtype).float()
            got = _quantize_guarded(xw.to(dtype).cuda(), bfloat, False)
            _check_quantizer(*got, xw, bfloat, False)
            c32, e32, s32 = mxq.quantize_mxint8(xw.cuda(), mx_specs(bfloat), with_signs=True)
            assert torch.equal(got[0], c32.cpu()) and torch.equal(got[1], e32.cpu())
            assert torch.equal(got[2], _words(s32))


# ---- 2. dense predictor scores ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("hd", H4)
def test_predict_scores(mxq, hd):
    q, k, _ = make_qkv(1, 2, 70, hd, seed=200 + hd, kind="edges", Nk=45)
    s = mxq.predict_scores(q.cuda(), k.cuda(), mx_specs()).cpu()
    qc, qe = O.quantize_mxint8(q)
    kc, ke = O.quantize_mxint8(k)
    assert torch.equal(s, O.pred_scores_integer(qc, qe, kc, ke))


# ---- 3. selection ----------------------------------------------------------------------------------------------------
def _check_selection(r, q, k, top_k, bfloat=32):
    Nk = k.shape[2]
    qc, qe = O.quantize_mxint8(q, 32, bfloat)
    kc, ke = O.quantize_mxint8(k, 32, bfloat)
    idx = O.canonical_topk(O.pred_scores_integer(qc, qe, kc, ke), top_k)
    # whole words: the bits past Nk in the last word must be clear
    assert torch.equal(r["mask"].to(torch.int64) & 0xFFFFFFFF, O.idx_to_mask_words(idx, Nk))
    assert torch.equal(r["idx"].to(torch.int64), torch.sort(idx, dim=-1).values)
    assert torch.equal(r["q_codes"], qc) and torch.equal(r["q_exps"], qe)
    assert torch.equal(r["k_codes"], kc) and torch.equal(r["k_exps"], ke)


@pytest.mark.parametrize("Nk", [77, 197, 256, 600])
@pytest.mark.parametrize("hd", H8)
def test_selection_tensor_core(mxq, hd, Nk):
    """Nk <= 256: k_predict_topk_tc; Nk = 600: the long-sequence selection (k_quantize_ops + k_select_long_tc)."""
    q, k, _ = make_qkv(1, 2, 70, hd, seed=300 + hd, kind="edges", Nk=Nk)
    top_k = max(1, int(0.3 * Nk))
    for bfloat in (32, 16):
        _check_selection(select_guarded(q.cuda(), k.cuda(), top_k, bfloat), q, k, top_k, bfloat)


@pytest.mark.parametrize("hd", H4)
def test_selection_cuda_core(mxq, hd):
    restore = _paths(mxq, predict="cuda_core")
    try:
        for Nk in (77, 256):
            q, k, _ = make_qkv(1, 2, 70, hd, seed=400 + hd, kind="edges", Nk=Nk)
            top_k = max(1, int(0.3 * Nk))
            _check_selection(select_guarded(q.cuda(), k.cuda(), top_k), q, k, top_k)
    finally:
        restore()


# ---- 4. the whole path -----------------------------------------------------------------------------------------------
FUSED_MAX_HD = 80       # larger head_dims do not fit the fused kernel's phase-1 staging: the call takes the three kernels

# variant: (B, H, Nq, Nk, top_k, path switches)
WHOLE_PATH = {
    "three_sparse": (2, 3, 197, 197, 20, dict(fused=1)),     # too few heads to fuse: three kernels, cost-follows-k epilogue
    "three_dense": (2, 3, 197, 197, 120, dict(fused=0)),     # three kernels, dense epilogue
    "fused": (8, 8, 160, 160, 40, dict(fused=2)),            # k_fused_pruned_attention
    "long": (1, 2, 300, 300, 75, dict(fused=1)),             # Nk > 256: long-sequence selection and k_attend_long_pair
    "key_bias": (2, 2, 100, 77, 30, dict(fused=1)),          # cross-attention: Nq != Nk, additive key bias
}


def _pruned_guarded(mxq, q, k, v, top_k, out_dtype=torch.float32, **kw):
    B, H, Nq, hd = q.shape
    out = _out_view((B, H, Nq, hd), out_dtype)
    _, mask = mxq.pruned_attention(q, k, v, mx_specs(), top_k, return_mask=True, out=out.t, **kw)
    launches = mxq.last_launch_count()
    out.assert_intact("out")
    return out.t.cpu(), mask, launches


@pytest.mark.parametrize("variant", list(WHOLE_PATH))
@pytest.mark.parametrize("hd", H8)
def test_pruned_attention(mxq, hd, variant):
    B, H, Nq, Nk, top_k, sw = WHOLE_PATH[variant]
    q, k, v = make_qkv(B, H, Nq, hd, seed=500 + hd, kind="randn", Nk=Nk)
    bias = None
    if variant == "key_bias":
        keep = torch.zeros(B, Nk)
        keep[0, :41] = 1
        keep[1, :66] = 1
        bias = ((1 - keep) * -10000.0).reshape(B, 1, 1, Nk)
    restore = _paths(mxq, **sw)
    try:
        out, mask, launches = _pruned_guarded(mxq, q.cuda(), k.cuda(), v.cuda(), top_k,
                                              key_bias=None if bias is None else bias.cuda())
    finally:
        restore()
    if variant == "fused":
        assert launches == (1 if hd <= FUSED_MAX_HD else 3), launches
    elif variant.startswith("three"):
        assert launches == 3, launches
    ref = O.pruned_attention(q, k, v, top_k, integer_scores=True, key_bias=bias)
    assert torch.equal(_words(mask), O.idx_to_mask_words(ref["idx"], Nk))
    assert_out_close(out, ref, v, Nk, 32, OUT_TOL)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("hd", H8)
def test_pruned_attention_16bit(mxq, hd, dtype):
    """16-bit q, k, v and out: the masks of the widened fp32 call, and its output rounded to nearest even."""
    B, H, N, top_k = 2, 2, 197, 40
    q, k, v = (t.to(dtype) for t in make_qkv(B, H, N, hd, seed=600 + hd, kind="randn"))
    qw, kw, vw = (t.float() for t in (q, k, v))
    out16, mask16, _ = _pruned_guarded(mxq, q.cuda(), k.cuda(), v.cuda(), top_k, out_dtype=dtype)
    out32, mask32, _ = _pruned_guarded(mxq, qw.cuda(), kw.cuda(), vw.cuda(), top_k)
    assert torch.equal(mask16, mask32)
    assert torch.equal(out16, out32.to(dtype))
    ref = O.pruned_attention(qw, kw, vw, top_k, integer_scores=True)
    assert torch.equal(_words(mask32), O.idx_to_mask_words(ref["idx"], N))
    assert_out_close(out32, ref, vw, N, 32, OUT_TOL)


# ---- 5. the exact stage alone ----------------------------------------------------------------------------------------
def _sparse_case(mxq, hd, seed):
    B, H, Nq, Nk = 1, 2, 100, 150
    top_k = 45
    q, k, v = make_qkv(B, H, Nq, hd, seed=seed, kind="randn", Nk=Nk)
    ref = O.pruned_attention(q, k, v, top_k, integer_scores=True)
    words = O.idx_to_mask_words(ref["idx"], Nk)
    mask = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32).cuda()
    qc, qe = mxq.quantize_mxint8(q.cuda(), mx_specs())
    kc, ke = mxq.quantize_mxint8(k.cuda(), mx_specs())
    out = _out_view((B, H, Nq, hd), torch.float32)
    mxq.sparse_attention(qc, qe, kc, ke, v.cuda(), mask, mx_specs(), scale=O.default_scale(hd), out=out.t)
    out.assert_intact("out")
    assert_out_close(out.t.cpu(), ref, v, Nk, 32, OUT_TOL)


@pytest.mark.parametrize("hd", H8)
def test_sparse_attention_tensor_core(mxq, hd):
    _sparse_case(mxq, hd, seed=700 + hd)


@pytest.mark.parametrize("hd", H4)
def test_sparse_attention_cuda_core(mxq, hd):
    restore = _paths(mxq, attention="cuda_core")
    try:
        _sparse_case(mxq, hd, seed=800 + hd)
    finally:
        restore()


# ---- 6. the other rankings -------------------------------------------------------------------------------------------
MODE_N, MODE_TOP_K = 256, 77
TWO_STEP_SMEM_HD = (120, 128)   # two operand parts per side: at 225-256 keys these exceed the CTA's shared memory
ELSA_MAX_HD = 80                # ELSA keeps the head_dim x head_dim projection in shared memory


def _elsa_head_margin(q, k, P):
    """Per head: the smallest |hash projection| relative to its row's norm over every query and key row.  Where it
    is within a few fp32 rounding errors of 0 the hash bit depends on the summation order."""
    def rel(x):
        c, e = O.quantize_mxint8(x)
        m = O.dequantize_mxint8(c, e)
        return ((m @ P.T).abs() / m.norm(dim=-1, keepdim=True).clamp(min=1e-30)).amin(dim=(-1, -2))
    return torch.minimum(rel(q), rel(k))


@pytest.mark.parametrize("mode", MODES + ["ELSA"])
@pytest.mark.parametrize("hd", H8)
def test_other_rankings(mxq, hd, mode):
    B, H, N, top_k = 1, 2, MODE_N, MODE_TOP_K
    q, k, v = make_qkv(B, H, N, hd, seed=900 + hd, kind="randn")
    kw = {}
    if mode == "ELSA":
        kw["orthogonal_matrix"] = torch.linalg.qr(torch.randn(hd, hd, generator=torch.Generator().manual_seed(hd)))[0]
    qc, kc, vc = q.cuda(), k.cuda(), v.cuda()
    limit = {"two_step_leading_ones": ("shared memory", hd in TWO_STEP_SMEM_HD),
             "ELSA": ("head_dim", hd > ELSA_MAX_HD)}.get(mode)
    if limit and limit[1]:
        ckw = {n: t.cuda() for n, t in kw.items()}
        with pytest.raises(ValueError, match=limit[0]):
            mxq.predict_topk(qc, kc, mx_specs(), top_k, pred_mode=mode, **ckw)
        with pytest.raises(ValueError, match=limit[0]):
            mxq.pruned_attention(qc, kc, vc, mx_specs(), top_k, pred_mode=mode, **ckw)
        return
    sel = mxq.predict_topk(qc, kc, mx_specs(), top_k, return_idx=True, pred_mode=mode,
                           **{n: t.cuda() for n, t in kw.items()})
    out, mask, _ = _pruned_guarded(mxq, qc, kc, vc, top_k, pred_mode=mode, **{n: t.cuda() for n, t in kw.items()})
    assert torch.equal(mask, sel["mask"])
    ref = O.pruned_attention(q, k, v, top_k, pred_mode=mode, **kw)
    got, want = unpack_mask(mask, N), O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    assert bool((got.sum(-1) == top_k).all())
    if mode == "ELSA":
        margin = _elsa_head_margin(q, k, kw["orthogonal_matrix"])
        rows_equal = (got == want).all(-1).float().mean(dim=-1)                 # (B, H)
        assert bool(((margin <= 1e-5) | (rows_equal == 1.0)).all()), (margin, rows_equal)
        assert float(rows_equal.min()) > 0.98
    else:
        assert torch.equal(got, want)
        assert torch.equal(sel["idx"].cpu().to(torch.int64), torch.sort(ref["idx"], dim=-1).values)
    ref2 = O.pruned_attention(q, k, v, top_k, idx=canonical_idx_from_mask(got, top_k))
    assert_out_close(out, ref2, v, N, 32, OUT_TOL)


# ---- 7. exponent_approximation ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("hd", [16, 48, 80, 112])
def test_exponent_approximation(mxq, hd):
    """The head_dims whose last MX block holds 16 elements."""
    from mx_quantization_b200.predictor import exponent_approximation
    q, k, _ = make_qkv(2, 3, 70, hd, seed=1000 + hd, kind="edges")
    for bfloat in (32, 16):
        ea = exponent_approximation(q.cuda(), k.cuda(), mx_specs(bfloat))
        (qc, kc), (qe, ke), (qs, ks) = ea.codes, ea.exps, ea.signbits
        aq, ak = ea.exponent_based_sign()
        for x, c, e, s, a in ((q, qc, qe, qs, aq), (k, kc, ke, ks, ak)):
            oc, oe = O.quantize_mxint8(x, 32, bfloat)
            assert torch.equal(c.cpu(), oc) and torch.equal(e.cpu(), oe)
            assert torch.equal(_words(s), O.sign_words(oc))
            assert torch.equal(a.cpu(), O.exponent_based_sign(oc, oe))
