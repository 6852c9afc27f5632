"""Long-sequence attention over the whole key range mxp_limits() advertises (Nk <= 8192, head_dim <= 128), against
the CPU oracle, and the limit itself.

The oracle (oracle.mxint8_oracle.pruned_attention with integer_scores=True) is exact per query row: a row's codes,
predicted scores, top-k and P windows depend only on that row and on the whole K and V (V is quantized along tokens,
over every key).  So each case runs the kernels on whole heads and compares three query tiles of 128 rows with the
oracle run on those rows alone: the first tile, one from the middle and the last (partial where Nq % 128 != 0).
Whole-head oracles at 8192 keys would take seconds each.  The checks that need no oracle run on every row: each row
keeps exactly top_k keys, no mask bit past Nk is set, and both predictor paths give the same masks.
"""
import contextlib

import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import Guarded, assert_out_close, long_inputs, make_qkv, mx_specs, select_guarded

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-3
MAX_KEYS = 8192         # mxp_limits()
TILE = 128              # query rows per tile of the long-sequence kernels
PATHS = ["tcgen05", "cuda_core"]


@pytest.fixture(scope="module")
def mxq():
    import mx_quantization_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


@contextlib.contextmanager
def _switches(mxq, predict="tcgen05", fused=1):
    mxq.set_predict_path(predict)
    mxq.set_fused_path(fused)
    try:
        yield
    finally:
        mxq.set_predict_path("tcgen05")
        mxq.set_fused_path(True)


def _words(t):
    return t.cpu().to(torch.int64) & 0xFFFFFFFF


def _tile_rows(Nq):
    """Row indices of the first query tile, a middle one and the last one."""
    n = (Nq + TILE - 1) // TILE
    return torch.cat([torch.arange(t * TILE, min((t + 1) * TILE, Nq)) for t in sorted({0, n // 2, n - 1})])


class RowOracle:
    """The oracle on some query rows of one head (b, h): the predicted scores once, then any top_k."""

    def __init__(self, q, k, v, rows, b=0, h=0, bfloat=32):
        self.b, self.h, self.rows, self.bfloat = b, h, rows, bfloat
        self.q = q[b:b + 1, h:h + 1, rows]
        self.k = k[b:b + 1, h:h + 1]
        self.v = None if v is None else v[b:b + 1, h:h + 1]
        self.qc, self.qe = O.quantize_mxint8(self.q, 32, bfloat)
        self.kc, self.ke = O.quantize_mxint8(self.k, 32, bfloat)
        self.pred = O.pred_scores_integer(self.qc, self.qe, self.kc, self.ke)

    def idx(self, top_k):
        return O.canonical_topk(self.pred, top_k)

    def result(self, top_k):
        return O.pruned_attention(self.q, self.k, self.v, top_k, bfloat=self.bfloat, idx=self.idx(top_k))

    def rows_of(self, t):
        return t[self.b:self.b + 1, self.h:self.h + 1, self.rows.to(t.device)].cpu()

    def check(self, top_k, mask=None, sel=None, out=None):
        """mask, predict_topk's dict and out (whole-tensor kernel results) on this oracle's rows."""
        Nk = self.k.shape[2]
        ref = self.result(top_k) if out is not None else {"idx": self.idx(top_k)}
        want = O.idx_to_mask_words(ref["idx"], Nk)         # whole words: the bits past Nk must be clear
        for m in (mask, None if sel is None else sel["mask"]):
            if m is not None:
                got = _words(self.rows_of(m))
                assert torch.equal(got, want), (
                    f"masks differ from the oracle in {int((got != want).any(-1).sum())} rows")
        if sel is not None and "idx" in sel:
            assert torch.equal(self.rows_of(sel["idx"]).to(torch.int64), torch.sort(ref["idx"], dim=-1).values)
        if sel is not None and "q_codes" in sel:
            assert torch.equal(self.rows_of(sel["q_codes"]), self.qc)
            assert torch.equal(self.rows_of(sel["q_exps"]), self.qe)
            kh = (slice(self.b, self.b + 1), slice(self.h, self.h + 1))
            assert torch.equal(sel["k_codes"][kh].cpu(), self.kc) and torch.equal(sel["k_exps"][kh].cpu(), self.ke)
        if out is not None:
            assert_out_close(self.rows_of(out).float(), ref, self.v, Nk, self.bfloat, OUT_TOL)


def _popcount(words):
    x = words.to(torch.int64) & 0xFFFFFFFF
    x = x - ((x >> 1) & 0x55555555)
    x = (x & 0x33333333) + ((x >> 2) & 0x33333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F
    return ((x * 0x01010101) & 0xFFFFFFFF) >> 24


def _check_every_row(mask, Nk, top_k):
    """On the device, every row of every head: exactly top_k keys kept and no bit set past Nk."""
    kept = _popcount(mask).sum(-1)
    assert bool((kept == top_k).all()), f"{int((kept != top_k).sum())} rows do not keep exactly top_k = {top_k} keys"
    if Nk % 32:
        assert not bool(((mask[..., -1].to(torch.int64) & 0xFFFFFFFF) >> (Nk % 32)).any()), "mask bits set past Nk"


def _run_paths(mxq, q, k, v, top_k, bfloat=32, paths=PATHS):
    """predict_topk (idx, codes) and pruned_attention on each predictor path; masks of both calls and of all paths are
    the same on every row."""
    specs = mx_specs(bfloat)
    res = {}
    for path in paths:
        with _switches(mxq, predict=path):
            sel = mxq.predict_topk(q, k, specs, top_k, return_idx=True, return_codes=True)
            out, mask = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
        assert torch.equal(mask, sel["mask"]), f"{path}: pruned_attention and predict_topk masks differ"
        _check_every_row(mask, k.shape[2], top_k)
        res[path] = (sel, out)
    first = res[paths[0]][0]
    for path in paths[1:]:
        assert torch.equal(res[path][0]["mask"], first["mask"]), f"{paths[0]} vs {path}: masks differ"
        assert torch.equal(res[path][0]["idx"], first["idx"]), f"{paths[0]} vs {path}: index lists differ"
    return res


# ---- 1. key-count edges ----------------------------------------------------------------------------------------------
# 257: the first long shape; 384 / 385: the last 128-key block holds 128 keys / one key; 1920 / 1921: 15 / 16 key
# blocks, where the selection's fine window goes from one sampled block to two; 5374 / 5375: where key records padded
# to 8 words would no longer fit the CUDA-core selection's shared memory at head_dim > 96; 8191 / 8192: the limit.
# Every key count at head_dim 64, 72 and 128, and 104 at the record-size edge and at the limit.
EDGE_NK = [257, 384, 385, 1920, 1921, 4097, 5374, 5375, 6000, 8191, 8192]
EDGE =[(Nk, hd) for Nk in EDGE_NK for hd in [64, 72, 128] + ([104] if Nk in (5374, 5375, 8192) else [])]


@pytest.mark.parametrize("Nk,hd", EDGE, ids=[f"Nk{Nk}-hd{hd}" for Nk, hd in EDGE])
def test_key_count_edges(mxq, Nk, hd):
    """top_k = 1, 10 %, 50 %, Nk - 1 and Nk on both predictor paths."""
    q, k, v = make_qkv(1, 1, Nk, hd, seed=Nk + hd)
    orc = RowOracle(q, k, v, _tile_rows(Nk))
    qd, kd, vd = q.cuda(), k.cuda(), v.cuda()
    for top_k in (1, Nk // 10, Nk // 2, Nk - 1, Nk):
        for sel, out in _run_paths(mxq, qd, kd, vd, top_k).values():
            orc.check(top_k, sel=sel, out=out)


# ---- 2. rectangular shapes -------------------------------------------------------------------------------------------
RECT = [  # Nq, Nk, hd, bfloat, top_k
    (1, 8192, 128, 32, 819),
    (129, 8192, 72, 32, 4096),
    (300, 8192, 128, 16, 819),         # three query tiles: one pair and a half pair
    (8192, 8192, 104, 16, 2048),
    (8192, 300, 128, 32, 75),
]


@pytest.mark.parametrize("Nq,Nk,hd,bfloat,top_k", RECT)
def test_rectangular(mxq, Nq, Nk, hd, bfloat, top_k):
    q, k, v = make_qkv(1, 1, Nq, hd, seed=Nq + Nk + hd, Nk=Nk)
    orc = RowOracle(q, k, v, _tile_rows(Nq), bfloat=bfloat)
    for sel, out in _run_paths(mxq, q.cuda(), k.cuda(), v.cuda(), top_k, bfloat).values():
        orc.check(top_k, sel=sel, out=out)


# ---- 3. many heads ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,H,N,hd,top_k,heads", [
    (16, 16, 4096, 72, 1024, (0, 137, 255)),      # bench.py's dit_long_c5: the selection splits pairs by a divisor
    (4, 300, 512, 64, 128, (0, 599, 1199)),       # enough heads that every head takes one CTA
])
def test_many_heads(mxq, B, H, N, hd, top_k, heads):
    q, k, v = make_qkv(B, H, N, hd, seed=B * H + N)
    qd, kd, vd = q.cuda(), k.cuda(), v.cuda()
    specs = mx_specs()
    out, mask = mxq.pruned_attention(qd, kd, vd, specs, top_k, return_mask=True)
    sel = mxq.predict_topk(qd, kd, specs, top_k, return_idx=True, return_codes=True)
    assert torch.equal(mask, sel["mask"])
    _check_every_row(mask, N, top_k)
    for head in heads:
        RowOracle(q, k, v, _tile_rows(N), b=head // H, h=head % H).check(top_k, sel=sel, out=out)
    # one (b, h) slice alone: the same bits as inside the batched call
    b, h = heads[1] // H, heads[1] % H
    out1, mask1 = mxq.pruned_attention(qd[b:b + 1, h:h + 1], kd[b:b + 1, h:h + 1], vd[b:b + 1, h:h + 1], specs, top_k,
                                       return_mask=True)
    assert torch.equal(mask1, mask[b:b + 1, h:h + 1]) and torch.equal(out1, out[b:b + 1, h:h + 1])
    with _switches(mxq, predict="cuda_core"):
        core = mxq.predict_topk(qd, kd, specs, top_k, return_idx=True)
    assert torch.equal(core["mask"], sel["mask"]) and torch.equal(core["idx"], sel["idx"])


# ---- 4. input kinds at the top of the range --------------------------------------------------------------------------
KINDS = ["randn", "lognormal0.25", "lognormal0.5", "lognormal1.5", "ties", "constant", "zeros", "skewed", "outliers"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("hd,kfrac", [(72, 0.1), (128, 0.5)])
def test_selection_paths_agree_at_the_limit(mxq, kind, hd, kfrac):
    """The sampled fine window, the radix levels alone (fused path 0) and the CUDA-core kernel give the same masks and
    index lists at 8192 keys.  outliers and lognormal1.5 send rows outside the tensor-core window to the CUDA-core
    kernel, which at head_dim 128 keeps the largest key records."""
    N = MAX_KEYS
    q, k = long_inputs(kind, 1, N, hd, seed=N + hd)
    top_k = int(kfrac * N)
    qd, kd = q.cuda(), k.cuda()
    res = {}
    for name, fused, pred in (("fine", 1, "tcgen05"), ("radix", 0, "tcgen05"), ("core", 1, "cuda_core")):
        with _switches(mxq, predict=pred, fused=fused):
            res[name] = mxq.predict_topk(qd, kd, mx_specs(), top_k, return_idx=True)
    _check_every_row(res["fine"]["mask"], N, top_k)
    for name in ("radix", "core"):
        assert torch.equal(res["fine"]["mask"], res[name]["mask"]), f"fine window vs {name}: masks differ"
        assert torch.equal(res["fine"]["idx"], res[name]["idx"]), f"fine window vs {name}: index lists differ"
    if kind in ("randn", "outliers"):
        RowOracle(q, k, None, _tile_rows(N)).check(top_k, sel=res["fine"])


# ---- 5. 16-bit inputs at 8192 keys -----------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_half_inputs_at_the_limit(mxq, dt):
    B, H, N, hd, top_k = 1, 2, MAX_KEYS, 128, 820
    q, k, v = make_qkv(B, H, N, hd, seed=17)
    qh, kh, vh = (x.to(dt).cuda() for x in (q, k, v))
    q32, k32, v32 = qh.float(), kh.float(), vh.float()
    sp = mx_specs()
    s16 = mxq.predict_topk(qh, kh, sp, top_k, return_idx=True)
    n16 = mxq.last_launch_count()
    s32 = mxq.predict_topk(q32, k32, sp, top_k, return_idx=True)
    n32 = mxq.last_launch_count()
    assert torch.equal(s16["mask"], s32["mask"]) and torch.equal(s16["idx"], s32["idx"]) and n16 == n32
    out16, mask16 = mxq.pruned_attention(qh, kh, vh, sp, top_k, return_mask=True)
    n16 = mxq.last_launch_count()
    out32, mask32 = mxq.pruned_attention(q32, k32, v32, sp, top_k, return_mask=True)
    n32 = mxq.last_launch_count()
    assert out16.dtype == dt and n16 == n32
    assert torch.equal(mask16, mask32) and torch.equal(mask32, s32["mask"])
    assert torch.equal(out16, out32.to(dt))
    RowOracle(q32.cpu(), k32.cpu(), v32.cpu(), _tile_rows(N), h=1).check(top_k, mask=mask32, out=out32)


# ---- 6. the exact stage alone ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("top_k", [1, MAX_KEYS])
def test_sparse_attention_at_the_limit(mxq, top_k):
    """The oracle's kept set at 8192 keys, head_dim 128: one key per row, and every key (the online softmax over 64
    dense key blocks).  The query rows are 300 rows of an 8192-row head (its first, a middle and part of its last
    tile): three query tiles, the last partial."""
    Nk, hd = MAX_KEYS, 128
    q, k, v = make_qkv(1, 1, Nk, hd, seed=23 + top_k)
    q = q[:, :, _tile_rows(Nk)[:300]]
    ref = O.pruned_attention(q, k, v, top_k, integer_scores=True)
    words = O.idx_to_mask_words(ref["idx"], Nk)
    mask = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32).cuda()
    out = Guarded(tuple(q.shape), torch.float32, row_pad=4)
    mxq.sparse_attention(ref["q_codes"].cuda(), ref["q_exps"].cuda(), ref["k_codes"].cuda(), ref["k_exps"].cuda(),
                         v.cuda(), mask, mx_specs(), scale=O.default_scale(hd), out=out.t)
    out.assert_intact("out")
    assert_out_close(out.t.cpu(), ref, v, Nk, 32, OUT_TOL)


# ---- 7. guard bands --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("hd", [72, 128])
@pytest.mark.parametrize("Nk,top_k", [(4097, 2048), (8191, 819), (8192, 8191)])
def test_selection_guard_bands(mxq, Nk, top_k, hd, path):
    """mask, idx and both code / exponent outputs inside canary bytes: no store past a row or past an output."""
    q, k, _ = make_qkv(1, 1, Nk, hd, seed=Nk + hd + 1, kind="edges")
    with _switches(mxq, predict=path):
        r = select_guarded(q.cuda(), k.cuda(), top_k)
    RowOracle(q, k, None, _tile_rows(Nk)).check(top_k, sel=r)


# ---- 8. the limits ---------------------------------------------------------------------------------------------------
def test_limits(mxq):
    assert mxq.limits() == (MAX_KEYS, 128)


def _rejected_untouched(mxq, rc, what, guards):
    """A call past the key limit: it enqueued nothing, wrote nothing and returned MXP_E_UNSUPPORTED."""
    from mx_quantization_b200 import _lib
    assert mxq.last_launch_count() == 0, f"{what}: {mxq.last_launch_count()} launches before the rejection"
    for name, g in guards.items():
        g.assert_untouched(f"{what} {name}")
    assert rc == _lib.MXP_E_UNSUPPORTED, f"{what}: returned {rc}"
    with pytest.raises(ValueError, match=str(MAX_KEYS + 1)):
        _lib.check(rc, what)


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_keys_past_the_limit_rejected(mxq, dt):
    """Nk = 8193 at head_dim 64, a shape every kernel could run: each entry point that takes keys rejects it before any
    launch, through the C ABI into canary-filled outputs and through the Python entry points."""
    from mx_quantization_b200 import _lib, ops
    lib, p, st = _lib.load(), ops._ptr, ops._stream()
    B, H, Nq, Nk, hd, top_k = 1, 2, 64, MAX_KEYS + 1, 64, 100
    nb, nw = (hd + 31) // 32, (Nk + 31) // 32
    code = ops.DTYPE_CODES[dt]
    q, k, v = (x.to(dt).cuda() for x in make_qkv(B, H, Nq, hd, seed=29, Nk=Nk))
    sp = mx_specs()

    if dt == torch.float32:         # the dense score aid reads fp32 only
        g = {"scores": Guarded((B, H, Nq, Nk), torch.float32)}
        rc = lib.mxp_predict_scores(p(q), *q.stride()[:3], p(k), *k.stride()[:3], B, H, Nq, Nk, hd, 32, 0,
                                    p(g["scores"].t), st)
        _rejected_untouched(mxq, rc, "mxp_predict_scores", g)
        with pytest.raises(ValueError):
            mxq.predict_scores(q, k, sp)

    g = {"mask": Guarded((B, H, Nq, nw), torch.int32), "idx": Guarded((B, H, Nq, top_k), torch.int32),
         "q_codes": Guarded((B, H, Nq, hd), torch.int8), "q_exps": Guarded((B, H, Nq, nb), torch.int8),
         "k_codes": Guarded((B, H, Nk, hd), torch.int8), "k_exps": Guarded((B, H, Nk, nb), torch.int8)}
    ws_bytes = lib.mxp_predict_topk_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device="cuda")
    rc = lib.mxp_predict_topk_dt(p(q), *q.stride()[:3], p(k), *k.stride()[:3], code, B, H, Nq, Nk, hd, top_k, 32, 0,
                                 *(p(g[n].t) for n in ("mask", "idx", "q_codes", "q_exps", "k_codes", "k_exps")),
                                 p(ws), ws_bytes, st)
    _rejected_untouched(mxq, rc, "mxp_predict_topk_dt", g)
    with pytest.raises(ValueError):
        mxq.predict_topk(q, k, sp, top_k, return_idx=True)

    # every key kept: valid operands for the exact stage
    qc = torch.zeros(B, H, Nq, hd, dtype=torch.int8, device="cuda")
    kc = torch.ones(B, H, Nk, hd, dtype=torch.int8, device="cuda")
    qe, ke = (torch.zeros(B, H, n, nb, dtype=torch.int8, device="cuda") for n in (Nq, Nk))
    mask = torch.full((B, H, Nq, nw), -1, dtype=torch.int32, device="cuda")
    mask[..., -1] = (1 << (Nk % 32)) - 1
    g = {"out": Guarded((B, H, Nq, hd), dt, row_pad=8)}
    o = g["out"].t
    ws_bytes = lib.mxp_sparse_attention_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device="cuda")
    rc = lib.mxp_sparse_attention_dt(p(qc), p(qe), p(kc), p(ke), p(v), *v.stride()[:3], code, p(mask), B, H, Nq, Nk,
                                     hd, O.default_scale(hd), 32, 0, p(o), *o.stride()[:3], code, p(ws), ws_bytes, st)
    _rejected_untouched(mxq, rc, "mxp_sparse_attention_dt", g)
    with pytest.raises(ValueError):
        mxq.sparse_attention(qc, qe, kc, ke, v, mask, sp)

    g = {"out": Guarded((B, H, Nq, hd), dt, row_pad=8), "mask": Guarded((B, H, Nq, nw), torch.int32)}
    o = g["out"].t
    ws_bytes = lib.mxp_pruned_attention_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    rc = lib.mxp_pruned_attention_dt(p(q), *q.stride()[:3], p(k), *k.stride()[:3], p(v), *v.stride()[:3], code, B, H,
                                     Nq, Nk, hd, top_k, O.default_scale(hd), 32, 0, p(o), *o.stride()[:3], code,
                                     p(None), 0, p(g["mask"].t), p(ws), ws_bytes, st)
    _rejected_untouched(mxq, rc, "mxp_pruned_attention_dt", g)
    with pytest.raises(ValueError):
        mxq.pruned_attention(q, k, v, sp, top_k)
    torch.cuda.synchronize()


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_quantizer_past_the_key_limit(mxq, dt):
    """The key limit is not a row limit: the quantizer takes 10 000 rows."""
    x = make_qkv(1, 2, 10000, 64, seed=31)[0].to(dt)
    codes, exps = mxq.quantize_mxint8(x.cuda(), mx_specs())
    oc, oe = O.quantize_mxint8(x.float())
    assert torch.equal(codes.cpu(), oc) and torch.equal(exps.cpu(), oe)
