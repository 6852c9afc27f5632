"""The additive key bias on the long-sequence path (257 <= Nk <= 8192): pruned_attention(..., key_bias=) against the CPU
oracle (masks bit-exact, outputs within the stated tolerance), the path switches, 16-bit inputs, guard bands, the
cross-attention modules with more than 256 text tokens, graph capture, and the rejections that stay.

Semantics are those of the <= 256-key kernels: the ranked value is fl32(pred_ij + bias_j), ties to the lower key index;
the true score is fl32(fl32(s_ij * scale) + bias_j).  As in test_gpu_long_range.py, the oracle runs per query row on the
first, a middle and the last 128-row tile of every (batch entry, head); the oracle-free checks run on every row.
"""
import contextlib

import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import Guarded, assert_out_close, mx_specs

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-3
TILE = 128


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


def _tile_rows(Nq):
    n = (Nq + TILE - 1) // TILE
    return torch.cat([torch.arange(t * TILE, min((t + 1) * TILE, Nq)) for t in sorted({0, n // 2, n - 1})])


def _top_k(Nk, which):
    return {"one": 1, "p10": max(1, Nk // 10), "p50": Nk // 2, "all": Nk}[which]


def _inputs(kind, B, H, Nq, Nk, hd, seed):
    """q, k, v (B, H, *, hd) and the bias (B, Nk) of one bias kind."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, H, Nq, hd, generator=g)
    k = torch.randn(B, H, Nk, hd, generator=g)
    v = torch.randn(B, H, Nk, hd, generator=g)
    if kind == "pixart":
        # diffusers' (1 - keep) * -10000 with a different valid length per batch entry: none masked, all but one
        # masked, and a third of the keys valid
        lengths = [Nk, 1, max(2, Nk // 3), Nk - 37][:B]
        keep = torch.zeros(B, Nk)
        for b, n in enumerate(lengths):
            keep[b, :n] = 1.0
        bias = (1 - keep) * -10000.0
    elif kind == "constant":
        bias = torch.full((B, Nk), 3.25)
    elif kind == "random":
        # finite fp32 values no integer key carries (24 significant bits, any exponent)
        bias = torch.randn(B, Nk, generator=g) * torch.exp(2.0 * torch.randn(B, Nk, generator=g))
    elif kind == "ties":
        # key rows and bias repeat with period 7: keys j and j + 7 have equal ranked values, so the lower index wins
        k = k[:, :, :7].repeat(1, 1, (Nk + 6) // 7, 1)[:, :, :Nk].contiguous()
        bias = (torch.randint(-4, 5, (B, 7), generator=g).float() * 0.25).repeat(1, (Nk + 6) // 7)[:, :Nk].contiguous()
    else:
        raise ValueError(kind)
    return q, k, v, bias


def _check_rows(q, k, v, bias, top_k, bfloat, flush, out, mask):
    """Oracle on three query tiles of every (batch entry, head): mask words bit-exact, output within tolerance."""
    B, H, Nq, _ = q.shape
    Nk = k.shape[2]
    rows = _tile_rows(Nq)
    m_all, o_all = mask.cpu().to(torch.int64) & 0xFFFFFFFF, out.float().cpu()
    for b in range(B):
        for h in range(H):
            ref = O.pruned_attention(q[b:b + 1, h:h + 1, rows], k[b:b + 1, h:h + 1], v[b:b + 1, h:h + 1], top_k,
                                     bfloat=bfloat, flush=flush, integer_scores=True,
                                     key_bias=bias[b].reshape(1, 1, 1, Nk))
            want = O.idx_to_mask_words(ref["idx"], Nk)
            assert torch.equal(m_all[b:b + 1, h:h + 1, rows], want), f"mask of batch entry {b}, head {h}"
            assert_out_close(o_all[b:b + 1, h:h + 1, rows], ref, v[b:b + 1, h:h + 1], Nk, bfloat, OUT_TOL)


def _every_row_keeps_top_k(mask, Nk, top_k):
    words = mask.cpu().to(torch.int64) & 0xFFFFFFFF
    bits = ((words.unsqueeze(-1) >> torch.arange(32)) & 1).flatten(-2)
    assert bool((bits.sum(-1) == top_k).all()), "a row does not keep exactly top_k keys"
    assert not bool(bits[..., Nk:].any()), "a mask bit past Nk is set"


def long_selection(q, k, bias, top_k, bfloat=32):
    """The long-sequence selection alone (mxp_predict_topk_mode, pred_mode 0) with a workspace of our own: the mask and
    the per-row flags the tensor-core selection leaves at the workspace's end (1: the row was ranked by the CUDA-core
    kernel), as (B, H, Nq) bools."""
    from mx_quantization_b200 import _lib, ops
    lib = _lib.load()
    B, H, Nq, hd = q.shape
    Nk = k.shape[2]
    mask = torch.empty((B, H, Nq, (Nk + 31) // 32), dtype=torch.int32, device="cuda")
    ws_bytes = lib.mxp_predict_topk_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.zeros((ws_bytes,), dtype=torch.uint8, device="cuda")
    kb = bias.reshape(B, Nk).contiguous().cuda()
    rc = lib.mxp_predict_topk_mode(ops._ptr(q), *q.stride()[:3], ops._ptr(k), *k.stride()[:3], B, H, Nq, Nk, hd, top_k,
                                   0, float(hd) ** -0.5, bfloat, 0, ops._ptr(kb), Nk, ops._ptr(mask), None,
                                   ops._ptr(ws), ws_bytes, ops._stream())
    _lib.check(rc, "mxp_predict_topk_mode")
    n = B * H * Nq
    start = ws_bytes - (n + 255) // 256 * 256                  # the flags are the workspace's last region
    return mask, ws[start:start + n].reshape(B, H, Nq).cpu() != 0


def _run(mxq, q, k, v, bias, top_k, specs, out=None):
    B, Nk = bias.shape
    return mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True, out=out,
                                key_bias=bias.reshape(B, 1, 1, Nk).cuda())


# ---------------------------------------------------------------------------------------------- oracle parity
# (Nk, Nq, head_dim, top_k, bfloat, flush, bias kind): every Nk with each bias kind, Nq != Nk throughout
CASES = [
    (257, 64, 64, "one", 32, False, "pixart"),
    (257, 1024, 72, "all", 16, True, "random"),
    (300, 256, 72, "p10", 16, True, "pixart"),
    (300, 1024, 128, "p50", 32, False, "constant"),
    (300, 64, 64, "p10", 32, False, "ties"),
    (1000, 256, 72, "p10", 32, True, "random"),
    (1000, 64, 64, "all", 16, False, "ties"),
    (1000, 1024, 128, "one", 32, False, "pixart"),
    (4096, 256, 128, "p50", 32, False, "pixart"),
    (4096, 1024, 72, "one", 16, True, "random"),
    (4096, 64, 64, "p10", 32, True, "constant"),
    (8192, 256, 72, "p10", 32, False, "pixart"),
    (8192, 64, 128, "p50", 16, False, "ties"),
    (8192, 1024, 64, "all", 32, True, "constant"),
    (8192, 64, 72, "one", 32, False, "random"),
]


@pytest.mark.parametrize("Nk,Nq,hd,tk,bfloat,flush,kind", CASES,
                         ids=[f"Nk{c[0]}-Nq{c[1]}-hd{c[2]}-{c[3]}-bf{c[4]}-{'flush' if c[5] else 'noflush'}-{c[6]}"
                              for c in CASES])
def test_long_key_bias_matches_oracle(mxq, Nk, Nq, hd, tk, bfloat, flush, kind):
    B, H = (4 if kind == "pixart" else 2), 1
    q, k, v, bias = _inputs(kind, B, H, Nq, Nk, hd, seed=Nk + Nq + hd)
    top_k = _top_k(Nk, tk)
    out, mask = _run(mxq, q.cuda(), k.cuda(), v.cuda(), bias, top_k, mx_specs(bfloat, flush))
    torch.cuda.synchronize()
    _every_row_keeps_top_k(mask, Nk, top_k)
    _check_rows(q, k, v, bias, top_k, bfloat, flush, out, mask)


def test_long_key_bias_several_heads(mxq):
    """Two heads per batch entry: the bias is shared by the heads of an entry and differs between entries."""
    B, H, Nq, Nk, hd = 3, 2, 200, 700, 72
    q, k, v, bias = _inputs("pixart", B, H, Nq, Nk, hd, seed=5)
    out, mask = _run(mxq, q.cuda(), k.cuda(), v.cuda(), bias, 60, mx_specs(32, True))
    _check_rows(q, k, v, bias, 60, 32, True, out, mask)


# ---------------------------------------------------------------------------------------------- paths agree
@pytest.mark.parametrize("kind", ["pixart", "random", "ties"])
@pytest.mark.parametrize("Nk,Nq,hd", [(600, 300, 72), (4096, 512, 64)])
def test_long_key_bias_paths_agree(mxq, kind, Nk, Nq, hd):
    """Default switches (tensor-core selection with the sampled fine window), the radix levels alone (set_fused_path(0))
    and the CUDA-core predictor give the same masks and outputs; a zero bias gives the unbiased call's."""
    B, H, top_k = 2, 2, Nk // 8
    q, k, v, bias = _inputs(kind, B, H, Nq, Nk, hd, seed=Nk + 3)
    q, k, v = q.cuda(), k.cuda(), v.cuda()
    sp = mx_specs(32, False)
    res = {}
    for name, kw in {"default": {}, "radix": dict(fused=0), "cuda_core": dict(predict="cuda_core")}.items():
        with _switches(mxq, **kw):
            res[name] = _run(mxq, q, k, v, bias, top_k, sp)
    for name in ("radix", "cuda_core"):
        assert torch.equal(res[name][1], res["default"][1]), name
        assert torch.equal(res[name][0], res["default"][0]), name
    zero = _run(mxq, q, k, v, torch.zeros(B, Nk), top_k, sp)
    plain = mxq.pruned_attention(q, k, v, sp, top_k, return_mask=True)
    assert torch.equal(zero[1], plain[1]) and torch.equal(zero[0], plain[0])


def test_long_key_bias_rows_take_the_tensor_core_selection(mxq):
    """PixArt's mask and a constant bias keep rows on the tensor-core selection; a batch entry with fewer valid keys
    than top_k puts its threshold below the window (every row to the CUDA-core kernel); a random fp32 bias, which no
    integer key carries, sends rows there too.  Every mask equals the CUDA-core predictor's."""
    B, H, Nq, Nk, hd, top_k = 4, 2, 256, 1000, 72, 50
    shares = {}
    for kind in ("pixart", "constant", "random"):
        q, k, v, bias = _inputs(kind, B, H, Nq, Nk, hd, seed=21)
        q, k = q.cuda(), k.cuda()
        mask, flags = long_selection(q, k, bias, top_k)
        with _switches(mxq, predict="cuda_core"):
            want = mxq.pruned_attention(q, k, v.cuda(), mx_specs(32, False), top_k, return_mask=True,
                                        key_bias=bias.reshape(B, 1, 1, Nk).cuda())[1]
        assert torch.equal(mask, want), kind
        shares[kind] = flags.float().mean(dim=(1, 2))
    assert float(shares["pixart"][0]) < 0.5 and float(shares["pixart"][2]) < 0.5, shares     # Nk and Nk / 3 valid keys
    assert float(shares["pixart"][1]) == 1.0, shares                                         # one valid key < top_k
    assert float(shares["constant"].max()) < 0.5, shares
    assert float(shares["random"].min()) > 0.5, shares


# ---------------------------------------------------------------------------------------------- 16-bit inputs
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("Nk,Nq,hd,kind", [(300, 256, 72, "pixart"), (2048, 300, 128, "random"),
                                           (8192, 128, 64, "pixart")])
def test_long_key_bias_half_inputs(mxq, dt, Nk, Nq, hd, kind):
    """16-bit q/k/v with an fp32 bias: the fp32 call's masks on the widened inputs, and its output rounded once;
    an fp32 ``out`` holds the fp32 call's output."""
    B, H, top_k = 2, 2, Nk // 5
    q, k, v, bias = _inputs(kind, B, H, Nq, Nk, hd, seed=Nk + 11)
    q, k, v = (t.cuda().to(dt) for t in (q, k, v))
    sp = mx_specs(32, False)
    out32, mask32 = _run(mxq, q.float(), k.float(), v.float(), bias, top_k, sp)
    out, mask = _run(mxq, q, k, v, bias, top_k, sp)
    assert out.dtype == dt
    assert torch.equal(mask, mask32)
    assert torch.equal(out, out32.to(dt))
    o32 = torch.empty(B, H, Nq, hd, device="cuda")
    _, mask_f = _run(mxq, q, k, v, bias, top_k, sp, out=o32)
    assert torch.equal(mask_f, mask32) and torch.equal(o32, out32)


# ---------------------------------------------------------------------------------------------- guard bands
@pytest.mark.parametrize("hd", [72, 128])
def test_long_key_bias_guard_bands(mxq, hd):
    """Nk = 8192: an output with a padded row stride inside canary bytes; nothing outside the rows is written."""
    B, H, Nq, Nk, top_k = 2, 1, 200, 8192, 500
    q, k, v, bias = _inputs("pixart", B, H, Nq, Nk, hd, seed=hd)
    g = Guarded((B, H, Nq, hd), torch.float32, row_pad=8)
    out, mask = _run(mxq, q.cuda(), k.cuda(), v.cuda(), bias, top_k, mx_specs(32, False), out=g.t)
    torch.cuda.synchronize()
    g.assert_intact("out")
    want, _ = _run(mxq, q.cuda(), k.cuda(), v.cuda(), bias, top_k, mx_specs(32, False))
    assert torch.equal(g.t, want)


# ---------------------------------------------------------------------------------------------- modules
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("S", [300, 1024])
def test_cross_attention_module_long_text(mxq, dt, S):
    """MXCrossAttention with S > 256 text tokens and a padding mask == to_out(core(...)) on its own projections."""
    from mx_quantization_b200.modules import MXCrossAttention
    torch.manual_seed(0)
    dim, heads, B, N, k = 576, 8, 2, 256, 30
    m = MXCrossAttention(dim, heads).cuda().set_config(mx_quant=True, mx_specs=mx_specs(32, True), top_k=True, k=k,
                                                       ex_pred=True, pred_mode="ex_pred").to(dt).eval()
    x = torch.randn(B, N, dim, device="cuda").to(dt)
    enc = torch.randn(B, S, dim, device="cuda").to(dt)
    keep = torch.zeros(B, S, device="cuda"); keep[0, :120] = 1; keep[1, :S - 3] = 1
    amask = ((1 - keep) * -10000.0).reshape(B, 1, S)
    with torch.no_grad():
        y = m(x, encoder_hidden_states=enc, attention_mask=amask)
        assert m.current_timestep == 1
        q = m.to_q(x).view(B, N, heads, dim // heads).transpose(1, 2)
        kk = m.to_k(enc).view(B, S, heads, dim // heads).transpose(1, 2)
        vv = m.to_v(enc).view(B, S, heads, dim // heads).transpose(1, 2)
        core = m.core(q, kk, vv, key_bias=amask.reshape(B, S))
        want = m.to_out(core)
    assert y.dtype == dt and torch.equal(y, want)


def test_pixart_block_long_text(mxq):
    """QuantizedPixArtBlock with S = 300 text tokens on top-k steps == the block expression, bit for bit."""
    from tests.test_gpu_pixart_block import _block_ref, _pixart_block, _text, _timestep
    sp = mx_specs(32, True)
    C, B, T, S = 128, 3, 100, 300
    blk = _pixart_block(torch.float32, sp, C)
    h = torch.randn(B, T, C, device="cuda")
    t = _timestep(B, C, torch.float32, seed=3)
    enc, mask = _text(B, S, C, torch.float32, seed=4)
    for step in range(2):
        with torch.no_grad():
            got = blk(h, encoder_hidden_states=enc, encoder_attention_mask=mask, timestep=t)
            assert blk.attn2.current_timestep == step + 1
            blk.attn1.current_timestep = blk.attn2.current_timestep = step
            want = _block_ref(blk, h, enc, mask, t)
        assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------- graph capture
def test_long_key_bias_graph_capture(mxq):
    B, H, Nq, Nk, hd, top_k = 2, 2, 300, 1000, 72, 100
    sp = mx_specs(32, False)
    g = torch.Generator(device="cuda").manual_seed(3)
    q, k, v = (torch.randn(B, H, n, hd, device="cuda", generator=g) for n in (Nq, Nk, Nk))
    bias = torch.zeros(B, 1, 1, Nk, device="cuda")
    bias[0, ..., 700:] = -10000.0
    out = torch.empty(B, H, Nq, hd, device="cuda")
    mxq.pruned_attention(q, k, v, sp, top_k, out=out, key_bias=bias)        # warm-up (attributes set)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        mxq.pruned_attention(q, k, v, sp, top_k, out=out, key_bias=bias)
    for t in (q, k, v):
        t.copy_(torch.randn(t.shape, device="cuda", generator=g))
    bias[1, ..., 10:] = -10000.0
    graph.replay()
    torch.cuda.synchronize()
    got = out.clone()
    want = mxq.pruned_attention(q, k, v, sp, top_k, key_bias=bias)
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------- kept rejections
def _no_error_pending():
    torch.cuda.synchronize()
    x = torch.ones(4, device="cuda")
    assert float((x + 1).sum()) == 8.0


@pytest.mark.parametrize("mode", ["partial_Q", "partial_K", "MXINT4", "exact"])
def test_other_rankings_with_bias_past_256_keys_raise(mxq, mode):
    B, H, Nq, Nk, hd = 1, 2, 64, 300, 64
    q, k, v, bias = _inputs("pixart", B, H, Nq, Nk, hd, seed=1)
    with pytest.raises(ValueError):
        mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), mx_specs(32, False), 30, pred_mode=mode,
                             key_bias=bias.reshape(B, 1, 1, Nk).cuda())
    _no_error_pending()


def test_cuda_core_attention_with_bias_raises(mxq):
    B, H, Nq, Nk, hd = 1, 2, 64, 300, 64
    q, k, v, bias = _inputs("pixart", B, H, Nq, Nk, hd, seed=2)
    mxq.set_attention_path("cuda_core")
    try:
        with pytest.raises(ValueError):
            mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), mx_specs(32, False), 30,
                                 key_bias=bias.reshape(B, 1, 1, Nk).cuda())
    finally:
        mxq.set_attention_path("tcgen05")
    _no_error_pending()


def test_predict_topk_ex_pred_with_bias_raises(mxq):
    q = torch.randn(1, 1, 64, 64, device="cuda")
    k = torch.randn(1, 1, 300, 64, device="cuda")
    with pytest.raises(ValueError):
        mxq.predict_topk(q, k, mx_specs(32, False), 10, key_bias=torch.zeros(1, 300, device="cuda"))
    _no_error_pending()


def test_cross_attention_excluded_step_past_256_tokens_raises(mxq):
    """An exclude_timesteps step ranks on the true scores (pred_mode="exact"), which stays limited to 256 keys."""
    from mx_quantization_b200.modules import MXCrossAttention
    torch.manual_seed(0)
    dim, heads, B, N, S = 128, 2, 2, 64, 300
    m = MXCrossAttention(dim, heads).cuda().set_config(mx_quant=True, mx_specs=mx_specs(32, True), top_k=True, k=20,
                                                       ex_pred=True, exclude_timesteps={0})
    x = torch.randn(B, N, dim, device="cuda")
    enc = torch.randn(B, S, dim, device="cuda")
    with torch.no_grad(), pytest.raises(ValueError):
        m(x, encoder_hidden_states=enc, attention_mask=torch.zeros(B, 1, S, device="cuda"))
    _no_error_pending()
