"""adaLN inside the MX Linear kernels: ``mx_linear`` / ``mx_mlp`` with ``shift`` / ``scale`` (the operand quantizer applies
``x * (1 + scale) + shift``) and ``residual`` / ``gate`` (the store computes ``residual + gate * y``) against the eager
torch composition with torch.equal, their launches, ``QuantizedDiTBlock`` against DiT's block expression on the same
modules, and the rejections of malformed adaLN arguments."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.helpers import mx_specs

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["fp32", "bf16", "fp16"]
APPROX = {"gelu": "none", "gelu_tanh": "tanh"}
BT = [(3, 100), (2, 256)]       # T = 100: batch boundaries inside 128-row tiles and a partial last tile


def _m():
    import mx_quantization_b200 as m
    return m


def _modulate(x, shift, scale):
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)


def _adaln(B, T, K, N, dt, seed):
    """x (B, T, K); shift / scale (B, K) as .chunk(6, dim=1) views of one (B, 6K) tensor, batch entry 1 with scale = -1
    and shift = 0 (all-zero MX blocks); gate (B, N) a column slice (row stride 2N); residual (B, T, N)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, K, generator=g) * torch.exp(0.5 * torch.randn(B, T, 1, generator=g))
    table = torch.randn(B, 6 * K, generator=g) * 0.5
    table[1, K:2 * K] = -1.0
    table[1, :K] = 0.0
    gtab = torch.randn(B, 2 * N, generator=g)
    residual = torch.randn(B, T, N, generator=g)
    x, table, gtab, residual = (t.cuda().to(dt) for t in (x, table, gtab, residual))
    shift, scale = table.chunk(6, dim=1)[:2]
    assert shift.stride() == (6 * K, 1) and not shift.is_contiguous()
    return x, shift, scale, residual, gtab[:, N:]


def _weights(N, K, seed, bias=True):
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(N, K, generator=g) * K ** -0.5).cuda()
    b = (torch.randn(N, generator=g) * 0.5).cuda() if bias else None
    return w, b


# ---------------------------------------------------------------------------------------------- mx_linear
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
def test_mx_linear_adaln_equals_composition(dt, bfloat, flush):
    """K = 192, N = 260 (a partial 256-column tile); raw and prepared weights, with and without a bias."""
    m = _m()
    sp = mx_specs(bfloat, flush)
    K, N = 192, 260
    for B, T in BT:
        x, shift, scale, residual, gate = _adaln(B, T, K, N, dt, seed=B * T + bfloat + int(flush))
        w, b = _weights(N, K, seed=bfloat)
        w_op = m.mx_linear_prepare_weight(w, sp)
        for weight, bias, nf in ((w, b.to(dt), None), (w_op, b, N), (w_op, None, N), (w.to(dt), None, None)):
            kw = dict(out_features=nf)
            y = m.mx_linear(x, weight, bias, sp, **kw)
            xm = _modulate(x, shift, scale)
            ym = m.mx_linear(xm, weight, bias, sp, **kw)
            got = m.mx_linear(x, weight, bias, sp, **kw, shift=shift, scale=scale)
            assert got.dtype == dt and got.shape == (B, T, N)
            assert torch.equal(got, ym)
            assert torch.equal(m.mx_linear(x, weight, bias, sp, **kw, residual=residual, gate=gate),
                               residual + gate.unsqueeze(1) * y)
            assert torch.equal(m.mx_linear(x, weight, bias, sp, **kw, shift=shift, scale=scale, residual=residual,
                                           gate=gate),
                               residual + gate.unsqueeze(1) * ym)


# ---------------------------------------------------------------------------------------------- mx_mlp
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
@pytest.mark.parametrize("act", list(APPROX))
def test_mx_mlp_adaln_equals_composition(dt, bfloat, flush, act):
    """K = 192, N1 = 320, N2 = 260: residual + gate * mx_mlp(modulate(x)), raw and prepared weights, with and without
    biases."""
    m = _m()
    sp = mx_specs(bfloat, flush)
    K, N1, N2 = 192, 320, 260
    for B, T in BT:
        x, shift, scale, residual, gate = _adaln(B, T, K, N2, dt, seed=B * T + bfloat + int(flush))
        w1, b1 = _weights(N1, K, seed=1)
        w2, b2 = _weights(N2, N1, seed=2)
        w1_op, w2_op = m.mx_linear_prepare_weight(w1, sp), m.mx_linear_prepare_weight(w2, sp)
        for a1, bb1, a2, bb2, kw in ((w1, b1.to(dt), w2, b2, {}), (w1_op, None, w2_op, None,
                                                                    dict(hidden_features=N1, out_features=N2))):
            want = residual + gate.unsqueeze(1) * m.mx_mlp(_modulate(x, shift, scale), a1, bb1, a2, bb2, sp, act=act, **kw)
            got = m.mx_mlp(x, a1, bb1, a2, bb2, sp, act=act, **kw, shift=shift, scale=scale, residual=residual, gate=gate)
            assert got.dtype == dt and got.shape == (B, T, N2)
            assert torch.equal(got, want)
            # and against the layer-by-layer composition with torch's GELU
            h = m.mx_linear(_modulate(x, shift, scale), a1, bb1, sp, out_features=kw.get("hidden_features"))
            y = m.mx_linear(F.gelu(h, approximate=APPROX[act]), a2, bb2, sp, out_features=kw.get("out_features"))
            assert torch.equal(got, residual + gate.unsqueeze(1) * y)


# ---------------------------------------------------------------------------------------------- launches
@pytest.mark.gpu
def test_adaln_calls_enqueue_the_launches_of_plain_calls():
    m = _m()
    sp = mx_specs(16)
    B, T, K, N = 3, 100, 192, 260
    x, shift, scale, residual, gate = _adaln(B, T, K, N, torch.bfloat16, seed=0)
    w, b = _weights(N, K, seed=0)
    w_op = m.mx_linear_prepare_weight(w, sp)
    for bias in (b, None):
        m.mx_linear(x, w_op, bias, sp, out_features=N)
        plain = m.last_launch_count()
        m.mx_linear(x, w_op, bias, sp, out_features=N, shift=shift, scale=scale, residual=residual, gate=gate)
        assert m.last_launch_count() == plain
    w1_op, w2_op = m.mx_linear_prepare_weight(_weights(320, K, 1)[0], sp), m.mx_linear_prepare_weight(_weights(N, 320, 2)[0], sp)
    m.mx_mlp(x, w1_op, None, w2_op, b, sp, hidden_features=320, out_features=N)
    plain = m.last_launch_count()
    m.mx_mlp(x, w1_op, None, w2_op, b, sp, hidden_features=320, out_features=N, shift=shift, scale=scale,
             residual=residual, gate=gate)
    assert m.last_launch_count() == plain == 4


# ---------------------------------------------------------------------------------------------- QuantizedDiTBlock
class _TimmMlp(nn.Module):
    def __init__(self, dim, act):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), act, nn.Linear(4 * dim, dim), nn.Dropout(0.0)


class _DiTBlock(nn.Module):
    """workloads/DiT/models.py:271-289 (DiTBlock.__init__) with the Attention shim."""

    def __init__(self, C, heads, sp, act, k, exclude_timesteps=()):
        super().__init__()
        from mx_quantization_b200.modules import Attention
        self.norm1 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn = Attention(C, num_heads=heads, qkv_bias=True, mx_quant=True, mx_specs=sp, top_k=True, k=k,
                              ex_pred=True, exclude_timesteps=exclude_timesteps)
        self.norm2 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.mlp = _TimmMlp(C, act)
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(C, 6 * C, bias=True))


def _block_ref(blk, x, c):
    """DiTBlock.forward (models.py:293-297) layer by layer on the wrapped block's modules."""
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = blk.adaLN_modulation(c).chunk(6, dim=1)
    x = x + gate_msa.unsqueeze(1) * blk.attn(_modulate(blk.norm1(x), shift_msa, scale_msa))
    mlp = blk.mlp
    return x + gate_mlp.unsqueeze(1) * mlp.fc2(mlp.act(mlp.fc1(_modulate(blk.norm2(x), shift_mlp, scale_mlp))))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("act", [nn.GELU("tanh"), nn.SiLU()], ids=["gelu_tanh", "silu"])
def test_quantized_dit_block_equals_reference(dt, act, monkeypatch):
    from mx_quantization_b200 import ops
    from mx_quantization_b200.modules import QuantizedDiTBlock
    torch.manual_seed(3)
    C, heads, B, T = 128, 2, 3, 100
    blk = QuantizedDiTBlock(_DiTBlock(C, heads, mx_specs(16), act, k=20, exclude_timesteps={0}), mx_specs=mx_specs(16))
    blk = blk.cuda().to(dt).eval()
    with torch.no_grad():                                   # adaLN-Zero initialises the modulation to 0: use random
        blk.adaLN_modulation[1].weight.normal_(0, 0.1)
        blk.adaLN_modulation[1].bias.normal_(0, 0.3)
    x = torch.randn(B, T, C, device="cuda").to(dt)
    c = torch.randn(B, C, device="cuda").to(dt)
    calls = []
    real = ops.mx_mlp
    monkeypatch.setattr(ops, "mx_mlp", lambda *a, **k: calls.append("gate" in k) or real(*a, **k))
    for step in range(2):                                   # step 0: dense (exclude_timesteps), step 1: top-k
        assert blk.attn.current_timestep == step
        with torch.no_grad():
            got = blk(x, c)
            assert blk.attn.current_timestep == step + 1
            blk.attn.current_timestep = step
            want = _block_ref(blk, x, c)
        assert got.dtype == dt and got.shape == x.shape
        assert torch.equal(got, want)
    assert calls == ([True, True] if type(act) is nn.GELU else [])


@pytest.mark.gpu
def test_quantized_dit_block_dropout_takes_the_composition(monkeypatch):
    from mx_quantization_b200 import ops
    from mx_quantization_b200.modules import QuantizedDiTBlock
    C = 128
    blk = QuantizedDiTBlock(_DiTBlock(C, 2, mx_specs(16), nn.GELU("tanh"), k=20), mx_specs=mx_specs(16)).cuda()
    blk.attn.proj_drop.p = blk.mlp.drop.p = 0.5
    blk.train()
    kwargs = []
    for name in ("mx_linear", "mx_mlp"):
        real = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _r=real, **k: kwargs.append(sorted(k)) or _r(*a, **k))
    with torch.no_grad():
        y = blk(torch.randn(2, 64, C, device="cuda"), torch.randn(2, C, device="cuda"))
    assert y.shape == (2, 64, C) and kwargs
    assert not any(k in ks for ks in kwargs for k in ("shift", "scale", "residual", "gate"))


def test_quantized_dit_block_needs_the_attention_shim():
    from mx_quantization_b200.modules import QuantizedDiTBlock

    class _Blk(nn.Module):
        def __init__(self):
            super().__init__()
            self.norm1, self.norm2 = nn.LayerNorm(64), nn.LayerNorm(64)
            self.attn = nn.MultiheadAttention(64, 2)
            self.mlp = _TimmMlp(64, nn.GELU())
            self.adaLN_modulation = nn.Linear(64, 384)

    with pytest.raises(TypeError, match="Attention"):
        QuantizedDiTBlock(_Blk(), mx_specs=mx_specs(16))


# ---------------------------------------------------------------------------------------------- rejections
@pytest.mark.gpu
def test_adaln_rejections_leave_no_cuda_error():
    from mx_quantization_b200 import _lib, ops
    m = _m()
    sp = mx_specs(16)
    B, T, K, N = 3, 100, 192, 260
    x, shift, scale, residual, gate = _adaln(B, T, K, N, torch.bfloat16, seed=4)
    w, b = _weights(N, K, seed=4)
    w1, _ = _weights(320, K, seed=5)
    w2, _ = _weights(N, 320, seed=6)
    bad = [
        dict(shift=shift),                                                   # a pair half given
        dict(residual=residual),
        dict(scale=scale, residual=residual, gate=gate),
        dict(shift=shift[:, :128], scale=scale[:, :128]),                    # wrong shapes
        dict(shift=shift[:2], scale=scale[:2]),
        dict(residual=residual[:, :, :256], gate=gate[:, :256]),
        dict(residual=residual, gate=gate[:2]),
        dict(shift=shift.float(), scale=scale.float()),                      # mixed dtypes
        dict(residual=residual, gate=gate.half()),
        dict(residual=torch.zeros(B, T, 2 * N, dtype=x.dtype, device="cuda")[:, :, ::2], gate=gate),   # stride 2
        dict(residual=residual, gate=torch.zeros(B, N + 1, dtype=x.dtype, device="cuda")[:, 1:]),     # misaligned
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            m.mx_linear(x, w, b, sp, **kw)
        with pytest.raises(ValueError):
            m.mx_mlp(x, w1, None, w2, b, sp, **kw)
    with pytest.raises(ValueError, match="B, T"):                            # 2-D x with modulation
        m.mx_linear(x.reshape(B * T, K), w, b, sp, shift=shift, scale=scale)
    with pytest.raises(ValueError, match="B, T"):
        m.mx_mlp(x.reshape(B * T, K), w1, None, w2, b, sp, residual=residual, gate=gate)
    # tokens not dividing M, through the C entry point (the Python layer takes tokens from x's shape)
    lib = _lib.load()
    w_op = m.mx_linear_prepare_weight(w, sp)
    out = torch.empty(B * T, N, dtype=x.dtype, device="cuda")
    ws_bytes = lib.mxp_mx_linear_workspace_bytes(B * T, N, K)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    p = ops._ptr
    for tokens in (7, 0):
        rc = lib.mxp_mx_linear_adaln_dt(p(x), _lib.MXP_DT_BF16, K, B * T, K, p(w_op), N, p(None), _lib.MXP_DT_F32, 16, 0,
                                        p(out), N, tokens, p(shift), 6 * K, p(scale), 6 * K, p(None), 0, p(None), 0,
                                        p(ws), ws_bytes, ops._stream())
        with pytest.raises(ValueError, match="tokens"):
            _lib.check(rc, "mxp_mx_linear_adaln_dt")
    torch.cuda.synchronize()
    got = m.mx_linear(x, w, b, sp, shift=shift, scale=scale, residual=residual, gate=gate)     # a valid call still runs
    torch.cuda.synchronize()
    assert torch.equal(got, residual + gate.unsqueeze(1) * m.mx_linear(_modulate(x, shift, scale), w, b, sp))
