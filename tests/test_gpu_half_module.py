"""bf16 / fp16 activations through MX Linear and the attention module shims: a 16-bit mx_linear call equals the fp32
call on the widened x, weight and bias with its result rounded to the 16-bit type, with the same kernel launches; a
16-bit shim equals the composition of fp32 ops calls with a rounding to the 16-bit type at every layer boundary, and
under bf16 + bfloat 16 (every boundary already a bf16 value) a DiT attention module equals the fp32 module bit for bit.
Also the CPU-side dtype and stride validation of mx_linear."""
import copy

import pytest
import torch
import torch.nn as nn

from tests.helpers import mx_specs

HALF = [torch.bfloat16, torch.float16]
HALF_IDS = ["bf16", "fp16"]


def _m():
    import mx_quantization_b200 as m
    return m


# ---------------------------------------------------------------------------------------------- CPU: validation
def test_mx_linear_dtype_and_stride_validation_cpu():
    from mx_quantization_b200 import ops
    with pytest.raises(ValueError, match="float64"):
        ops._linear_rows(torch.zeros(4, 64, dtype=torch.float64))
    with pytest.raises(TypeError):
        ops._linear_rows([[0.0] * 64])
    wide = torch.zeros(4, 68, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="multiple of 8"):
        ops._linear_rows(wide[:, :64])                             # row stride 68
    with pytest.raises(ValueError, match="multiple of 8"):
        ops._linear_rows(torch.zeros(64, 4, dtype=torch.float16).t())   # innermost stride 4
    with pytest.raises(ValueError, match="multiple of 8"):
        ops._linear_rows(torch.zeros(3, 4, 64, dtype=torch.bfloat16).transpose(0, 1))   # rows are not one 2-D view
    ok = torch.zeros(4, 72, dtype=torch.bfloat16)[:, :64]
    r = ops._linear_rows(ok)
    assert r.data_ptr() == ok.data_ptr() and r.stride() == (72, 1)  # 16-bit rows are never copied
    r3 = ops._linear_rows(torch.zeros(2, 3, 64, dtype=torch.float16))
    assert r3.shape == (6, 64)
    f = torch.zeros(64, 4).t()                                      # fp32 keeps its copy rule
    assert ops._linear_rows(f).is_contiguous()
    with pytest.raises(ValueError, match="CUDA"):
        ops.mx_linear(torch.zeros(4, 64, dtype=torch.bfloat16), torch.zeros(4, 64), None, mx_specs())


# ---------------------------------------------------------------------------------------------- GPU: MX Linear
LIN = [  # M, K, N, bias
    (300, 768, 2304, True),        # DeiT-base qkv projection
    (257, 1152, 1152, True),       # DiT / PixArt output projection
    (64, 64, 4, False),
    (1000, 3072, 768, True),       # DeiT-base MLP fc2
]


def _lin_inputs(M, K, N, bias, seed=51):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g) * torch.exp(0.5 * torch.randn(M, 1, generator=g))
    w = torch.randn(N, K, generator=g) * K ** -0.5
    b = torch.randn(N, generator=g) * 0.1 if bias else None
    return x.cuda(), w.cuda(), (b.cuda() if bias else None)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("shape", LIN, ids=lambda s: f"{s[0]}x{s[1]}to{s[2]}{'_bias' if s[3] else ''}")
def test_mx_linear_matches_fp32(dt, bfloat, shape):
    m = _m()
    M, K, N, bias = shape
    sp = mx_specs(bfloat)
    x, w, b = _lin_inputs(M, K, N, bias)
    xh, wh = x.to(dt), w.to(dt)
    bh = None if b is None else b.to(dt)
    wide = torch.zeros(M, K + 64, dtype=dt, device="cuda")       # row-strided view of a wider buffer
    wide[:, :K] = xh
    for xin in (xh, wide[:, :K], xh.reshape(2, M // 2, K) if M % 2 == 0 else xh.reshape(1, M, K)):
        y = m.mx_linear(xin, wh, bh, sp)
        n16 = m.last_launch_count()
        y32 = m.mx_linear(xin.float(), wh.float(), None if bh is None else bh.float(), sp)
        n32 = m.last_launch_count()
        assert y.dtype == dt and y.shape == (*xin.shape[:-1], N)
        assert torch.equal(y, y32.to(dt))
        assert n16 == n32
        if dt == torch.bfloat16 and bfloat == 16:
            assert torch.equal(y.float(), y32)                     # A1-rounded fp32 result: the bf16 store is lossless
    # the weight and the bias may be of any of the three types, independently of x
    y_mixed = m.mx_linear(xh, w, b, sp)
    y_ref = m.mx_linear(xh.float(), w, b, sp)
    assert y_mixed.dtype == dt and torch.equal(y_mixed, y_ref.to(dt))
    assert torch.equal(m.mx_linear(x, wh, bh, sp), m.mx_linear(x, wh.float(), None if bh is None else bh.float(), sp))


@pytest.mark.gpu
@pytest.mark.parametrize("bfloat", [16, 32])
def test_prepared_weight_and_bias_dtypes(bfloat):
    m = _m()
    sp = mx_specs(bfloat)
    M, K, N = 130, 768, 1152
    x, w, b = _lin_inputs(M, K, N, True, seed=7)
    for dt in HALF:
        wh = w.to(dt)
        op16 = m.mx_linear_prepare_weight(wh, sp)
        op32 = m.mx_linear_prepare_weight(wh.float(), sp)
        assert torch.equal(op16, op32)                             # byte-equal operands
        wide = torch.zeros(N, K + 8, dtype=dt, device="cuda")
        wide[:, :K] = wh
        assert torch.equal(m.mx_linear_prepare_weight(wide[:, :K], sp), op32)
        bh = b.to(dt)
        for xin in (x, x.to(torch.bfloat16), x.to(torch.float16)):
            y16b = m.mx_linear(xin, op32, bh, sp, out_features=N)
            y32b = m.mx_linear(xin, op32, bh.float(), sp, out_features=N)
            assert torch.equal(y16b, y32b)
    assert torch.equal(m.mx_linear_prepare_weight(w, sp), m.mx_linear_prepare_weight(w.clone(), sp))

    from mx_quantization_b200.modules import MxLinear
    lin = MxLinear(K, N, mx_specs=sp).cuda()
    with torch.no_grad():
        lin.weight.copy_(w)
        lin.bias.copy_(b)
        y32 = lin(x.to(torch.bfloat16))
        lin.to(torch.bfloat16)                                    # new weight dtype: the cached operand is rebuilt
        y16 = lin(x.to(torch.bfloat16))
        want = m.mx_linear(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(),
                           b.to(torch.bfloat16).float(), sp).to(torch.bfloat16)
    assert y32.dtype == y16.dtype == torch.bfloat16
    assert torch.equal(y16, want)
    assert torch.equal(y32, m.mx_linear(x.to(torch.bfloat16), w, b, sp))


# ---------------------------------------------------------------------------------------------- GPU: module shims
def _lin_ref(lin, x):
    """One MxLinear as the fp32 ops call on the widened tensors, rounded to x's dtype."""
    m = _m()
    b = None if lin.bias is None else lin.bias.detach().float()
    return m.mx_linear(x.float(), lin.weight.detach().float(), b, lin.mx_specs).to(x.dtype)


def _core_ref(core, q, k, v, key_bias=None, dense=False):
    """PrunedAttentionCore as the fp32 pruned_attention call on the widened q, k, v, rounded to q's dtype."""
    m = _m()
    B, H, N, hd = q.shape
    top_k = core.k if (core.k > 0 and not dense) else k.shape[2]
    o = m.pruned_attention(q.float(), k.float(), v.float(), core.mx_specs, top_k, scale=core.scale, key_bias=key_bias)
    return o.permute(0, 2, 1, 3).reshape(B, N, H * hd).to(q.dtype)


def _qkv_attention_ref(mod, x, dense=False):
    """QuantizedAttention / DiT Attention forward, layer by layer: qkv -> core -> proj."""
    B, N, C = x.shape
    H = mod.num_heads
    qkv = _lin_ref(mod.qkv, x).reshape(B, N, 3, H, C // H).permute(2, 0, 3, 1, 4)
    return _lin_ref(mod.proj, _core_ref(mod.core, qkv[0], qkv[1], qkv[2], dense=dense))


def _mlp_ref(mlp, x):
    return _lin_ref(mlp.fc2, mlp.act(_lin_ref(mlp.fc1, x)))


class _TimmAttn(nn.Module):              # the attributes QuantizedAttention takes from timm's Attention
    def __init__(self, dim, heads):
        super().__init__()
        self.num_heads, self.scale = heads, (dim // heads) ** -0.5
        self.qkv, self.proj, self.proj_drop = nn.Linear(dim, 3 * dim), nn.Linear(dim, dim), nn.Dropout(0.0)


class _TimmMlp(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), nn.GELU(), nn.Linear(4 * dim, dim), nn.Dropout(0.0)


class _TimmBlock(nn.Module):
    def __init__(self, dim, heads):
        super().__init__()
        self.norm1, self.attn, self.norm2, self.mlp = nn.LayerNorm(dim), _TimmAttn(dim, heads), nn.LayerNorm(dim), _TimmMlp(dim)

    def forward(self, x):
        x = x + self.attn(self.norm1(x))
        return x + self.mlp(self.norm2(x))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
def test_quantized_attention_and_mlp(dt, bfloat):
    from mx_quantization_b200.modules import QuantizedAttention, QuantizedMlp
    torch.manual_seed(0)
    sp = mx_specs(bfloat)
    attn = QuantizedAttention(_TimmAttn(128, 2), mx_quant=True, mx_specs=sp, top_k=True, k=30).cuda().to(dt)   # hd 64
    mlp = QuantizedMlp(_TimmMlp(128), mx_specs=sp).cuda().to(dt)
    x = torch.randn(2, 197, 128, device="cuda").to(dt)
    with torch.no_grad():
        y = attn(x)
        z = mlp(x)
        assert y.dtype == z.dtype == dt
        assert torch.equal(y, _qkv_attention_ref(attn, x))
        assert torch.equal(z, _mlp_ref(mlp, x))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
def test_dit_attention(dt, bfloat):
    """DiT Attention, head_dim 72, step 0 an excluded (dense) timestep, step 1 pruned."""
    from mx_quantization_b200.modules import Attention
    torch.manual_seed(1)
    sp = mx_specs(bfloat)
    m32 = Attention(576, num_heads=8, qkv_bias=True, mx_quant=True, mx_specs=sp, top_k=True, k=154, ex_pred=True,
                    exclude_timesteps=[0]).cuda()
    m16 = copy.deepcopy(m32).to(dt)
    widened = copy.deepcopy(m16).float()                      # the fp32 module on the widened parameters
    x = (torch.randn(2, 256, 576, device="cuda") * 2).to(dt)
    with torch.no_grad():
        for dense in (True, False):
            y = m16(x)
            y32 = widened(x.float())
            assert y.dtype == dt
            assert torch.equal(y, _qkv_attention_ref(m16, x, dense=dense))
            if dt == torch.bfloat16 and bfloat == 16:
                assert torch.equal(y.float(), y32)             # lossless end to end


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_pixart_self_and_cross_attention(dt):
    from mx_quantization_b200.modules import MXCrossAttention, MXSelfAttention
    torch.manual_seed(2)
    sp = mx_specs(32, True)
    dim, heads, B, N, S = 128, 2, 2, 64, 40
    sa = MXSelfAttention(dim, heads).cuda().set_config(mx_quant=True, mx_specs=sp, top_k=True, k=20, ex_pred=True).to(dt)
    ca = MXCrossAttention(dim, heads).cuda().set_config(mx_quant=True, mx_specs=sp, top_k=True, k=20, ex_pred=True,
                                                        exclude_timesteps=[5]).to(dt)
    x = torch.randn(B, N, dim, device="cuda").to(dt)
    enc = torch.randn(B, S, dim, device="cuda").to(dt)
    keep = torch.zeros(B, S, device="cuda")
    keep[0, :13] = 1
    keep[1, :27] = 1
    amask = ((1 - keep) * -10000.0).reshape(B, 1, S)
    hd = dim // heads
    with torch.no_grad():
        y = sa(x)
        q, k, v = (_lin_ref(lin, x).view(B, N, heads, hd).transpose(1, 2) for lin in (sa.to_q, sa.to_k, sa.to_v))
        assert y.dtype == dt and torch.equal(y, _lin_ref(sa.to_out[0], _core_ref(sa.core, q, k, v)))
        yc = ca(x, encoder_hidden_states=enc, attention_mask=amask)
        q = _lin_ref(ca.to_q, x).view(B, N, heads, hd).transpose(1, 2)
        k, v = (_lin_ref(lin, enc).view(B, S, heads, hd).transpose(1, 2) for lin in (ca.to_k, ca.to_v))
        want = _lin_ref(ca.to_out[0], _core_ref(ca.core, q, k, v, key_bias=amask.reshape(B, S)))
        assert yc.dtype == dt and torch.equal(yc, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_apply_quantization_to_deit_half(dt):
    from mx_quantization_b200.modules import apply_quantization_to_deit
    torch.manual_seed(3)
    model = nn.Module()
    model.blocks = nn.ModuleList([_TimmBlock(128, 2) for _ in range(3)])
    cfg = {"blocks": [0, 1, 2], "components": ["attn", "ffn"], "mx_specs": mx_specs(32, False)}
    apply_quantization_to_deit(model, cfg, top_k=True, k=10, dense_blocks=(2,))
    model.cuda().to(dt)
    x = torch.randn(2, 50, 128, device="cuda").to(dt)
    with torch.no_grad():
        y = x
        for b in model.blocks:
            y = b(y)
        want = x
        for b in model.blocks:
            want = want + _qkv_attention_ref(b.attn, b.norm1(want), dense=b.attn.core.k == 0)
            want = want + _mlp_ref(b.mlp, b.norm2(want))
    assert y.dtype == dt and torch.equal(y, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_rejections_leave_no_cuda_error(dt):
    m = _m()
    from mx_quantization_b200.modules import MXCrossAttention, QuantizedAttention
    torch.manual_seed(4)
    sp = mx_specs()
    x = torch.randn(2, 64, 128, device="cuda").to(dt)
    qa = QuantizedAttention(_TimmAttn(128, 2), mx_quant=True, mx_specs=sp, top_k=True, k=8,
                            pred_mode="partial_Q").cuda().to(dt)
    with torch.no_grad():
        with pytest.raises(ValueError):
            qa(x)
        ca = MXCrossAttention(128, 2).cuda().set_config(mx_quant=True, mx_specs=sp, top_k=True, k=8, ex_pred=True,
                                                        exclude_timesteps=[0]).to(dt)
        with pytest.raises(ValueError):
            ca(x, encoder_hidden_states=x.clone())              # excluded step: "exact" ranking, outside the 16-bit scope
    w = torch.randn(256, 128, device="cuda")
    with pytest.raises(ValueError):
        m.mx_linear(torch.zeros(64, 128, dtype=torch.float64, device="cuda"), w, None, sp)
    wide = torch.zeros(64, 132, dtype=dt, device="cuda")
    with pytest.raises(ValueError):
        m.mx_linear(wide[:, :128], w, None, sp)                    # row stride 132: not a multiple of 8
    torch.cuda.synchronize()
    y = m.mx_linear(x, w, None, sp)                                 # a valid call still runs, no error is pending
    torch.cuda.synchronize()
    assert y.dtype == dt and torch.equal(y, m.mx_linear(x.float(), w, None, sp).to(dt))
