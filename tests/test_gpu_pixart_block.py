"""PixArt-alpha's adaLN-single block in the MX kernels: ``MXSelfAttention.forward_adaln`` (q, k and v from one GEMM on the
concatenated weight, the modulation in its quantizer, the gated residual in to_out's store) against the torch expression
with torch.equal, ``QuantizedMlp`` built from diffusers' ``FeedForward``, ``QuantizedPixArtBlock`` against the block
expression written layer by layer on the same modules, the launches, the q/k/v operand cache, the dropout fallback and the
rejections."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.helpers import mx_specs

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["fp32", "bf16", "fp16"]
BT = [(3, 100), (2, 256)]       # T = 100: batch boundaries inside 128-row tiles and a partial last tile
HEADS = [(128, 2), (576, 8)]    # head_dim 64 and 72


class _GELU(nn.Module):
    """diffusers.models.activations.GELU: owns the feed-forward's first Linear."""

    def __init__(self, dim_in, dim_out, approximate="none", bias=True):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out, bias=bias)
        self.approximate = approximate

    def forward(self, x):
        return F.gelu(self.proj(x), approximate=self.approximate)


class _GEGLU(nn.Module):
    """diffusers.models.activations.GEGLU: a projection without an ``approximate`` GELU."""

    def __init__(self, dim_in, dim_out):
        super().__init__()
        self.proj = nn.Linear(dim_in, 2 * dim_out)


class _FeedForward(nn.Module):
    """diffusers.models.attention.FeedForward (PixArt: activation_fn="gelu-approximate")."""

    def __init__(self, dim, approximate="tanh", dropout=0.0, final_dropout=False, act=None):
        super().__init__()
        self.net = nn.ModuleList([act or _GELU(dim, 4 * dim, approximate), nn.Dropout(dropout), nn.Linear(4 * dim, dim)])
        if final_dropout:
            self.net.append(nn.Dropout(dropout))


class _PixArtBlock(nn.Module):
    """BasicTransformerBlock(norm_type="ada_norm_single") as PixArt builds it, with the attention shims after set_config."""

    def __init__(self, C, heads, sp, k=20, k_cross=30, exclude_self=(), exclude_cross=(), ff=None, has_bias=True):
        super().__init__()
        from mx_quantization_b200.modules import MXCrossAttention, MXSelfAttention
        self.norm1 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn1 = MXSelfAttention(C, heads, has_bias=has_bias).set_config(
            mx_quant=True, mx_specs=sp, top_k=True, k=k, ex_pred=True, exclude_timesteps=exclude_self)
        self.norm2 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn2 = MXCrossAttention(C, heads).set_config(
            mx_quant=True, mx_specs=sp, top_k=True, k=k_cross, ex_pred=True, exclude_timesteps=exclude_cross)
        self.ff = ff or _FeedForward(C)
        self.scale_shift_table = nn.Parameter(torch.randn(6, C) / C ** 0.5)


def _modulate(x, shift, scale):
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)


def _adaln(B, T, C, dt, seed):
    """x, residual (B, T, C); shift / scale / gate (B, C) as .squeeze(1) of (B, 1, C) chunks of one (B, 6, C) tensor (row
    stride 6C), batch entry 1 with scale = -1 and shift = 0 (all-zero MX blocks)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, C, generator=g) * torch.exp(0.5 * torch.randn(B, T, 1, generator=g))
    residual = torch.randn(B, T, C, generator=g)
    table = torch.randn(B, 6, C, generator=g) * 0.5
    table[1, 1] = -1.0
    table[1, 0] = 0.0
    x, residual, table = (t.cuda().to(dt) for t in (x, residual, table))
    shift, scale, gate = (t.squeeze(1) for t in table.chunk(6, dim=1)[:3])
    assert shift.stride() == (6 * C, 1)
    return x, shift, scale, residual, gate


def _self_attention(C, heads, sp, dt, has_bias=True, seed=0):
    from mx_quantization_b200.modules import MXSelfAttention
    torch.manual_seed(seed)
    a = MXSelfAttention(C, heads, has_bias=has_bias).set_config(mx_quant=True, mx_specs=sp, top_k=True, k=20,
                                                                ex_pred=True)
    return a.cuda().to(dt).eval()


def _attn_ref(a, x, shift, scale, residual, gate):
    """The expression forward_adaln computes, on forward's three projections; leaves current_timestep where it was."""
    step = a.current_timestep
    y = residual + gate.unsqueeze(1) * a(_modulate(x, shift, scale))
    a.current_timestep = step
    return y


# ---------------------------------------------------------------------------------------------- self-attention half
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
@pytest.mark.parametrize("has_bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("C,heads", HEADS, ids=["hd64", "hd72"])
def test_self_attention_forward_adaln_equals_expression(dt, bfloat, flush, has_bias, C, heads):
    sp = mx_specs(bfloat, flush)
    a = _self_attention(C, heads, sp, dt, has_bias, seed=bfloat + int(flush))
    with torch.no_grad():
        for B, T in BT:
            x, shift, scale, residual, gate = _adaln(B, T, C, dt, seed=B * T + C)
            got = a.forward_adaln(x, shift, scale, residual, gate)
            assert a.current_timestep == 1
            a.current_timestep = 0
            assert got.dtype == dt and got.shape == (B, T, C)
            assert torch.equal(got, _attn_ref(a, x, shift, scale, residual, gate))


@pytest.mark.gpu
def test_self_attention_forward_adaln_makes_one_qkv_call(monkeypatch):
    """forward_adaln: one mx_linear call for q/k/v (with the modulation) and one for to_out (with the gated residual),
    each enqueueing a plain call's launches; forward: three projection calls and to_out."""
    from mx_quantization_b200 import ops
    sp = mx_specs(32, True)
    C, B, T = 576, 2, 256
    a = _self_attention(C, 8, sp, torch.bfloat16)
    x, shift, scale, residual, gate = _adaln(B, T, C, torch.bfloat16, seed=1)
    calls = []
    real = ops.mx_linear

    def spy(*args, **kw):
        y = real(*args, **kw)
        calls.append((sorted(k for k in kw if kw[k] is not None and k != "out_features"), ops.last_launch_count()))
        return y

    monkeypatch.setattr(ops, "mx_linear", spy)
    with torch.no_grad():
        a.forward_adaln(x, shift, scale, residual, gate)
        fused, calls[:] = list(calls), []
        a(_modulate(x, shift, scale))
        plain = list(calls)
    assert [kw for kw, _ in fused] == [["scale", "shift"], ["gate", "residual"]]
    assert [kw for kw, _ in plain] == [[], [], [], []]
    launches = {n for _, n in fused + plain}
    assert len(launches) == 1 and launches.pop() > 0


@pytest.mark.gpu
def test_self_attention_qkv_operand_cache():
    """The concatenated operand is built once, rebuilt after a weight written through .data plus invalidate(), and
    after load_state_dict; the parameters stay to_q / to_k / to_v's own."""
    sp = mx_specs(32, True)
    C, B, T = 128, 3, 100
    a = _self_attention(C, 2, sp, torch.float32)
    x, shift, scale, residual, gate = _adaln(B, T, C, torch.float32, seed=2)
    params = [a.to_q.weight, a.to_k.weight, a.to_v.weight]
    with torch.no_grad():
        y0 = a.forward_adaln(x, shift, scale, residual, gate)
        op = a._qkv_op
        a.current_timestep = 0
        assert torch.equal(a.forward_adaln(x, shift, scale, residual, gate), y0) and a._qkv_op is op
        a.current_timestep = 0

        a.to_k.weight.data.mul_(-0.5)
        a.to_k.invalidate()
        y1 = a.forward_adaln(x, shift, scale, residual, gate)
        a.current_timestep = 0
        assert not torch.equal(y1, y0)
        assert torch.equal(y1, _attn_ref(a, x, shift, scale, residual, gate))

        other = _self_attention(C, 2, sp, torch.float32, seed=7)
        a.load_state_dict(other.state_dict())
        y2 = a.forward_adaln(x, shift, scale, residual, gate)
        a.current_timestep = 0
        assert not torch.equal(y2, y1)
        assert torch.equal(y2, other.forward_adaln(x, shift, scale, residual, gate))
        assert torch.equal(y2, _attn_ref(a, x, shift, scale, residual, gate))
    assert all(p is q for p, q in zip([a.to_q.weight, a.to_k.weight, a.to_v.weight], params))


# ---------------------------------------------------------------------------------------------- QuantizedPixArtBlock
def _timestep(B, C, dt, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 6 * C, generator=g) * 0.5).cuda().to(dt)


def _text(B, S, C, dt, seed):
    """Encoder states (B, S, C) and diffusers' additive mask (1 - keep) * -10000 as (B, 1, S): batch entry b masks its
    last 7 * b tokens."""
    g = torch.Generator().manual_seed(seed)
    enc = torch.randn(B, S, C, generator=g).cuda().to(dt)
    keep = torch.ones(B, S)
    for b in range(B):
        keep[b, S - 7 * b:] = 0.0
    return enc, ((1 - keep) * -10000.0).unsqueeze(1).cuda()


def _block_ref(blk, h, enc, mask, timestep):
    """BasicTransformerBlock.forward (ada_norm_single) layer by layer on the wrapped block's modules."""
    B = h.shape[0]
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = (
        blk.scale_shift_table[None] + timestep.reshape(B, 6, -1)).chunk(6, dim=1)
    h = gate_msa * blk.attn1(blk.norm1(h) * (1 + scale_msa) + shift_msa) + h
    h = blk.attn2(h, enc, attention_mask=mask) + h
    ff = blk.ff
    return gate_mlp * ff.fc2(ff.act(ff.fc1(blk.norm2(h) * (1 + scale_mlp) + shift_mlp))) + h


def _pixart_block(dt, sp, C=128, heads=2, **kw):
    from mx_quantization_b200.modules import QuantizedPixArtBlock
    torch.manual_seed(5)
    return QuantizedPixArtBlock(_PixArtBlock(C, heads, sp, **kw), mx_specs=sp).cuda().to(dt).eval()


@pytest.mark.gpu
def test_quantized_pixart_block_equals_reference(monkeypatch):
    """fp32, S = 120 text tokens with a mask: step 0 runs attn1 dense and attn2 on the true scores (exclude_timesteps),
    step 1 both top-k.  The block makes two mx_linear calls for attn1 (q/k/v, to_out), four for attn2 and one mx_mlp
    call with the adaLN arguments."""
    from mx_quantization_b200 import ops
    sp = mx_specs(32, True)
    C, B, T, S = 128, 3, 100, 120
    blk = _pixart_block(torch.float32, sp, C, exclude_self={0}, exclude_cross={0})
    h = torch.randn(B, T, C, device="cuda")
    t = _timestep(B, C, torch.float32, seed=3)
    enc, mask = _text(B, S, C, torch.float32, seed=4)
    calls = []
    for name in ("mx_linear", "mx_mlp"):
        real = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _n=name, _r=real, **k: calls.append(
            (_n, sorted(x for x in k if x in ("shift", "scale", "residual", "gate")))) or _r(*a, **k))
    for step in range(2):
        with torch.no_grad():
            calls.clear()
            got = blk(h, encoder_hidden_states=enc, encoder_attention_mask=mask, timestep=t)
            assert calls == [("mx_linear", ["scale", "shift"]), ("mx_linear", ["gate", "residual"])] + \
                [("mx_linear", [])] * 4 + [("mx_mlp", ["gate", "residual", "scale", "shift"])]
            assert blk.attn1.current_timestep == blk.attn2.current_timestep == step + 1
            blk.attn1.current_timestep = blk.attn2.current_timestep = step
            want = _block_ref(blk, h, enc, mask, t)
        assert got.dtype == torch.float32 and got.shape == h.shape
        assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_quantized_pixart_block_16bit(dt):
    """16-bit blocks on top-k steps equal the expression; on a cross-attention exclude_timesteps step (ranking on the
    true scores, an fp32-only mode) the block raises the core's ValueError rather than widening."""
    sp = mx_specs(32, True)
    C, B, T, S = 128, 2, 256, 120
    blk = _pixart_block(dt, sp, C, exclude_cross={1})
    h = torch.randn(B, T, C, device="cuda").to(dt)
    t = _timestep(B, C, dt, seed=6)
    enc, mask = _text(B, S, C, dt, seed=7)
    with torch.no_grad():
        got = blk(h, encoder_hidden_states=enc, encoder_attention_mask=mask, timestep=t)
        blk.attn1.current_timestep = blk.attn2.current_timestep = 0
        assert torch.equal(got, _block_ref(blk, h, enc, mask, t))
        with pytest.raises(ValueError, match="ex_pred"):
            blk(h, encoder_hidden_states=enc, encoder_attention_mask=mask, timestep=t)


@pytest.mark.gpu
def test_quantized_pixart_block_dropout_takes_the_expression(monkeypatch):
    from mx_quantization_b200 import ops
    sp = mx_specs(32, True)
    C, B, T, S = 128, 2, 64, 120
    blk = _pixart_block(torch.float32, sp, C, ff=_FeedForward(C, dropout=0.5)).train()
    blk.attn1.to_out[1].p = 0.5
    assert blk.ff.drop_hidden.p == 0.5
    kwargs = []
    for name in ("mx_linear", "mx_mlp"):
        real = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _n=name, _r=real, **k: kwargs.append((_n, sorted(k))) or _r(*a, **k))
    enc, mask = _text(B, S, C, torch.float32, seed=8)
    with torch.no_grad():
        y = blk(torch.randn(B, T, C, device="cuda"), encoder_hidden_states=enc, encoder_attention_mask=mask,
                timestep=_timestep(B, C, torch.float32, seed=9))
    assert y.shape == (B, T, C) and kwargs
    assert not any(k in ks for _, ks in kwargs for k in ("shift", "scale", "residual", "gate"))
    assert all(n == "mx_linear" for n, _ in kwargs)     # the hidden dropout sits between GELU and fc2: no fused MLP


# ---------------------------------------------------------------------------------------------- structure (no GPU)
def test_quantized_mlp_from_feed_forward():
    from mx_quantization_b200.modules import MxLinear, QuantizedMlp
    sp = mx_specs(32, True)
    for approximate in ("none", "tanh"):
        ff = _FeedForward(64, approximate=approximate, dropout=0.25, final_dropout=True)
        m = QuantizedMlp(ff, mx_specs=sp)
        assert isinstance(m.fc1, MxLinear) and isinstance(m.fc2, MxLinear)
        assert m.fc1.weight is ff.net[0].proj.weight and m.fc1.bias is ff.net[0].proj.bias
        assert m.fc2.weight is ff.net[2].weight and m.fc2.bias is ff.net[2].bias
        assert type(m.act) is nn.GELU and m.act.approximate == approximate
        assert m.drop_hidden.p == 0.25 and m.drop.p == 0.25
        assert m.eval()._fused() and not m.train()._fused()
    m = QuantizedMlp(_FeedForward(64), mx_specs=sp)
    assert m.drop_hidden.p == 0.0 and m.drop.p == 0.0 and m.train()._fused()


def test_quantized_mlp_rejects_other_feed_forwards():
    from mx_quantization_b200.modules import QuantizedMlp
    sp = mx_specs(32, True)
    with pytest.raises(TypeError, match="net\\[0\\]"):
        QuantizedMlp(_FeedForward(64, act=_GEGLU(64, 256)), mx_specs=sp)
    gelu = _GELU(64, 256, approximate="erf")
    with pytest.raises(TypeError, match="net\\[0\\]"):
        QuantizedMlp(_FeedForward(64, act=gelu), mx_specs=sp)
    ff = _FeedForward(64)
    ff.net[1] = nn.Identity()
    with pytest.raises(TypeError, match="Dropout"):
        QuantizedMlp(ff, mx_specs=sp)


def test_quantized_pixart_block_structure():
    from mx_quantization_b200.modules import MXCrossAttention, MXSelfAttention, QuantizedMlp, QuantizedPixArtBlock
    sp = mx_specs(32, True)
    src = _PixArtBlock(64, 2, sp)
    blk = QuantizedPixArtBlock(src, mx_specs=sp)
    assert isinstance(blk.ff, QuantizedMlp) and blk.ff.act.approximate == "tanh"
    assert blk.attn1 is src.attn1 and blk.attn2 is src.attn2 and blk.norm1 is src.norm1 and blk.norm2 is src.norm2
    assert blk.scale_shift_table is src.scale_shift_table
    assert QuantizedPixArtBlock(blk, mx_specs=sp).ff is blk.ff
    src.attn2 = None
    assert QuantizedPixArtBlock(src, mx_specs=sp).attn2 is None
    with pytest.raises(ValueError, match="attention_mask"):
        blk(torch.zeros(1, 4, 64), attention_mask=torch.zeros(1, 1, 4), timestep=torch.zeros(1, 6 * 64))
    with pytest.raises(TypeError, match="no adaLN form"):
        MXCrossAttention(64, 2).forward_adaln(None, None, None, None, None)

    for attr, bad, err in (("attn1", nn.MultiheadAttention(64, 2), TypeError),
                           ("attn1", MXCrossAttention(64, 2).set_config(mx_quant=True, mx_specs=sp), TypeError),
                           ("attn1", MXSelfAttention(64, 2), RuntimeError),            # set_config not called
                           ("attn2", nn.MultiheadAttention(64, 2), TypeError),
                           ("ff", nn.Linear(64, 64), TypeError),
                           ("ff", _FeedForward(64, act=_GEGLU(64, 256)), TypeError)):
        b = _PixArtBlock(64, 2, sp)
        setattr(b, attr, bad)
        with pytest.raises(err):
            QuantizedPixArtBlock(b, mx_specs=sp)
