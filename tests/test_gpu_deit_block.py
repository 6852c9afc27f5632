"""``QuantizedDeiTBlock`` (DeiT's pre-norm block with norm1 / norm2 in the qkv / fc1 quantizers and both residual adds
in the proj / fc2 stores) against the timm block's forward on the same modules with torch.equal; the fallbacks and
rejections; and the DiT and PixArt blocks routing their norms into the quantizer and PixArt's cross-attention residual
into to_out's store."""
import pytest
import torch
import torch.nn as nn

from tests.helpers import mx_specs

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["fp32", "bf16", "fp16"]


class _TimmAttn(nn.Module):             # the attributes QuantizedAttention takes from timm's Attention
    def __init__(self, dim, heads):
        super().__init__()
        self.num_heads, self.scale = heads, (dim // heads) ** -0.5
        self.qkv, self.proj, self.proj_drop = nn.Linear(dim, 3 * dim), nn.Linear(dim, dim), nn.Dropout(0.0)


class _TimmMlp(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), nn.GELU(), nn.Linear(4 * dim, dim), nn.Dropout(0.0)

    def forward(self, x):
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


class _DropPath(nn.Module):             # timm's DropPath: per-sample stochastic depth while training
    def __init__(self, drop_prob):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.dim() - 1)).bernoulli_(keep)
        return x * mask / keep


class _TimmBlock(nn.Module):            # timm 0.4.12 vision_transformer.Block
    def __init__(self, dim, heads, drop_path=0.0, norm=nn.LayerNorm):
        super().__init__()
        self.norm1, self.attn = norm(dim), _TimmAttn(dim, heads)
        self.drop_path = _DropPath(drop_path) if drop_path > 0 else nn.Identity()
        self.norm2, self.mlp = norm(dim), _TimmMlp(dim)

    def forward(self, x):
        x = x + self.drop_path(self.attn(self.norm1(x)))
        return x + self.drop_path(self.mlp(self.norm2(x)))


def _randomize_norms(blk, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n in (blk.norm1, blk.norm2):
            if isinstance(n, nn.LayerNorm) and n.weight is not None:
                n.weight.copy_(1 + 0.3 * torch.randn(n.weight.shape, generator=g))
                n.bias.copy_(0.3 * torch.randn(n.bias.shape, generator=g))


def _quantized(blk, sp, **attn_kw):
    """The timm block with the shims apply_quantization_to_deit puts in (QuantizedAttention, QuantizedMlp)."""
    from mx_quantization_b200.modules import QuantizedAttention, QuantizedMlp
    kw = dict(mx_quant=True, mx_specs=sp, top_k=True, k=20)
    kw.update(attn_kw)
    blk.attn = QuantizedAttention(blk.attn, **kw)
    blk.mlp = QuantizedMlp(blk.mlp, mx_specs=sp)
    return blk


def _spy(monkeypatch, names=("mx_linear", "mx_mlp")):
    from mx_quantization_b200 import ops
    calls = []
    for name in names:
        real = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _n=name, _r=real, **k: calls.append(
            (_n, sorted(x for x in k if k[x] is not None and x in ("ln_eps", "ln_weight", "add", "shift", "residual"))))
            or _r(*a, **k))
    return calls


# ---------------------------------------------------------------------------------------------- block == timm block
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("T", [197, 50])
def test_deit_block_equals_timm_block(dt, bfloat, T, monkeypatch):
    """C = 192 (3 heads of 64), random LayerNorm affine parameters: two mx_linear calls (qkv with the norm, proj with
    add) and one mx_mlp call (the norm and add)."""
    from mx_quantization_b200.modules import QuantizedDeiTBlock
    torch.manual_seed(T + bfloat)
    sp = mx_specs(bfloat)
    src = _quantized(_TimmBlock(192, 3), sp).cuda().to(dt).eval()
    _randomize_norms(src, seed=T)
    keys = sorted(src.state_dict())
    blk = QuantizedDeiTBlock(src, mx_specs=sp)
    assert sorted(blk.state_dict()) == keys
    x = (1 + torch.randn(2, T, 192, device="cuda")).to(dt)
    calls = _spy(monkeypatch)
    with torch.no_grad():
        got = blk(x)
        assert calls == [("mx_linear", ["ln_eps", "ln_weight"]), ("mx_linear", ["add"]),
                         ("mx_mlp", ["add", "ln_eps", "ln_weight"])]
        want = src(x)
    assert got.dtype == dt and got.shape == x.shape
    assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["dense", "partial_Q", "anal"])
def test_deit_block_variants(variant, capsys):
    """A dense block (top_k=False), an exclude_block_type block (pred_mode 'partial_Q') and anal=True behave as the
    attention shim's forward: same output, same printed chosen-k, current_timestep advanced once per call."""
    from mx_quantization_b200.modules import QuantizedDeiTBlock
    torch.manual_seed(5)
    sp = mx_specs(32)
    kw = {"dense": dict(top_k=False), "partial_Q": dict(pred_mode="partial_Q"), "anal": dict(anal=True)}[variant]
    src = _quantized(_TimmBlock(128, 2), sp, **kw).cuda().eval()
    _randomize_norms(src, seed=6)
    blk = QuantizedDeiTBlock(src, mx_specs=sp)
    x = torch.randn(2, 197, 128, device="cuda")
    with torch.no_grad():
        got = blk(x)
        out_fused = capsys.readouterr().out
        want = src(x)
        out_ref = capsys.readouterr().out
    assert torch.equal(got, want)
    assert out_fused == out_ref and (("Average chosen k" in out_fused) == (variant == "anal"))
    assert src.attn.current_timestep == 2


@pytest.mark.gpu
def test_deit_base_model_wrapped_equals_unwrapped():
    """12 blocks of DeiT-base (dim 768, 12 heads) after apply_quantization_to_deit (block 11 dense): wrapping every
    block in QuantizedDeiTBlock leaves the model's output bit-identical."""
    from mx_quantization_b200.modules import QuantizedDeiTBlock, apply_quantization_to_deit
    torch.manual_seed(7)
    model = nn.Module()
    model.blocks = nn.ModuleList([_TimmBlock(768, 12) for _ in range(12)])
    for i, b in enumerate(model.blocks):
        _randomize_norms(b, seed=i)
    cfg = {"blocks": list(range(12)), "components": ["attn", "ffn"], "mx_specs": mx_specs(32)}
    apply_quantization_to_deit(model, cfg, top_k=True, k=30)
    model.cuda().eval()
    wrapped = nn.ModuleList([QuantizedDeiTBlock(b) for b in model.blocks])
    x = torch.randn(4, 197, 768, device="cuda")
    with torch.no_grad():
        want, got = x, x
        for b in model.blocks:
            want = b(want)
        for b in wrapped:
            got = b(got)
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_deit_block_fallbacks(monkeypatch):
    """Training with an active drop_path runs the expression (no norm or add in the kernels); a norm that does not
    qualify (a LayerNorm subclass, a weight-only LayerNorm) runs in torch and the result is still the block's."""
    from mx_quantization_b200.modules import QuantizedDeiTBlock
    torch.manual_seed(8)
    sp = mx_specs(32)
    blk = QuantizedDeiTBlock(_quantized(_TimmBlock(128, 2, drop_path=0.2), sp).cuda(), mx_specs=sp).train()
    calls = _spy(monkeypatch)
    with torch.no_grad():
        y = blk(torch.randn(2, 64, 128, device="cuda"))
    assert y.shape == (2, 64, 128) and calls and all(ks == [] for _, ks in calls)

    class _SubLN(nn.LayerNorm):
        pass

    for norm in (_SubLN, lambda d: nn.LayerNorm(d, bias=False)):
        src = _quantized(_TimmBlock(128, 2, norm=norm), sp).cuda().eval()
        blk = QuantizedDeiTBlock(src, mx_specs=sp)
        x = torch.randn(2, 64, 128, device="cuda")
        calls.clear()
        with torch.no_grad():
            got = blk(x)
            assert calls == [("mx_linear", []), ("mx_linear", ["add"]), ("mx_mlp", ["add"])]
            assert torch.equal(got, src(x))


@pytest.mark.gpu
def test_deit_block_refuses_grad_mode():
    from mx_quantization_b200.modules import QuantizedDeiTBlock
    sp = mx_specs(32)
    blk = QuantizedDeiTBlock(_quantized(_TimmBlock(128, 2), sp).cuda().eval(), mx_specs=sp)
    with pytest.raises(RuntimeError, match="inference"):
        blk(torch.randn(2, 64, 128, device="cuda"))


# ---------------------------------------------------------------------------------------------- DiT / PixArt routing
@pytest.mark.gpu
def test_dit_block_routes_its_norms_into_the_quantizer(monkeypatch):
    """DiT's nn.LayerNorm(C, elementwise_affine=False, eps=1e-6) goes into the qkv and fc1 quantizers (ln_eps 1e-6); a
    LayerNorm subclass runs in torch; both equal the block expression."""
    from tests.test_gpu_dit_block import _DiTBlock, _block_ref
    from mx_quantization_b200.modules import QuantizedDiTBlock
    torch.manual_seed(9)
    sp = mx_specs(16)

    class _SubLN(nn.LayerNorm):
        pass

    for sub in (False, True):
        src = _DiTBlock(128, 2, sp, nn.GELU("tanh"), k=20)
        if sub:
            src.norm1, src.norm2 = _SubLN(128, elementwise_affine=False, eps=1e-6), _SubLN(128, elementwise_affine=False,
                                                                                             eps=1e-6)
        blk = QuantizedDiTBlock(src, mx_specs=sp).cuda().eval()
        with torch.no_grad():
            blk.adaLN_modulation[1].weight.normal_(0, 0.1)
        x, c = torch.randn(2, 100, 128, device="cuda"), torch.randn(2, 128, device="cuda")
        calls = _spy(monkeypatch)
        with torch.no_grad():
            got = blk(x, c)
            ln = [] if sub else ["ln_eps"]
            assert calls == [("mx_linear", sorted(ln + ["shift"])), ("mx_linear", ["residual"]),
                             ("mx_mlp", sorted(ln + ["residual", "shift"]))]
            blk.attn.current_timestep = 0
            want = _block_ref(blk, x, c)
        assert torch.equal(got, want)
        monkeypatch.undo()


@pytest.mark.gpu
def test_pixart_block_routes_norms_and_cross_attention_add(monkeypatch):
    from tests.test_gpu_pixart_block import _block_ref, _pixart_block, _text, _timestep
    sp = mx_specs(32, True)
    C, B, T, S = 128, 2, 100, 120
    blk = _pixart_block(torch.float32, sp, C)
    h = torch.randn(B, T, C, device="cuda")
    t = _timestep(B, C, torch.float32, seed=10)
    enc, mask = _text(B, S, C, torch.float32, seed=11)
    calls = _spy(monkeypatch)
    with torch.no_grad():
        got = blk(h, encoder_hidden_states=enc, encoder_attention_mask=mask, timestep=t)
        assert calls == [("mx_linear", ["ln_eps", "shift"]), ("mx_linear", ["residual"])] + [("mx_linear", [])] * 3 + \
            [("mx_linear", ["add"]), ("mx_mlp", ["ln_eps", "residual", "shift"])]
        blk.attn1.current_timestep = blk.attn2.current_timestep = 0
        want = _block_ref(blk, h, enc, mask, t)
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------- structure (no GPU)
def test_deit_block_structure_and_rejections():
    from mx_quantization_b200.modules import QuantizedAttention, QuantizedDeiTBlock, QuantizedMlp, _fused_norm
    sp = mx_specs(32)
    src = _quantized(_TimmBlock(64, 2), sp)
    keys = sorted(src.state_dict())
    blk = QuantizedDeiTBlock(src, mx_specs=sp)
    assert isinstance(blk.attn, QuantizedAttention) and isinstance(blk.mlp, QuantizedMlp)
    assert blk.norm1 is src.norm1 and blk.norm2 is src.norm2 and blk.mlp is src.mlp
    assert sorted(blk.state_dict()) == keys
    # a raw timm Mlp is wrapped
    src2 = _TimmBlock(64, 2)
    src2.attn = QuantizedAttention(src2.attn, mx_quant=True, mx_specs=sp, top_k=True, k=20)
    assert isinstance(QuantizedDeiTBlock(src2, mx_specs=sp).mlp, QuantizedMlp)
    with pytest.raises(TypeError, match="QuantizedAttention"):
        QuantizedDeiTBlock(_TimmBlock(64, 2), mx_specs=sp)
    src.ls1 = nn.Linear(64, 64)
    with pytest.raises(TypeError, match="ls1"):
        QuantizedDeiTBlock(src, mx_specs=sp)
    src.ls1, src.ls2 = nn.Identity(), nn.Identity()
    QuantizedDeiTBlock(src, mx_specs=sp)
    # which norms the quantizer takes
    x = torch.zeros(2, 3, 64)

    class _SubLN(nn.LayerNorm):
        pass

    ln = nn.LayerNorm(64, eps=1e-6)
    kw = _fused_norm(ln, x)
    assert kw["ln_eps"] == 1e-6 and kw["ln_weight"] is not None and kw["ln_bias"] is not None
    assert _fused_norm(nn.LayerNorm(64, elementwise_affine=False), x) == {"ln_eps": 1e-5}
    assert _fused_norm(None, x) == {}
    for other in (_SubLN(64), nn.LayerNorm(64, bias=False), nn.LayerNorm(32), nn.LayerNorm(64).half(), nn.Identity(),
                  nn.GroupNorm(1, 64)):
        assert _fused_norm(other, x) is None
