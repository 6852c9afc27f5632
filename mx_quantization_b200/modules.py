"""Attention-module integration hooks.

The three attention modules the reference patches all run the same sequence between their qkv
projection and their output projection (SURVEY.md 3a):
    workloads/deit/scripts/main.py:85-157                       QuantizedAttention.forward
    workloads/DiT/models.py:154-230                             Attention.forward
    workloads/PixArt/models/MX_transformer_block.py:624-717     MXSelfAttention.forward
``PrunedAttentionCore`` is that sequence (lines 101-152 of the DeiT file) as one call into
libmxprune; the three shims keep the reference constructors' / ``set_config`` argument names so a
maintainer can swap the body of ``forward`` (INTEGRATION.md shows the patch).  The qkv / output
projections are ``MxLinear`` (the reference's ``mx.Linear`` forward on the tcgen05 GEMM, SURVEY 8f2) when the shim is
built with ``mx_quant=True``, else whatever the host model uses.

Implemented: mx_quant && top_k && approx/ex_pred with pred_mode "ex_pred" (the pruned hot path),
"partial_Q", "partial_K", "MXINT4", "two_step_leading_ones", "true_ex" or "ELSA" (with the caller's orthogonal matrix);
mx_quant && top_k && !approx (top-k of the true scores); and mx_quant && !top_k (dense MXINT8 attention, what the
reference runs in the last block of each model - same kernels with every key kept).  mx_quant=False (the reference's
unquantized torch path) raises - no silent fallback.

``QuantizedDiTBlock`` wraps a whole DiT block (workloads/DiT/models.py:271-297): its adaLN modulations and gated residuals
run inside the MX Linear kernels of the Attention shim and of QuantizedMlp.  ``QuantizedPixArtBlock`` does the same for
PixArt-alpha's adaLN-single block, with q, k and v from one projection GEMM.
"""
from typing import Optional

import torch
import torch.nn as nn

from . import ops
from .specs import resolve_linear_specs, resolve_specs


class PrunedAttentionCore(nn.Module):
    """q, k, v (B,H,N,hd) views -> x (B,N,H*hd), ready for the output projection, in q's dtype.

    q, k, v: float32, or all bfloat16 or all float16 (the 16-bit scope of ops.pruned_attention: the exponent-sign
    predictor, top-k or dense, head_dim a multiple of 8 in [32, 128]; other pred_modes, ELSA and an "exact" per-call
    override raise ValueError rather than widen).  A 16-bit x is the fp32 result rounded to nearest even."""

    def __init__(self, mx_specs, k: int, scale: Optional[float] = None, pred_mode: str = "ex_pred",
                 orthogonal_matrix: Optional[torch.Tensor] = None):
        super().__init__()
        resolve_specs(mx_specs)
        self.mx_specs = mx_specs
        self.k = int(k)
        self.scale = scale
        self.pred_mode = pred_mode
        if pred_mode == "ELSA" and orthogonal_matrix is None:
            raise ValueError("pred_mode='ELSA' needs orthogonal_matrix (workloads/deit/scripts/main.py:119-121)")
        self.orthogonal_matrix = orthogonal_matrix
        # --anal (main.py:134-136): "Average chosen k" = funcs/analysis.py total_chosen_k, from the kept-key bitmask;
        # the per-timestep diff_idx text dumps (main.py:137-143) are not produced
        self.anal = False
        self.avg_chosen_k = None

    def forward(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                key_bias: Optional[torch.Tensor] = None, dense: bool = False,
                pred_mode: Optional[str] = None) -> torch.Tensor:
        """dense / pred_mode: per-call overrides for the reference's exclude_timesteps steps."""
        B, H, N, hd = q.shape
        buf = torch.empty((B, N, H, hd), dtype=q.dtype, device=q.device)
        # write straight into (B,N,H,hd): the reference's x.transpose(1,2).reshape(B,N,C) is free
        # k <= 0: dense MXINT8 attention (the reference's top_k=False blocks) = every key kept
        top_k = self.k if (self.k > 0 and not dense) else k.shape[2]
        mode = pred_mode or self.pred_mode
        res = ops.pruned_attention(q, k, v, self.mx_specs, top_k, scale=self.scale, out=buf.permute(0, 2, 1, 3),
                                   key_bias=key_bias, pred_mode=mode, return_mask=self.anal,
                                   orthogonal_matrix=self.orthogonal_matrix if mode == "ELSA" else None)
        if self.anal:
            from .analysis import coverage_rate
            self.avg_chosen_k = coverage_rate(res[1])
            print(f"Average chosen k: {self.avg_chosen_k:.3f}")         # as main.py:136
        return buf.reshape(B, N, H * hd)


def _require_hot_path(mx_quant, top_k, approx, pred_mode, where) -> str:
    """Validate the reference's flag combination; returns the ops.PRED_MODES key that ranks the keys
    (workloads/deit/scripts/main.py:104-131: approx_flag picks the predictor, else top-k of the true scores)."""
    if mx_quant and not top_k:
        return "ex_pred"    # dense MXINT8 attention (deit main.py:282-296: the last block runs top_k=False)
    if not mx_quant:
        raise NotImplementedError(f"{where}: mx_quant=False (the fp32 attention of the host model) is not on the "
                                  "B200 path and there is no fallback")
    if not approx:
        return "exact"
    if pred_mode not in ("ex_pred", "partial_Q", "partial_K", "MXINT4", "two_step_leading_ones", "true_ex", "ELSA"):
        raise NotImplementedError(
            f"{where}: pred_mode={pred_mode!r} is not built (built: 'ex_pred', 'partial_Q', 'partial_K', 'MXINT4', "
            "'two_step_leading_ones', 'true_ex', 'ELSA' and approx=False) "
            "(SURVEY.md 8f3) and there is no fallback")
    return pred_mode


def to_mx_linear(lin: nn.Linear, mx_specs) -> "MxLinear":
    """nn.Linear -> MxLinear sharing the parameters (what apply_quantization_to_deit /
    MXBasicTransformerBlock.set_config do with mx.Linear: deit main.py:231-318,
    MX_transformer_block.py:344-362)."""
    if isinstance(lin, MxLinear):
        return lin
    m = MxLinear(lin.in_features, lin.out_features, bias=lin.bias is not None, mx_specs=mx_specs)
    m.weight = lin.weight
    if lin.bias is not None:
        m.bias = lin.bias
    return m


class QuantizedAttention(nn.Module):
    """DeiT shim - constructor mirrors workloads/deit/scripts/main.py:42."""

    def __init__(self, orig_attn, mx_quant=False, mx_specs=None, top_k=True, k=20, approx_flag=True,
                 pred_mode="ex_pred", anal=False, file_name_dict=None, block_idx=None, orthogonal_matrix=None):
        super().__init__()
        mode = _require_hot_path(mx_quant, top_k, approx_flag, pred_mode, "QuantizedAttention")
        self.num_heads = orig_attn.num_heads
        self.scale = orig_attn.scale
        # the reference swaps the projections for mx.Linear as well (main.py:262-281)
        self.qkv, self.proj = to_mx_linear(orig_attn.qkv, mx_specs), to_mx_linear(orig_attn.proj, mx_specs)
        self.proj_drop = getattr(orig_attn, "proj_drop", nn.Identity())
        self.block_idx = block_idx
        self.current_timestep = 0
        self.core = PrunedAttentionCore(mx_specs, k if top_k else 0, scale=self.scale, pred_mode=mode,
                                        orthogonal_matrix=orthogonal_matrix)
        self.core.anal = bool(anal) and bool(top_k)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        x = self.core(qkv[0], qkv[1], qkv[2])         # strided views of the fused buffer, no copies
        x = self.proj_drop(self.proj(x))
        self.current_timestep += 1
        return x


def _feed_forward_layers(net):
    """diffusers' FeedForward.net (PixArt's feed-forward) -> (fc1, act, hidden dropout p, fc2, output dropout p):
    net[0] a GELU module that owns fc1 as ``.proj`` and applies ``F.gelu(approximate=.approximate)``, net[1] the Dropout
    between the activation and fc2, net[2] fc2, and an optional trailing Dropout.  Recognised by structure (diffusers is
    not a dependency); anything else raises TypeError."""
    act = net[0] if len(net) else None
    if not isinstance(getattr(act, "proj", None), nn.Linear) or getattr(act, "approximate", None) not in ("none", "tanh"):
        raise TypeError(f"QuantizedMlp: net[0] must be a GELU module with a Linear .proj and .approximate 'none' or "
                        f"'tanh' (diffusers' FeedForward), got {type(act).__name__}")
    if (len(net) not in (3, 4) or not isinstance(net[1], nn.Dropout) or not isinstance(net[2], nn.Linear)
            or (len(net) == 4 and not isinstance(net[3], nn.Dropout))):
        raise TypeError("QuantizedMlp: a FeedForward's net must be [GELU, Dropout, Linear] with an optional trailing "
                        f"Dropout, got [{', '.join(type(m).__name__ for m in net)}]")
    return act.proj, nn.GELU(approximate=act.approximate), net[1].p, net[2], net[3].p if len(net) == 4 else 0.0


class QuantizedMlp(nn.Module):
    """DeiT MLP with MX Linear layers - mirrors workloads/deit/scripts/main.py:159-196 (fc1 -> act -> fc2 -> drop;
    the activation stays the host model's own module, as in the reference).

    ``orig_mlp`` may also be diffusers' ``FeedForward`` (PixArt: ``net = [GELU(proj=fc1), Dropout, fc2, (Dropout)]``,
    recognised by structure): fc1 is ``net[0].proj``, the activation ``nn.GELU(approximate=net[0].approximate)`` and fc2
    ``net[2]``; its dropout between the activation and fc2 is ``drop_hidden``.

    When the activation is exactly ``torch.nn.GELU`` (either approximation) and fc1 / fc2 share one MX configuration, the
    forward is one ops.mx_mlp call on the layers' cached weight operands: bit for bit the layer-by-layer composition, with
    the hidden activation never written in a float type.  Any other activation (a subclass or another GELU class too),
    and an active ``drop_hidden`` while training, runs the composition."""

    def __init__(self, orig_mlp, mx_specs=None):
        super().__init__()
        self.mx_specs = mx_specs
        net = getattr(orig_mlp, "net", None)
        if net is not None:
            fc1, self.act, p_hidden, fc2, p = _feed_forward_layers(net)
        else:
            fc1, self.act, fc2 = orig_mlp.fc1, orig_mlp.act, orig_mlp.fc2
            p_hidden, p = 0.0, getattr(getattr(orig_mlp, "drop", None), "p", 0.0)
        self.drop_hidden = nn.Dropout(p_hidden)
        self.drop = nn.Dropout(p)
        self.fc1, self.fc2 = to_mx_linear(fc1, mx_specs), to_mx_linear(fc2, mx_specs)

    def _fused(self) -> bool:
        return (type(self.act) is nn.GELU and not (self.training and self.drop_hidden.p > 0)
                and resolve_linear_specs(self.fc1.mx_specs) == resolve_linear_specs(self.fc2.mx_specs))

    def _mx_mlp(self, x, **adaln):
        self.fc1._check_inference(x.requires_grad)
        self.fc2._check_inference(False)
        b1 = None if self.fc1.bias is None else self.fc1.bias.detach()
        b2 = None if self.fc2.bias is None else self.fc2.bias.detach()
        return ops.mx_mlp(x, self.fc1._operand(), b1, self.fc2._operand(), b2, self.fc1.mx_specs,
                          act="gelu_tanh" if self.act.approximate == "tanh" else "gelu",
                          hidden_features=self.fc1.out_features, out_features=self.fc2.out_features, **adaln)

    def forward(self, x):
        if self._fused():
            return self.drop(self._mx_mlp(x))
        return self.drop(self.fc2(self.drop_hidden(self.act(self.fc1(x)))))

    def forward_adaln(self, x, shift, scale, residual, gate):
        """The MLP half of DiT's DiTBlock.forward (workloads/DiT/models.py:297) on an already-normalized x (B, T, C):
        ``residual + gate.unsqueeze(1) * self(modulate(x, shift, scale))``, modulate(x, shift, scale) =
        ``x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)`` (models.py:101-102).  On the fused route (that of forward,
        while no dropout is active) it is one ops.mx_mlp call whose quantizer applies the modulation and whose fc2 store
        applies the gated residual, bit for bit the expression; otherwise the expression runs as written."""
        if self._fused() and not (self.training and self.drop.p > 0):
            return self._mx_mlp(x, shift=shift, scale=scale, residual=residual, gate=gate)
        return residual + gate.unsqueeze(1) * self(x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1))


def apply_quantization_to_deit(model, config, mx_quant=True, top_k=True, k=20, approx_flag=True, pred_mode="ex_pred",
                               anal=False, file_name_dict=None, exclude_blocks=(), exclude_block_type="ex_pred",
                               orthogonal_matrix=None, dense_blocks=(11,)):
    """Swap the attention / MLP modules of a timm-style DeiT (``model.blocks[i].attn`` / ``.mlp``) for the shims, with
    the reference's block policy (workloads/deit/scripts/main.py:231-318): the blocks in ``dense_blocks`` - index 11, as
    the reference hard-codes it (:266,:281,:296) - run dense MXINT8 attention (top_k=False), blocks in
    ``exclude_blocks`` use ``exclude_block_type`` as their pred_mode, every other listed block uses ``pred_mode``."""
    block_indices = config.get('blocks', [])
    components = config.get('components', ['attn', 'ffn'])
    mx_specs = config.get('mx_specs')
    if mx_specs is None:
        raise ValueError("config['mx_specs'] is required (the reference's default dict lacks keys this path validates)")
    dense_blocks = set(dense_blocks)
    for idx in block_indices:
        if idx >= len(model.blocks):
            continue
        block = model.blocks[idx]
        if 'attn' in components:
            dense, excluded = idx in dense_blocks, idx in exclude_blocks
            block.attn = QuantizedAttention(
                orig_attn=block.attn, mx_quant=mx_quant, mx_specs=mx_specs, top_k=top_k and not dense, k=k,
                approx_flag=approx_flag, pred_mode=exclude_block_type if (dense or excluded) else pred_mode,
                anal=anal, file_name_dict=file_name_dict, block_idx=idx, orthogonal_matrix=orthogonal_matrix)
        if 'ffn' in components:
            block.mlp = QuantizedMlp(orig_mlp=block.mlp, mx_specs=mx_specs)
    return model


class Attention(nn.Module):
    """DiT shim - constructor mirrors workloads/DiT/models.py:105-126."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_norm=False, proj_bias=True, attn_drop=0.,
                 proj_drop=0., norm_layer=nn.LayerNorm, mx_quant=False, mx_specs=None, top_k=False, k=20,
                 ex_pred=False, pred_mode="ex_pred", anal=False, file_name_dict=None, block_idx=None,
                 exclude_timesteps=None, orthogonal_matrix=None):
        super().__init__()
        assert dim % num_heads == 0, 'dim should be divisible by num_heads'
        mode = _require_hot_path(mx_quant, top_k, ex_pred, pred_mode, "Attention")
        # steps listed here run dense attention (models.py:172: `top_k and current_timestep not in exclude_timesteps`)
        self.exclude_timesteps = set(exclude_timesteps or ())
        self.num_heads, self.head_dim = num_heads, dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = MxLinear(dim, dim * 3, bias=qkv_bias, mx_specs=mx_specs)        # models.py:129 (mx Linear)
        self.q_norm = norm_layer(self.head_dim) if qk_norm else nn.Identity()
        self.k_norm = norm_layer(self.head_dim) if qk_norm else nn.Identity()
        self.proj = MxLinear(dim, dim, bias=proj_bias, mx_specs=mx_specs)
        self.proj_drop = nn.Dropout(proj_drop)
        self.block_idx = block_idx
        self.current_timestep = 0
        self.core = PrunedAttentionCore(mx_specs, k if top_k else 0, scale=self.scale, pred_mode=mode,
                                        orthogonal_matrix=orthogonal_matrix)
        self.core.anal = bool(anal) and bool(top_k)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        q, k = self.q_norm(q), self.k_norm(k)
        x = self.core(q, k, v, dense=self.current_timestep in self.exclude_timesteps)
        x = self.proj_drop(self.proj(x))
        self.current_timestep += 1
        return x

    def forward_adaln(self, x, shift, scale, residual, gate):
        """The attention half of DiT's DiTBlock.forward (workloads/DiT/models.py:296) on an already-normalized x (B, N, C):
        ``residual + gate.unsqueeze(1) * self(x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1))``, bit for bit.  The
        qkv projection's quantizer applies the modulation as it loads x, and the output projection's store applies the
        gated residual; the core call between them is forward's (dense on exclude_timesteps steps), and
        current_timestep advances as in forward.  While proj_drop is active (training, p > 0) the expression runs as
        written."""
        if self.training and self.proj_drop.p > 0:
            return residual + gate.unsqueeze(1) * self(x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1))
        B, N, C = x.shape
        qkv = self.qkv.forward_adaln(x, shift=shift, scale=scale)
        q, k, v = qkv.reshape(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4).unbind(0)
        q, k = self.q_norm(q), self.k_norm(k)
        x = self.core(q, k, v, dense=self.current_timestep in self.exclude_timesteps)
        x = self.proj.forward_adaln(x, residual=residual, gate=gate)
        self.current_timestep += 1
        return x


class QuantizedDiTBlock(nn.Module):
    """DiT block with adaLN-Zero conditioning - mirrors workloads/DiT/models.py:271-297 (DiTBlock.forward, SURVEY.md 3c):
        shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = adaLN_modulation(c).chunk(6, dim=1)
        x = x + gate_msa.unsqueeze(1) * attn(modulate(norm1(x), shift_msa, scale_msa))
        x = x + gate_mlp.unsqueeze(1) * mlp(modulate(norm2(x), shift_mlp, scale_mlp))
    with the modulations and gated residuals inside the MX Linear kernels (Attention.forward_adaln,
    QuantizedMlp.forward_adaln): bit for bit that expression on the same modules, without its elementwise passes.

    ``orig_block``: a DiT-style block with ``norm1``, ``attn``, ``norm2``, ``mlp`` and ``adaLN_modulation``.  ``attn`` must
    be the ``Attention`` shim; ``mlp`` (timm Mlp, models.py:287) is wrapped in QuantizedMlp unless it already is one.  The
    norms (torch LayerNorm) and adaLN_modulation stay the host model's modules."""

    def __init__(self, orig_block, mx_specs=None):
        super().__init__()
        if not isinstance(orig_block.attn, Attention):
            raise TypeError(f"QuantizedDiTBlock: attn must be modules.Attention (the DiT shim), got "
                            f"{type(orig_block.attn).__name__}")
        self.norm1, self.attn, self.norm2 = orig_block.norm1, orig_block.attn, orig_block.norm2
        mlp = orig_block.mlp
        self.mlp = mlp if isinstance(mlp, QuantizedMlp) else QuantizedMlp(mlp, mx_specs=mx_specs)
        self.adaLN_modulation = orig_block.adaLN_modulation

    def forward(self, x, c):
        shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = self.adaLN_modulation(c).chunk(6, dim=1)
        x = self.attn.forward_adaln(self.norm1(x), shift_msa, scale_msa, x, gate_msa)
        return self.mlp.forward_adaln(self.norm2(x), shift_mlp, scale_mlp, x, gate_mlp)


class MXSelfAttention(nn.Module):
    """PixArt-alpha shim - mirrors workloads/PixArt/models/MX_transformer_block.py:567-717."""

    def __init__(self, dim, num_heads: int, has_bias: bool = True):
        super().__init__()
        self.dim, self.num_heads, self.head_dim, self.has_bias = dim, num_heads, dim // num_heads, has_bias
        self.to_q = nn.Linear(dim, dim, bias=has_bias)
        self.to_k = nn.Linear(dim, dim, bias=has_bias)
        self.to_v = nn.Linear(dim, dim, bias=has_bias)
        self.to_out = nn.Sequential(nn.Linear(dim, dim, bias=has_bias), nn.Dropout(p=0.0))
        self.core = None
        self.current_timestep = 0
        self._qkv_op = self._qkv_bias = self._qkv_key = None

    def set_config(self, mx_quant=False, mx_specs=None, top_k=False, k=20, ex_pred=False, exclude_timesteps=None,
                   pred_mode="ex_pred", block_idx=None, anal=False, file_name_dict=None, orthogonal_matrix=None):
        mode = _require_hot_path(mx_quant, top_k, ex_pred, pred_mode, "MXSelfAttention.set_config")
        # self-attention: listed steps run dense (MX_transformer_block.py:656); cross-attention: listed steps rank
        # on the true scores instead of the predictor's (:806, else-branch :845-848)
        self.exclude_timesteps = set(exclude_timesteps or ())
        self.block_idx = block_idx
        # the block's set_config swaps nn.Linear -> mx.Linear (MX_transformer_block.py:344-362)
        self.to_q, self.to_k, self.to_v = (to_mx_linear(m, mx_specs) for m in (self.to_q, self.to_k, self.to_v))
        self.to_out[0] = to_mx_linear(self.to_out[0], mx_specs)
        # reference: scale_factor = 1 / math.sqrt(q.size(-1)) applied as an fp32 scalar (:647-653)
        self.core = PrunedAttentionCore(mx_specs, k if top_k else 0, scale=1.0 / (self.head_dim ** 0.5),
                                        pred_mode=mode, orthogonal_matrix=orthogonal_matrix)
        self.core.anal = bool(anal) and bool(top_k)
        return self

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kwargs):
        if self.core is None:
            raise RuntimeError("MXSelfAttention.set_config(...) must be called first")
        B, N, C = hidden_states.shape
        q = self.to_q(hidden_states).view(B, N, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.to_k(hidden_states).view(B, N, self.num_heads, self.head_dim).transpose(1, 2)
        v = self.to_v(hidden_states).view(B, N, self.num_heads, self.head_dim).transpose(1, 2)
        x = self.to_out(self.core(q, k, v, dense=self.current_timestep in self.exclude_timesteps))
        self.current_timestep += 1
        return x

    def _qkv_operand(self):
        """(operand, bias) of to_q, to_k and to_v as one (3C, C) layer: ``mx_linear_prepare_weight(cat([Wq, Wk, Wv]))``
        and ``cat([bq, bk, bv])``.  Cached; rebuilt when any of the six tensors changes (data_ptr, version, device, dtype,
        as MxLinear._operand keys its own) or after any of the three layers' invalidate(), which load_state_dict calls."""
        layers = (self.to_q, self.to_k, self.to_v)
        key = tuple((m._w_gen,) + tuple((t.data_ptr(), t._version, str(t.device), t.dtype)
                                        for t in (m.weight, m.bias) if t is not None) for m in layers)
        if self._qkv_key != key:
            self._qkv_op = ops.mx_linear_prepare_weight(torch.cat([m.weight.detach() for m in layers]), self.to_q.mx_specs)
            self._qkv_bias = None if self.to_q.bias is None else torch.cat([m.bias.detach() for m in layers])
            self._qkv_key = key
        return self._qkv_op, self._qkv_bias

    def forward_adaln(self, x, shift, scale, residual, gate):
        """The self-attention half of PixArt's adaLN-single block (diffusers' BasicTransformerBlock) on the normalized
        hidden states x (B, N, C): ``residual + gate.unsqueeze(1) * self(x * (1 + scale.unsqueeze(1)) +
        shift.unsqueeze(1))``, bit for bit.  shift / scale / gate: (B, C) rows, e.g. ``.squeeze(1)`` of the block's
        (B, 1, C) chunks, read in place.

        q, k and v come from ONE mx_linear call on the concatenated (3C, C) weight, whose quantizer applies the
        modulation: the GEMM has no split-K, so every output column is reduced in the same order whichever 256-column
        tile holds it, and its bits are those of the separate projection.  The core reads q, k, v as strided views of
        the (B, N, 3C) result (dense on exclude_timesteps steps, as forward), to_out[0]'s store applies the gated
        residual, and current_timestep advances.  While to_out's dropout is active (training, p > 0), or when the three
        projections have different MX configurations, the expression runs as written."""
        if self.core is None:
            raise RuntimeError("MXSelfAttention.set_config(...) must be called first")
        layers = (self.to_q, self.to_k, self.to_v)
        if ((self.training and self.to_out[1].p > 0)
                or len({resolve_linear_specs(m.mx_specs) for m in layers}) != 1):
            return residual + gate.unsqueeze(1) * self(x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1))
        for m in layers:
            m._check_inference(x.requires_grad)
        B, N, C = x.shape
        w_op, b = self._qkv_operand()
        qkv = ops.mx_linear(x, w_op, b, self.to_q.mx_specs, out_features=3 * C, shift=shift, scale=scale)
        q, k, v = qkv.view(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4).unbind(0)
        x = self.core(q, k, v, dense=self.current_timestep in self.exclude_timesteps)
        x = self.to_out[0].forward_adaln(x, residual=residual, gate=gate)
        self.current_timestep += 1
        return x


class MXCrossAttention(MXSelfAttention):
    """PixArt-alpha cross-attention shim - mirrors workloads/PixArt/models/MX_transformer_block.py:720-859:
    keys / values come from the text encoder states (S tokens), and the additive attention_mask
    (B,1,S) is applied to the true and the predicted scores (:794-803, :821-822)."""

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, **kwargs):
        if self.core is None:
            raise RuntimeError("MXCrossAttention.set_config(...) must be called first")
        if encoder_hidden_states is None:
            raise ValueError("MXCrossAttention needs encoder_hidden_states")
        B, N, C = hidden_states.shape
        S = encoder_hidden_states.shape[1]
        q = self.to_q(hidden_states).view(B, N, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.to_k(encoder_hidden_states).reshape(B, S, self.num_heads, self.head_dim).transpose(1, 2)
        v = self.to_v(encoder_hidden_states).reshape(B, S, self.num_heads, self.head_dim).transpose(1, 2)
        if attention_mask is not None and attention_mask.dtype == torch.bool:
            raise NotImplementedError("boolean masks (-inf bias) are not on the path; pass the additive fp32 mask")
        bias = None if attention_mask is None else attention_mask.to(torch.float32).reshape(B, S)
        excluded = self.current_timestep in self.exclude_timesteps
        x = self.to_out(self.core(q, k, v, key_bias=bias, pred_mode="exact" if excluded else None))
        self.current_timestep += 1
        return x

    def forward_adaln(self, *args, **kwargs):
        raise TypeError("MXCrossAttention has no adaLN form (PixArt's block adds its output without a gate); "
                        "forward_adaln is the self-attention half's")


class QuantizedPixArtBlock(nn.Module):
    """PixArt-alpha transformer block: diffusers' BasicTransformerBlock with norm_type="ada_norm_single", which the
    reference's MXBasicTransformerBlock keeps.  forward computes, bit for bit on the same modules:
        shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = (
            scale_shift_table[None] + timestep.reshape(B, 6, -1)).chunk(6, dim=1)
        h = gate_msa * attn1(norm1(h) * (1 + scale_msa) + shift_msa) + h
        h = attn2(h, encoder_hidden_states, attention_mask=encoder_attention_mask) + h
        h = gate_mlp * ff(norm2(h) * (1 + scale_mlp) + shift_mlp) + h
    The self-attention and feed-forward halves run with their modulations and gated residuals inside the MX Linear
    kernels (MXSelfAttention.forward_adaln, with q, k and v from one GEMM, and QuantizedMlp.forward_adaln); IEEE add and
    multiply commute, so the kernels' ``h + gate * y`` is ``gate * y + h``.  attn2 runs its own forward and its residual
    is a torch add.

    ``orig_block``: ``attn1`` an MXSelfAttention and ``attn2`` an MXCrossAttention (or None), both after set_config;
    ``ff`` a QuantizedMlp or diffusers' FeedForward (wrapped in QuantizedMlp); ``norm1`` / ``norm2`` (torch LayerNorm)
    and the (6, C) ``scale_shift_table`` stay the host model's."""

    def __init__(self, orig_block, mx_specs=None):
        super().__init__()
        attn1, attn2, ff = orig_block.attn1, orig_block.attn2, orig_block.ff
        if not isinstance(attn1, MXSelfAttention) or isinstance(attn1, MXCrossAttention):
            raise TypeError(f"QuantizedPixArtBlock: attn1 must be modules.MXSelfAttention, got {type(attn1).__name__}")
        if attn2 is not None and not isinstance(attn2, MXCrossAttention):
            raise TypeError(f"QuantizedPixArtBlock: attn2 must be modules.MXCrossAttention or None, got "
                            f"{type(attn2).__name__}")
        for name, a in (("attn1", attn1), ("attn2", attn2)):
            if a is not None and a.core is None:
                raise RuntimeError(f"QuantizedPixArtBlock: {name}.set_config(...) must be called first")
        if not isinstance(ff, QuantizedMlp) and not hasattr(ff, "net"):
            raise TypeError(f"QuantizedPixArtBlock: ff must be QuantizedMlp or diffusers' FeedForward, got "
                            f"{type(ff).__name__}")
        self.norm1, self.attn1, self.attn2, self.norm2 = orig_block.norm1, attn1, attn2, orig_block.norm2
        self.ff = ff if isinstance(ff, QuantizedMlp) else QuantizedMlp(ff, mx_specs=mx_specs)
        self.scale_shift_table = orig_block.scale_shift_table

    def forward(self, hidden_states, attention_mask=None, encoder_hidden_states=None, encoder_attention_mask=None,
                timestep=None, **kwargs):
        """BasicTransformerBlock.forward's arguments; ``encoder_attention_mask`` is the additive (B, 1, S) text bias the
        diffusers transformer builds.  The other keyword arguments are ignored, as the attention shims ignore theirs."""
        if attention_mask is not None:
            raise ValueError("QuantizedPixArtBlock: a self-attention attention_mask cannot be applied on the fused path "
                             "(PixArt passes none)")
        if timestep is None:
            raise ValueError("QuantizedPixArtBlock: timestep (the adaLN-single embedding, (B, 6 * C)) is required")
        h = hidden_states
        shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = (
            t.squeeze(1) for t in (self.scale_shift_table[None] + timestep.reshape(h.shape[0], 6, -1)).chunk(6, dim=1))
        h = self.attn1.forward_adaln(self.norm1(h), shift_msa, scale_msa, h, gate_msa)
        if self.attn2 is not None:
            h = self.attn2(h, encoder_hidden_states, attention_mask=encoder_attention_mask) + h
        return self.ff.forward_adaln(self.norm2(h), shift_mlp, scale_mlp, h, gate_mlp)


class MxLinear(nn.Linear):
    """Drop-in for the reference's mx.Linear (microxscaling/mx/linear.py:227-320) on the MXINT8
    configuration of the workloads: same constructor (in_features, out_features, bias, mx_specs),
    forward = ops.mx_linear.  The MX-quantized weight operand is cached and rebuilt when the weight
    tensor changes (inference: once; also after ``.to(dtype)``).  The output has the input's dtype (float32, bfloat16
    or float16), whatever the parameters' dtype."""

    def __init__(self, in_features, out_features, bias=True, mx_specs=None, name=None):
        super().__init__(in_features, out_features, bias)
        resolve_linear_specs(mx_specs)          # also w_elem_format / round_weight / round (mx/linear.py:36-75)
        self.mx_specs = mx_specs
        self.name = name
        self._w_op = None
        self._w_key = None
        self._w_gen = 0             # counts invalidate() calls: keys operands cached outside the layer (MXSelfAttention's)
        # a loaded checkpoint writes the weight through .data (no version bump): drop the cached operand
        self.register_load_state_dict_post_hook(lambda module, incompatible_keys: module.invalidate())

    def invalidate(self):
        """Drop the cached MX-quantized weight operand (call after writing the weight through ``.data``)."""
        self._w_op = None
        self._w_key = None
        self._w_gen += 1

    def _check_inference(self, inputs_require_grad: bool):
        if torch.is_grad_enabled() and (self.weight.requires_grad or inputs_require_grad):
            raise RuntimeError("MxLinear is the inference forward of mx.Linear (the reference's backward is out of scope): "
                               "call it under torch.no_grad() / inference_mode, or freeze the parameters")

    def _operand(self) -> torch.Tensor:
        """The cached MX-quantized weight operand, rebuilt when the weight tensor has changed."""
        key = (self.weight.data_ptr(), self.weight._version, str(self.weight.device), self.weight.dtype)
        if self._w_op is None or self._w_key != key:
            self._w_op = ops.mx_linear_prepare_weight(self.weight.detach(), self.mx_specs)
            self._w_key = key
        return self._w_op

    def forward(self, inputs):
        return self.forward_adaln(inputs)

    def forward_adaln(self, inputs, **adaln):
        """forward with ops.mx_linear's adaLN arguments (shift=, scale=, residual=, gate=)."""
        self._check_inference(inputs.requires_grad)
        w_op = self._operand()
        b = None if self.bias is None else self.bias.detach()
        return ops.mx_linear(inputs, w_op, b, self.mx_specs, out_features=self.out_features, **adaln)
