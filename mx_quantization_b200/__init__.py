"""mx_quantization_b200 - the MXINT8 exponent-sign pruned-attention hot path of
d9bjo0522/mx_quantization as hand-written sm_100a CUDA behind a C ABI (include/mxprune.h).

Public API (mirrors the reference's operator interface for this path):
    exponent_approximation(Q, K, mx_specs).exponent_based_sign()
    pruned_attention(q, k, v, mx_specs, top_k, scale=None, return_mask=False)
    predict_topk / sparse_attention / quantize_mxint8 / predict_scores / exp_sign_approx
    mx_linear / mx_mlp (MX Linear, and the fused fc1 -> GELU -> fc2 MLP; both take adaLN's shift / scale / residual / gate)
    modules.QuantizedAttentionCore / DeiT, DiT, PixArt attention shims / QuantizedMlp (timm Mlp or diffusers FeedForward)
    / QuantizedDiTBlock (a DiT block) / QuantizedPixArtBlock (a PixArt-alpha adaLN-single block)
"""
from .ops import (exp_sign_approx, last_launch_count, limits, mx_linear, mx_linear_prepare_weight,  # noqa: F401
                  mx_mlp, predict_scores, predict_topk,
                  pruned_attention, quantize_mxint8, set_attention_path, set_fused_path, set_predict_path, sparse_attention)
from .analysis import coverage_rate, diff_idx_analysis, topk_overlap  # noqa: F401
from .predictor import exponent_approximation  # noqa: F401
from .specs import PathSpecs, resolve_specs  # noqa: F401

__all__ = ["exponent_approximation", "pruned_attention", "predict_topk", "sparse_attention",
           "quantize_mxint8", "predict_scores", "exp_sign_approx", "resolve_specs", "PathSpecs",
           "limits", "last_launch_count", "set_attention_path", "set_predict_path", "set_fused_path", "coverage_rate", "topk_overlap", "diff_idx_analysis", "mx_linear", "mx_linear_prepare_weight", "mx_mlp"]
