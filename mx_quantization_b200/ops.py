"""Tensor-level entry points over the C ABI (include/mxprune.h).

PyTorch is plumbing here: it owns device memory and the current stream; every computation
happens in libmxprune's sm_100a kernels.  CPU tensors are rejected - there is no CPU path.
"""
from ctypes import c_void_p
from typing import Optional, Tuple

import torch

from . import _lib
from .specs import resolve_linear_specs, resolve_specs


def _stream() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> c_void_p:
    return c_void_p(0 if t is None else t.data_ptr())


# Element types of the activations (MXP_DT_* of include/mxprune.h).  fp32 is the reference's fake-quant dtype; bf16 and
# fp16 are what autocast / 16-bit pipelines hand over, read natively by the exponent-sign path (widening is exact).
DTYPE_CODES = {torch.float32: _lib.MXP_DT_F32, torch.bfloat16: _lib.MXP_DT_BF16, torch.float16: _lib.MXP_DT_F16}


def _dtype_code(dtype: torch.dtype, name: str) -> int:
    if dtype not in DTYPE_CODES:
        raise ValueError(f"{name}: expected float32, bfloat16 or float16, got {dtype}")
    return DTYPE_CODES[dtype]


def _same_dtype(*named) -> torch.dtype:
    """The one element type shared by the (name, tensor) pairs; mixed dtypes raise."""
    for name, t in named:
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor")
    dt = named[0][1].dtype
    for name, t in named[1:]:
        if t.dtype != dt:
            raise ValueError(f"{named[0][0]} is {dt} but {name} is {t.dtype}: q, k and v must share one dtype")
    return dt


def _view4(t: torch.Tensor, name: str, half_ok: bool = False) -> torch.Tensor:
    """Accept the strided (B,H,N,hd) views the attention modules produce.  fp32: copy only when the
    layout is outside what the kernels address (innermost stride 1, 16-byte aligned rows).  bf16 / fp16
    (``half_ok``: the entry point reads them natively): the same 16-byte rules (strides multiples of 8
    elements), and a view that breaks them raises - a copy would be the conversion pass the native path avoids."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if t.device.type != "cuda":
        raise ValueError(f"{name}: expected a CUDA tensor (device={t.device}); there is no CPU fallback")
    if t.dim() != 4:
        raise ValueError(f"{name}: expected a 4-D (B,H,N,head_dim) tensor, got shape {tuple(t.shape)}")
    if t.dtype in (torch.bfloat16, torch.float16) and half_ok:
        if not (t.stride(-1) == 1 and t.data_ptr() % 16 == 0 and all(s % 8 == 0 for s in t.stride()[:3])):
            raise ValueError(f"{name}: a {t.dtype} view needs innermost stride 1, a 16-byte aligned base and strides "
                             f"that are multiples of 8 elements, got strides {tuple(t.stride())}")
        return t
    if t.dtype != torch.float32:
        raise ValueError(f"{name}: expected float32 (the reference's fake-quant dtype)"
                         f"{', bfloat16 or float16' if half_ok else ''}, got {t.dtype}")
    ok = t.stride(-1) == 1 and t.data_ptr() % 16 == 0 and all(s % 4 == 0 for s in t.stride()[:3])
    return t if ok else t.contiguous()


def _out_tensor(out, shape, in_dtype, dev):
    """The output buffer and its MXP_DT_* code: a new (B,H,Nq,hd) tensor of the inputs' dtype (as
    torch.nn.functional.scaled_dot_product_attention), or the caller's fp32 / input-dtype view with innermost
    stride 1."""
    if out is None:
        out = torch.empty(shape, dtype=in_dtype, device=dev)
    elif (tuple(out.shape) != tuple(shape) or out.dtype not in (torch.float32, in_dtype) or out.stride(-1) != 1
          or out.device != dev):
        raise ValueError(f"out must be a (B,H,Nq,head_dim) view of dtype float32 or {in_dtype} with innermost stride 1 "
                         "on the inputs' device")
    return out, _dtype_code(out.dtype, "out")


def _strides(t: torch.Tensor) -> Tuple[int, int, int]:
    return t.stride(0), t.stride(1), t.stride(2)


def _same_device(*ts):
    dev = ts[0].device
    for t in ts[1:]:
        if t is not None and t.device != dev:
            raise ValueError("all tensors must live on the same CUDA device")
    return dev


def limits() -> Tuple[int, int]:
    import ctypes
    a, b = ctypes.c_int(), ctypes.c_int()
    _lib.load().mxp_limits(ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def set_attention_path(path: str) -> None:
    """'tcgen05' (default: both GEMMs of the exact stage on the tensor cores) or 'cuda_core' (dp4a)."""
    codes = {"tcgen05": 0, "cuda_core": 1}
    if path not in codes:
        raise ValueError(f"attention path must be one of {sorted(codes)}")
    _lib.check(_lib.load().mxp_set_attention_path(codes[path]), "mxp_set_attention_path")


def set_predict_path(path: str) -> None:
    """'tcgen05' (default: predictor scored on the tensor cores, keys selected in registers) or
    'cuda_core' (XOR/POPC kernel; also used automatically outside the tensor-core kernel's domain)."""
    codes = {"tcgen05": 0, "cuda_core": 1}
    if path not in codes:
        raise ValueError(f"predict path must be one of {sorted(codes)}")
    _lib.check(_lib.load().mxp_set_predict_path(codes[path]), "mxp_set_predict_path")


def set_fused_path(mode) -> None:
    """True / 1 (default): the round-2 launch plans where they are measured faster - the fused one-launch kernel (DeiT-shaped
    calls: 129-256 keys staged in 128-row steps, top_k / Nk <= 0.35), the cost-follows-k attention kernel (Nk <= 256, same
    bound) and the sampled fine window of the long-sequence selection; 2: the fused launch wherever the shape is in its domain;
    False / 0: always the three kernels with the dense epilogue, and for Nk > 256 the long-sequence selection on its radix
    levels alone (the attention kernel for Nk > 256 is the same in every mode).  Results agree (A/B aid)."""
    _lib.check(_lib.load().mxp_set_fused_path(int(mode)), "mxp_set_fused_path")


def last_launch_count() -> int:
    return _lib.load().mxp_last_launch_count()


def quantize_mxint8(x: torch.Tensor, mx_specs, with_signs: bool = False):
    """MXINT8 codes/exponents of ``x`` along head_dim (replaces quantize_mx_op on this path).

    ``x``: float32, bfloat16 or float16 (head_dim a multiple of 8); a 16-bit x gives exactly the result of
    ``x.float()``.
    Returns (codes int8 (B,H,N,hd), exps int8 (B,H,N,nb)[, signs int32 (B,H,N,nb)])."""
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    x = _view4(x, "x", half_ok=True)
    B, H, N, hd = x.shape
    nb = (hd + 31) // 32
    with torch.cuda.device(x.device):
        codes = torch.empty((B, H, N, hd), dtype=torch.int8, device=x.device)
        exps = torch.empty((B, H, N, nb), dtype=torch.int8, device=x.device)
        signs = torch.empty((B, H, N, nb), dtype=torch.int32, device=x.device) if with_signs else None
        rc = lib.mxp_quantize_mxint8_dt(_ptr(x), _dtype_code(x.dtype, "x"), *_strides(x), B, H, N, hd, sp.bfloat_bits,
                                        int(sp.flush), _ptr(codes), _ptr(exps), _ptr(signs), _stream())
    _lib.check(rc, "mxp_quantize_mxint8")
    return (codes, exps, signs) if with_signs else (codes, exps)


def exp_sign_approx(x: torch.Tensor, mx_specs) -> torch.Tensor:
    """Dense (code<0 ? -1 : +1) * 2^e tensor, fp32 (B,H,N,hd)."""
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    x = _view4(x, "x")
    B, H, N, hd = x.shape
    with torch.cuda.device(x.device):
        out = torch.empty((B, H, N, hd), dtype=torch.float32, device=x.device)
        rc = lib.mxp_exp_sign_approx(_ptr(x), *_strides(x), B, H, N, hd, sp.bfloat_bits, int(sp.flush),
                                     _ptr(out), _stream())
    _lib.check(rc, "mxp_exp_sign_approx")
    return out


# The reference's sources of the top-k ranking (workloads/deit/scripts/main.py:105-131): pred_mode strings as
# the reference spells them, plus "exact" for its `top_k and not approx_flag` branch (top-k of the true scores).
PRED_MODES = {"ex_pred": 0, "partial_Q": 1, "partial_K": 2, "exact": 3, "MXINT4": 4, "two_step_leading_ones": 5,
              "true_ex": 6}


def _pred_mode_code(pred_mode: str) -> int:
    if pred_mode not in PRED_MODES:
        raise NotImplementedError(f"pred_mode={pred_mode!r}: built modes are {sorted(PRED_MODES)} and 'ELSA'; "
                                  "there is no fallback")
    return PRED_MODES[pred_mode]


ELSA_THETA_BIAS = 0.127     # funcs/elsa_approximation.py:101


def elsa_rank_cap(d: int) -> float:
    """d - 2 h_c, h_c the largest Hamming distance the reference's clamp maps to angle 0
    (funcs/elsa_approximation.py:135-136: clamp((pi / k) * hamming - theta_bias, min=0), evaluated in fp32 as torch does):
    hash dot products at or above this value tie."""
    h = torch.arange(0, d + 1, dtype=torch.float32)
    corrected = torch.clamp((torch.pi / d) * h - ELSA_THETA_BIAS, min=0)
    hc = int(torch.nonzero(corrected == 0).max())
    return float(d - 2 * hc)


def _elsa_proj(orthogonal_matrix, hd, dev):
    if orthogonal_matrix is None:
        raise ValueError("pred_mode='ELSA' needs orthogonal_matrix (the reference's (head_dim, head_dim) projection)")
    P = orthogonal_matrix.to(device=dev, dtype=torch.float32).contiguous()
    if tuple(P.shape) != (hd, hd):
        raise ValueError(f"orthogonal_matrix must be ({hd}, {hd}), got {tuple(P.shape)}")
    return P


def _qk_shapes(q, k):
    B, H, Nq, hd = q.shape
    if k.shape[0] != B or k.shape[1] != H or k.shape[3] != hd:
        raise ValueError(f"q {tuple(q.shape)} and k {tuple(k.shape)} disagree on (B,H,head_dim)")
    return B, H, Nq, k.shape[2], hd


def predict_scores(q: torch.Tensor, k: torch.Tensor, mx_specs) -> torch.Tensor:
    """Dense predicted scores (B,H,Nq,Nk) - parity aid, O(N^2) output."""
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    q, k = _view4(q, "q"), _view4(k, "k")
    _same_device(q, k)
    B, H, Nq, Nk, hd = _qk_shapes(q, k)
    with torch.cuda.device(q.device):
        out = torch.empty((B, H, Nq, Nk), dtype=torch.float32, device=q.device)
        rc = lib.mxp_predict_scores(_ptr(q), *_strides(q), _ptr(k), *_strides(k), B, H, Nq, Nk, hd,
                                    sp.bfloat_bits, int(sp.flush), _ptr(out), _stream())
    _lib.check(rc, "mxp_predict_scores")
    return out


def predict_topk(q: torch.Tensor, k: torch.Tensor, mx_specs, top_k: int, return_idx: bool = False,
                 return_codes: bool = False, pred_mode: str = "ex_pred", scale: Optional[float] = None,
                 key_bias: Optional[torch.Tensor] = None, orthogonal_matrix: Optional[torch.Tensor] = None):
    """Fused quantize + predictor + per-row top-k.

    Returns a dict: mask int32 (B,H,Nq,ceil(Nk/32)) [bit j%32 of word j//32 = key j kept],
    optionally idx int32 (B,H,Nq,top_k) ascending key order, and q/k codes+exps.
    pred_mode: "ex_pred" (exponent-sign, default), "partial_Q", "partial_K", "MXINT4" or "exact" (top-k of the
    true scores * scale) - see PRED_MODES.
    q, k: float32, or (pred_mode "ex_pred", head_dim a multiple of 8 in [32, 128]) both bfloat16 or both float16 -
    the result of the same call on q.float(), k.float()."""
    if pred_mode == "ELSA":
        return _predict_topk_elsa(q, k, mx_specs, top_k, return_idx, return_codes, key_bias, orthogonal_matrix)
    mode = _pred_mode_code(pred_mode)
    if mode != 0:
        return _predict_topk_mode(q, k, mx_specs, top_k, mode, scale, return_idx, return_codes, key_bias)
    if key_bias is not None:
        raise ValueError("predict_topk with pred_mode='ex_pred' takes no key_bias (use pruned_attention)")
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    dt = _dtype_code(_same_dtype(("q", q), ("k", k)), "q")
    q, k = _view4(q, "q", half_ok=True), _view4(k, "k", half_ok=True)
    dev = _same_device(q, k)
    B, H, Nq, Nk, hd = _qk_shapes(q, k)
    nb, nw = (hd + 31) // 32, (Nk + 31) // 32
    res = {}
    with torch.cuda.device(dev):
        res["mask"] = torch.empty((B, H, Nq, nw), dtype=torch.int32, device=dev)
        if return_idx:
            res["idx"] = torch.empty((B, H, Nq, int(top_k)), dtype=torch.int32, device=dev)
        if return_codes:
            res["q_codes"] = torch.empty((B, H, Nq, hd), dtype=torch.int8, device=dev)
            res["q_exps"] = torch.empty((B, H, Nq, nb), dtype=torch.int8, device=dev)
            res["k_codes"] = torch.empty((B, H, Nk, hd), dtype=torch.int8, device=dev)
            res["k_exps"] = torch.empty((B, H, Nk, nb), dtype=torch.int8, device=dev)
        ws_bytes = lib.mxp_predict_topk_workspace_bytes(B, H, Nq, Nk, hd)
        ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev) if ws_bytes else None
        rc = lib.mxp_predict_topk_dt(_ptr(q), *_strides(q), _ptr(k), *_strides(k), dt, B, H, Nq, Nk, hd, int(top_k),
                                     sp.bfloat_bits, int(sp.flush), _ptr(res["mask"]), _ptr(res.get("idx")),
                                     _ptr(res.get("q_codes")), _ptr(res.get("q_exps")),
                                     _ptr(res.get("k_codes")), _ptr(res.get("k_exps")),
                                     _ptr(ws), ws_bytes, _stream())
    _lib.check(rc, "mxp_predict_topk")
    return res


def _key_bias_2d(key_bias, B, Nk, dev):
    if key_bias.dtype != torch.float32 or key_bias.numel() != B * Nk or key_bias.device != dev:
        raise ValueError("key_bias must be an fp32 tensor with B*Nk elements, (B, ..., Nk), on q's device")
    return key_bias.reshape(B, Nk).contiguous()


def _predict_topk_mode(q, k, mx_specs, top_k, mode, scale, return_idx, return_codes, key_bias=None):
    if return_codes:
        raise ValueError("return_codes is available with pred_mode='ex_pred' only")
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    q, k = _view4(q, "q"), _view4(k, "k")
    dev = _same_device(q, k)
    B, H, Nq, Nk, hd = _qk_shapes(q, k)
    scale = float(hd) ** -0.5 if scale is None else float(scale)
    res = {}
    with torch.cuda.device(dev):
        res["mask"] = torch.empty((B, H, Nq, (Nk + 31) // 32), dtype=torch.int32, device=dev)
        if return_idx:
            res["idx"] = torch.empty((B, H, Nq, int(top_k)), dtype=torch.int32, device=dev)
        kb = None if key_bias is None else _key_bias_2d(key_bias, B, Nk, q.device)
        rc = lib.mxp_predict_topk_mode(_ptr(q), *_strides(q), _ptr(k), *_strides(k), B, H, Nq, Nk, hd, int(top_k),
                                       mode, scale, sp.bfloat_bits, int(sp.flush), _ptr(kb), Nk, _ptr(res["mask"]),
                                       _ptr(res.get("idx")), _ptr(None), 0, _stream())
    _lib.check(rc, "mxp_predict_topk_mode")
    return res


def _predict_topk_elsa(q, k, mx_specs, top_k, return_idx, return_codes, key_bias, orthogonal_matrix):
    if return_codes or key_bias is not None:
        raise ValueError("pred_mode='ELSA' takes neither return_codes nor key_bias")
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    q, k = _view4(q, "q"), _view4(k, "k")
    dev = _same_device(q, k)
    B, H, Nq, Nk, hd = _qk_shapes(q, k)
    if Nq != Nk:
        raise ValueError("pred_mode='ELSA' needs Nq == Nk (the reference broadcasts the key norms over query rows)")
    P = _elsa_proj(orthogonal_matrix, hd, dev)
    res = {}
    with torch.cuda.device(dev):
        res["mask"] = torch.empty((B, H, Nq, (Nk + 31) // 32), dtype=torch.int32, device=dev)
        if return_idx:
            res["idx"] = torch.empty((B, H, Nq, int(top_k)), dtype=torch.int32, device=dev)
        rc = lib.mxp_predict_topk_elsa(_ptr(q), *_strides(q), _ptr(k), *_strides(k), B, H, Nq, hd, int(top_k),
                                       _ptr(P), elsa_rank_cap(hd), sp.bfloat_bits, int(sp.flush),
                                       _ptr(res["mask"]), _ptr(res.get("idx")), _stream())
    _lib.check(rc, "mxp_predict_topk_elsa")
    return res


def sparse_attention(q_codes, q_exps, k_codes, k_exps, v: torch.Tensor, mask: torch.Tensor, mx_specs,
                     scale: Optional[float] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Exact MXINT8 softmax(QK^T*scale)V over the keys selected by ``mask``.

    ``v``: float32, bfloat16 or float16 (head_dim a multiple of 8 in [32, 128] for 16-bit); the output is of v's
    dtype unless an fp32 ``out`` is given."""
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    v = _view4(v, "v", half_ok=True)
    B, H, Nk, hd = v.shape
    if q_codes.dim() != 4:
        raise ValueError(f"q_codes: expected a 4-D (B,H,Nq,head_dim) tensor, got shape {tuple(q_codes.shape)}")
    Nq = q_codes.shape[2]
    nb, nw = (hd + 31) // 32, (Nk + 31) // 32
    dev = _same_device(v, q_codes, q_exps, k_codes, k_exps, mask)
    for name, t, dt, shape in (("q_codes", q_codes, torch.int8, (B, H, Nq, hd)), ("q_exps", q_exps, torch.int8, (B, H, Nq, nb)),
                               ("k_codes", k_codes, torch.int8, (B, H, Nk, hd)), ("k_exps", k_exps, torch.int8, (B, H, Nk, nb)),
                               ("mask", mask, torch.int32, (B, H, Nq, nw))):
        if t.dtype != dt or not t.is_contiguous():
            raise ValueError(f"{name}: expected a contiguous {dt} tensor")
        if tuple(t.shape) != shape:
            raise ValueError(f"{name}: expected shape {shape} (from v {tuple(v.shape)}), got {tuple(t.shape)}")
    scale = float(hd) ** -0.5 if scale is None else float(scale)
    with torch.cuda.device(dev):
        out, out_dt = _out_tensor(out, (B, H, Nq, hd), v.dtype, dev)
        ws_bytes = lib.mxp_sparse_attention_workspace_bytes(B, H, Nq, Nk, hd)
        ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
        rc = lib.mxp_sparse_attention_dt(_ptr(q_codes), _ptr(q_exps), _ptr(k_codes), _ptr(k_exps),
                                         _ptr(v), *_strides(v), _dtype_code(v.dtype, "v"), _ptr(mask), B, H, Nq, Nk, hd,
                                         scale, sp.bfloat_bits, int(sp.flush),
                                         _ptr(out), *_strides(out), out_dt, _ptr(ws), ws_bytes, _stream())
    _lib.check(rc, "mxp_sparse_attention")
    return out


def pruned_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, mx_specs, top_k: int,
                     scale: Optional[float] = None, return_mask: bool = False,
                     out: Optional[torch.Tensor] = None, _kernel_ms: Optional[list] = None,
                     key_bias: Optional[torch.Tensor] = None, pred_mode: str = "ex_pred",
                     orthogonal_matrix: Optional[torch.Tensor] = None):
    """MXINT8 exponent-sign predicted top-k attention: q,k,v (B,H,N,hd) -> out (B,H,Nq,hd).

    q, k, v: float32, or all bfloat16 or all float16 (pred_mode "ex_pred", head_dim a multiple of 8 in [32, 128],
    the default path switches): a 16-bit call gives the masks of the same call on q.float(), k.float(), v.float()
    and the same fp32 output before its final store.  The output dtype is ``out``'s, else q's (a 16-bit output is
    the fp32 result rounded to nearest even).  No conversion pass runs: the same launches as the fp32 call.

    ``pred_mode``: what ranks the keys - "ex_pred" (default), "partial_Q", "partial_K", "MXINT4" (the reference's
    pred_mode values, workloads/deit/scripts/main.py:109-118) or "exact" (its approx_flag=False branch:
    top-k of the true scores, main.py:130), or "ELSA" with ``orthogonal_matrix`` (head_dim, head_dim) as the
    reference's modules receive it (main.py:119-121).  Everything after the selection is the same.

    Drop-in for lines 101-152 of workloads/deit/scripts/main.py (DiT models.py:168-225, PixArt
    MX_transformer_block.py:647-710) when mx_quant, top_k, approx_flag and pred_mode=="ex_pred".
    ``out`` may be any fp32 or q-dtype (B,H,Nq,hd) *view* with innermost stride 1, e.g. a permuted
    (B,Nq,H,hd) buffer so that the module's transpose(1,2).reshape(B,N,C) is free.

    ``key_bias``: PixArt cross-attention's additive text mask (MX_transformer_block.py:794-803,
    821-822), any fp32 tensor (also with 16-bit q, k, v) with B * Nk elements laid out (B, ..., Nk) - e.g. the reference's
    (B,1,1,S) attention_mask; it is added to the true AND the predicted scores.  Nq may differ
    from Nk; with pred_mode "ex_pred" a bias takes every Nk up to 8192, the other modes keep Nk <= 256.
    """
    sp = resolve_specs(mx_specs)
    lib = _lib.load()
    in_dtype = _same_dtype(("q", q), ("k", k), ("v", v))
    dt = _dtype_code(in_dtype, "q")
    if dt != _lib.MXP_DT_F32 and (pred_mode != "ex_pred" or _kernel_ms is not None):
        raise ValueError(f"{in_dtype} q/k/v: pred_mode='ex_pred' without the per-kernel profile entry only "
                         f"(got pred_mode={pred_mode!r}); pass float32 tensors for the other modes")
    q, k, v = _view4(q, "q", half_ok=True), _view4(k, "k", half_ok=True), _view4(v, "v", half_ok=True)
    dev = _same_device(q, k, v, out)
    B, H, Nq, Nk, hd = _qk_shapes(q, k)
    if tuple(v.shape) != (B, H, Nk, hd):
        raise ValueError(f"v {tuple(v.shape)} must be (B,H,Nk,head_dim) = {(B, H, Nk, hd)}")
    scale = float(hd) ** -0.5 if scale is None else float(scale)
    elsa = pred_mode == "ELSA"
    if elsa and (key_bias is not None or _kernel_ms is not None or Nq != Nk):
        raise ValueError("pred_mode='ELSA' needs Nq == Nk and takes neither key_bias nor the per-kernel profile entry")
    P = _elsa_proj(orthogonal_matrix, hd, dev) if elsa else None
    mode = 0 if elsa else _pred_mode_code(pred_mode)
    if mode != 0 and _kernel_ms is not None:
        raise ValueError("the per-kernel profile entry is available with pred_mode='ex_pred' only")
    with torch.cuda.device(dev):
        out, out_dt = _out_tensor(out, (B, H, Nq, hd), in_dtype, dev)
        mask = torch.empty((B, H, Nq, (Nk + 31) // 32), dtype=torch.int32, device=dev) if return_mask else None
        ws_bytes = lib.mxp_pruned_attention_workspace_bytes(B, H, Nq, Nk, hd)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        args = (_ptr(q), *_strides(q), _ptr(k), *_strides(k), _ptr(v), *_strides(v),
                B, H, Nq, Nk, hd, int(top_k), scale, sp.bfloat_bits, int(sp.flush),
                _ptr(out), *_strides(out), _ptr(mask), _ptr(ws), ws_bytes, _stream())
        kb = None if key_bias is None else _key_bias_2d(key_bias, B, Nk, q.device)
        if elsa:
            rc = lib.mxp_pruned_attention_elsa(*args[:12], B, H, Nq, hd, int(top_k), _ptr(P), elsa_rank_cap(hd),
                                               *args[18:])
        elif mode != 0:
            rc = lib.mxp_pruned_attention_mode(*args[:18], mode, *args[18:-4], _ptr(kb), Nk, *args[-4:])
        elif dt != _lib.MXP_DT_F32 or out_dt != _lib.MXP_DT_F32:
            rc = lib.mxp_pruned_attention_dt(*args[:12], dt, *args[12:25], out_dt, _ptr(kb), Nk if kb is not None else 0,
                                             *args[-4:])
        elif key_bias is not None:
            if _kernel_ms is not None:
                raise ValueError("the per-kernel profile entry takes no key_bias")
            rc = lib.mxp_pruned_attention_biased(*args[:-4], _ptr(kb), Nk, *args[-4:])
        elif _kernel_ms is None:
            rc = lib.mxp_pruned_attention(*args)
        else:       # measurement aid: per-kernel CUDA-event times (synchronises)
            import ctypes
            ms = (ctypes.c_float * 3)()
            rc = lib.mxp_pruned_attention_profile(*args, ms)
            _kernel_ms[:] = [float(x) for x in ms]
    _lib.check(rc, "mxp_pruned_attention")
    return (out, mask) if return_mask else out


# ---- MX Linear (SURVEY.md 8 f2) -------------------------------------------------------------------
def mx_linear_prepare_weight(weight: torch.Tensor, mx_specs) -> torch.Tensor:
    """MX-quantize an (out_features, in_features) weight once into the GEMM's operand order.  ``weight``: float32,
    bfloat16 or float16; a 16-bit weight gives the bytes of ``weight.float()``'s operand."""
    sp = resolve_linear_specs(mx_specs)
    lib = _lib.load()
    if not isinstance(weight, torch.Tensor) or weight.dim() != 2 or weight.dtype not in DTYPE_CODES or not weight.is_cuda:
        raise ValueError("weight must be a CUDA float32, bfloat16 or float16 (out_features, in_features) tensor")
    w = weight if weight.stride(1) == 1 else weight.contiguous()
    N, K = w.shape
    with torch.cuda.device(w.device):
        w_op = torch.empty((lib.mxp_mx_linear_weight_bytes(N, K),), dtype=torch.uint8, device=w.device)
        rc = lib.mxp_mx_linear_prepare_weight_dt(_ptr(w), DTYPE_CODES[w.dtype], w.stride(0), N, K, sp.bfloat_bits,
                                                 int(sp.flush), _ptr(w_op), _stream())
    _lib.check(rc, "mxp_mx_linear_prepare_weight")
    return w_op


def _linear_rows(x: torch.Tensor) -> torch.Tensor:
    """x (..., K) as (M, K) rows.  fp32: copied when the rows are not one strided 2-D view.  bf16 / fp16 (read
    natively): a view with innermost stride 1, a 16-byte aligned base and a row stride that is a multiple of 8 elements,
    else this raises - a copy would be the conversion-sized pass the native path avoids."""
    if not isinstance(x, torch.Tensor):
        raise TypeError("x: expected a torch.Tensor")
    if x.dtype not in DTYPE_CODES:
        raise ValueError(f"x: expected float32, bfloat16 or float16, got {x.dtype}")
    K = x.shape[-1]
    if x.dtype == torch.float32:
        x2 = x.reshape(-1, K)
        return x2 if x2.stride(1) == 1 else x2.contiguous()
    try:
        x2 = x.view(-1, K)
    except RuntimeError:
        x2 = None
    if x2 is None or x2.stride(1) != 1 or x2.stride(0) % 8 or x2.data_ptr() % 16:
        raise ValueError(f"x: a {x.dtype} input needs rows that form one 2-D view with innermost stride 1, a 16-byte "
                         f"aligned base and a row stride that is a multiple of 8 elements, got shape {tuple(x.shape)} "
                         f"strides {tuple(x.stride())}")
    return x2


def _weight_operand(weight: torch.Tensor, K: int, out_features: Optional[int], mx_specs,
                    what: str = "out_features") -> Tuple[torch.Tensor, int]:
    """(w_op, N): a prepared operand checked against (out_features, K), or a raw (N, K) weight quantized now."""
    lib = _lib.load()
    if weight.dtype == torch.uint8:
        if out_features is None:
            raise ValueError(f"{what} is required with a prepared weight operand")
        N = int(out_features)
        if not weight.is_contiguous() or weight.numel() != lib.mxp_mx_linear_weight_bytes(N, K):
            raise ValueError(f"prepared weight operand: expected {lib.mxp_mx_linear_weight_bytes(N, K)} contiguous bytes for "
                             f"out_features={N}, in_features={K}, got {weight.numel()}")
        return weight, N
    return mx_linear_prepare_weight(weight, mx_specs), weight.shape[0]


def _check_bias(bias: Optional[torch.Tensor], N: int) -> None:
    if bias is not None and (bias.dtype not in DTYPE_CODES or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("bias must be a contiguous float32, bfloat16 or float16 tensor with out_features elements")


def _adaln_args(x: torch.Tensor, K: int, N: int, shift, scale, residual, gate) -> tuple:
    """The adaLN arguments of mxp_mx_*_adaln_dt (tokens, then each tensor's pointer and row stride) for a (B, T, K) x:
    shift / scale (B, K) and gate (B, N) rows with innermost stride 1 (e.g. ``.chunk(6, dim=1)`` views, read in
    place), a residual (B, T, N) whose rows form one (B*T, N) view with innermost stride 1; all of x's dtype."""
    if (shift is None) != (scale is None):
        raise ValueError("shift and scale: pass both or neither")
    if (residual is None) != (gate is None):
        raise ValueError("residual and gate: pass both or neither")
    if x.dim() != 3:
        raise ValueError(f"shift / scale / residual / gate need x of shape (B, T, in_features), got {tuple(x.shape)}")
    B, T = x.shape[0], x.shape[1]
    args = [T]
    for name, t, shape in (("shift", shift, (B, K)), ("scale", scale, (B, K)), ("residual", residual, (B, T, N)),
                           ("gate", gate, (B, N))):
        if t is None:
            args += [_ptr(None), 0]
            continue
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor")
        if t.dtype != x.dtype:
            raise ValueError(f"{name} is {t.dtype} but x is {x.dtype}: shift, scale, residual and gate take x's dtype")
        if tuple(t.shape) != shape:
            raise ValueError(f"{name}: expected shape {shape}, got {tuple(t.shape)}")
        rows = t
        if t.dim() == 3:
            try:
                rows = t.view(-1, N)
            except RuntimeError:
                rows = None
        if rows is None or rows.stride(1) != 1:
            raise ValueError(f"{name}: needs rows with innermost stride 1{' forming one 2-D view' if t.dim() == 3 else ''}, "
                             f"got strides {tuple(t.stride())}")
        # a single row's stride is never used: pass the row width, which meets the library's rules
        args += [_ptr(t), rows.stride(0) if rows.shape[0] > 1 else shape[-1]]
    _same_device(x, shift, scale, residual, gate)
    return tuple(args)


def _norm_args(x: torch.Tensor, K: int, ln_eps, ln_weight, ln_bias) -> tuple:
    """The LayerNorm arguments of mxp_mx_*_ex_dt (layer_norm, ln_weight, ln_bias, ln_eps): the norm is on when ``ln_eps``
    is given; ``ln_weight`` / ``ln_bias`` are (K,) contiguous tensors of x's dtype, both or neither."""
    if (ln_weight is None) != (ln_bias is None):
        raise ValueError("ln_weight and ln_bias: pass both or neither")
    if ln_eps is None:
        if ln_weight is not None:
            raise ValueError("ln_weight / ln_bias need ln_eps (the LayerNorm's eps)")
        return (0, None, None, 0.0)
    eps = float(ln_eps)
    if not eps >= 0.0:
        raise ValueError(f"ln_eps: need a number >= 0, got {ln_eps!r}")
    for name, t in (("ln_weight", ln_weight), ("ln_bias", ln_bias)):
        if t is None:
            continue
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor")
        if t.dtype != x.dtype or tuple(t.shape) != (K,) or not t.is_contiguous() or t.data_ptr() % 16:
            raise ValueError(f"{name}: expected a contiguous, 16-byte aligned ({K},) tensor of x's dtype {x.dtype}, got "
                             f"{t.dtype} {tuple(t.shape)} strides {tuple(t.stride())}")
    _same_device(x, ln_weight, ln_bias)
    return (1, _ptr(ln_weight), _ptr(ln_bias), eps)


def _ex_args(x: torch.Tensor, M: int, K: int, N: int, ln_eps, ln_weight, ln_bias, add, shift, scale, residual,
             gate) -> tuple:
    """The norm and block arguments of mxp_mx_*_ex_dt.  ``add`` (x.shape[:-1] + (N,), x's dtype, rows with innermost
    stride 1 forming one 2-D view) takes the residual slot without a gate; the adaLN tensors need a (B, T, K) x."""
    norm = _norm_args(x, K, ln_eps, ln_weight, ln_bias)
    if add is not None and (residual is not None or gate is not None):
        raise ValueError("add is the plain residual add: pass it without residual / gate")
    if any(t is not None for t in (shift, scale, residual, gate)):
        ad = list(_adaln_args(x, K, N, shift, scale, residual, gate))
    else:
        ad = [M] + [_ptr(None), 0] * 4
    if add is not None:
        if not isinstance(add, torch.Tensor):
            raise TypeError("add: expected a torch.Tensor")
        shape = tuple(x.shape[:-1]) + (N,)
        if add.dtype != x.dtype or tuple(add.shape) != shape:
            raise ValueError(f"add: expected shape {shape} of x's dtype {x.dtype}, got {add.dtype} {tuple(add.shape)}")
        try:
            rows = add.view(-1, N)
        except RuntimeError:
            rows = None
        if rows is None or rows.stride(1) != 1 or rows.data_ptr() % (16 if x.dtype == torch.float32 else 8) \
                or (rows.shape[0] > 1 and rows.stride(0) % 4):
            raise ValueError(f"add: needs rows with innermost stride 1 forming one 2-D view, an aligned base and a row "
                             f"stride that is a multiple of 4, got strides {tuple(add.stride())}")
        _same_device(x, add)
        ad[5:7] = [_ptr(add), rows.stride(0) if rows.shape[0] > 1 else N]
    return norm + tuple(ad)


def layer_norm(x: torch.Tensor, weight: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
               eps: float = 1e-5) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The LayerNorm mx_linear / mx_mlp apply with ``ln_eps`` (parity aid): ``torch.native_layer_norm(x, (K,), weight,
    bias, eps)`` on CUDA bit for bit - (y, mean, rstd), mean and rstd fp32 of shape x.shape[:-1] + (1,).  ``x``: a CUDA
    float32, bfloat16 or float16 tensor whose rows form one 2-D view with innermost stride 1 (K a multiple of 4);
    ``weight`` / ``bias``: (K,) tensors of x's dtype, both or neither."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda or x.dtype not in DTYPE_CODES or x.dim() < 1:
        raise ValueError("x must be a CUDA float32, bfloat16 or float16 tensor")
    K = x.shape[-1]
    try:
        x2 = x.view(-1, K)
    except RuntimeError:
        x2 = None
    if x2 is None or x2.stride(1) != 1 or (x2.shape[0] > 1 and x2.stride(0) % 4) or \
            x2.data_ptr() % (16 if x.dtype == torch.float32 else 8):
        raise ValueError(f"x: needs rows with innermost stride 1 forming one 2-D view, an aligned base and a row stride "
                         f"that is a multiple of 4, got strides {tuple(x.stride())}")
    _, w, b, e = _norm_args(x, K, eps, weight, bias)
    M = x2.shape[0]
    with torch.cuda.device(x.device):
        y = torch.empty(x.shape, dtype=x.dtype, device=x.device)
        stats = torch.empty((2, M), dtype=torch.float32, device=x.device)
        rc = _lib.load().mxp_layer_norm_dt(_ptr(x2), DTYPE_CODES[x.dtype], x2.stride(0) if M > 1 else K, M, K, w, b, e,
                                           _ptr(y), _ptr(stats[0]), _ptr(stats[1]), _stream())
    _lib.check(rc, "mxp_layer_norm_dt")
    shape = tuple(x.shape[:-1]) + (1,)
    return y, stats[0].view(shape), stats[1].view(shape)


def mx_linear(x: torch.Tensor, weight, bias: Optional[torch.Tensor], mx_specs,
              out_features: Optional[int] = None, *, shift: Optional[torch.Tensor] = None,
              scale: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
              gate: Optional[torch.Tensor] = None, ln_eps: Optional[float] = None,
              ln_weight: Optional[torch.Tensor] = None, ln_bias: Optional[torch.Tensor] = None,
              add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Forward of the reference's mx.Linear (microxscaling/mx/linear.py:20-103) for MXINT8:
    y = A1(A1(MXq(A1(x)) @ MXq(A1(W))^T) + A1(bias)).  ``weight`` is either the (N,K) tensor or
    the operand returned by mx_linear_prepare_weight (then pass out_features).

    ``x``: float32, bfloat16 or float16; the result has x's dtype.  The weight and the bias may each be any of the
    three types, independently of x.  A 16-bit call is the fp32 call on the widened x, weight and bias, its result
    rounded to nearest even (lossless under bfloat 16 for a bf16 x: the fp32 result is a bf16 value), with the same
    kernel launches (no conversion pass).

    adaLN (DiT's DiTBlock, models.py:293-297), for x of shape (B, T, K), each pair optional:
      ``shift``, ``scale`` (B, K): the layer runs on ``x * (1 + scale[:, None]) + shift[:, None]`` (the quantizer
          modulates the elements it loads; nothing is written);
      ``residual`` (B, T, N), ``gate`` (B, N): the result is ``residual + gate[:, None] * y`` (the GEMM's store does it).
    Bit for bit the eager torch composition on tensors of x's dtype, with the launches of the plain call.  The four
    tensors have x's dtype; shift / scale / gate may be column slices of one (B, 6C) tensor (``.chunk(6, dim=1)``).

    Pre-norm block (DeiT's timm Block), for any x, each optional:
      ``ln_eps`` (with ``ln_weight``, ``ln_bias`` (K,) of x's dtype, both or neither): the layer runs on
          ``F.layer_norm(x, (K,), ln_weight, ln_bias, ln_eps)`` (a row statistics kernel, then the quantizer normalizes
          the elements it loads), before any modulation;
      ``add`` (x.shape[:-1] + (N,)): the result is ``add + y`` (the GEMM's store does it); not with residual / gate.
    The result is ``add + f(modulate(F.layer_norm(x)))`` bit for bit, f the plain call; the norm adds one launch."""
    sp = resolve_linear_specs(mx_specs)
    lib = _lib.load()
    x2 = _linear_rows(x)
    if not x.is_cuda:
        raise ValueError("x must be a CUDA tensor; there is no CPU fallback")
    K, M = x2.shape[1], x2.shape[0]
    w_op, N = _weight_operand(weight, K, out_features, mx_specs)
    _check_bias(bias, N)
    _same_device(x, w_op, bias)
    ex = ln_eps is not None or ln_weight is not None or ln_bias is not None or add is not None
    adaln = any(t is not None for t in (shift, scale, residual, gate))
    if ex:
        ad = _ex_args(x, M, K, N, ln_eps, ln_weight, ln_bias, add, shift, scale, residual, gate)
    else:
        ad = _adaln_args(x, K, N, shift, scale, residual, gate) if adaln else ()
    with torch.cuda.device(x.device):
        out = torch.empty((M, N), dtype=x.dtype, device=x.device)
        ws_bytes = (lib.mxp_mx_linear_ex_workspace_bytes if ex else lib.mxp_mx_linear_workspace_bytes)(M, N, K)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=x.device)
        args = (_ptr(x2), DTYPE_CODES[x.dtype], x2.stride(0), M, K, _ptr(w_op), N, _ptr(bias),
                DTYPE_CODES[bias.dtype] if bias is not None else _lib.MXP_DT_F32, sp.bfloat_bits,
                int(sp.flush), _ptr(out), out.stride(0))
        if ex:
            rc = lib.mxp_mx_linear_ex_dt(*args, *ad, _ptr(ws), ws_bytes, _stream())
        elif adaln:
            rc = lib.mxp_mx_linear_adaln_dt(*args, *ad, _ptr(ws), ws_bytes, _stream())
        else:
            rc = lib.mxp_mx_linear_dt(*args, _ptr(ws), ws_bytes, _stream())
    _lib.check(rc, "mxp_mx_linear")
    return out.reshape(*x.shape[:-1], N)


# ---- fused MX MLP -----------------------------------------------------------------------------------------------------
ACTIVATIONS = {"gelu": _lib.MXP_ACT_GELU, "gelu_tanh": _lib.MXP_ACT_GELU_TANH}


def _act_code(act: str) -> int:
    if act not in ACTIVATIONS:
        raise ValueError(f"act must be one of {sorted(ACTIVATIONS)}, got {act!r}")
    return ACTIVATIONS[act]


def mx_mlp(x: torch.Tensor, w1, b1: Optional[torch.Tensor], w2, b2: Optional[torch.Tensor], mx_specs,
           act: str = "gelu", hidden_features: Optional[int] = None, out_features: Optional[int] = None, *,
           shift: Optional[torch.Tensor] = None, scale: Optional[torch.Tensor] = None,
           residual: Optional[torch.Tensor] = None, gate: Optional[torch.Tensor] = None,
           ln_eps: Optional[float] = None, ln_weight: Optional[torch.Tensor] = None,
           ln_bias: Optional[torch.Tensor] = None, add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A transformer MLP (fc1 -> GELU -> fc2) on MX Linear layers, fused:
    ``mx_linear(F.gelu(mx_linear(x, w1, b1), approximate=...), w2, b2)`` bit for bit, with the hidden activation never
    written in a float type (fc1's epilogue applies the GELU and writes fc2's MXINT8 operand).

    ``act``: "gelu" (``approximate='none'``, DeiT) or "gelu_tanh" (``approximate='tanh'``, DiT, PixArt).  ``w1`` / ``w2``:
    the (N1, K) / (N2, N1) weights, or operands from mx_linear_prepare_weight (then pass ``hidden_features`` /
    ``out_features``).  ``x``, weights and biases: the dtype and stride rules of mx_linear; the result has x's dtype.
    K and N1 must be multiples of 64, N2 a multiple of 4.

    ``shift``, ``scale`` (B, K), ``residual`` (B, T, N2), ``gate`` (B, N2): the adaLN arguments of mx_linear for a
    (B, T, K) x, the modulation applied to fc1's input and the gated residual to fc2's output:
    ``residual + gate[:, None] * mlp(x * (1 + scale[:, None]) + shift[:, None])`` bit for bit, same launches.

    ``ln_eps``, ``ln_weight``, ``ln_bias``, ``add``: mx_linear's pre-norm arguments, the norm applied to fc1's input
    and ``add`` (x.shape[:-1] + (N2,)) to fc2's output: ``add + mlp(F.layer_norm(x, (K,), ln_weight, ln_bias, ln_eps))``
    bit for bit."""
    sp = resolve_linear_specs(mx_specs)
    code = _act_code(act)
    lib = _lib.load()
    x2 = _linear_rows(x)
    if not x.is_cuda:
        raise ValueError("x must be a CUDA tensor; there is no CPU fallback")
    K, M = x2.shape[1], x2.shape[0]
    for name, w, k_in in (("w1", w1, K), ("w2", w2, None)):
        if not isinstance(w, torch.Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor")
        if w.dtype != torch.uint8 and (w.dim() != 2 or (k_in is not None and w.shape[1] != k_in)):
            raise ValueError(f"{name}: expected an (out_features, {k_in or 'in_features'}) weight, got {tuple(w.shape)}")
    w1_op, N1 = _weight_operand(w1, K, hidden_features, mx_specs, "hidden_features")
    if w2.dtype != torch.uint8 and w2.shape[1] != N1:
        raise ValueError(f"w2: expected ({w2.shape[0]}, {N1}) for {N1} hidden features, got {tuple(w2.shape)}")
    w2_op, N2 = _weight_operand(w2, N1, out_features, mx_specs)
    _check_bias(b1, N1)
    _check_bias(b2, N2)
    _same_device(x, w1_op, b1, w2_op, b2)
    ex = ln_eps is not None or ln_weight is not None or ln_bias is not None or add is not None
    adaln = any(t is not None for t in (shift, scale, residual, gate))
    if ex:
        ad = _ex_args(x, M, K, N2, ln_eps, ln_weight, ln_bias, add, shift, scale, residual, gate)
    else:
        ad = _adaln_args(x, K, N2, shift, scale, residual, gate) if adaln else ()
    with torch.cuda.device(x.device):
        out = torch.empty((M, N2), dtype=x.dtype, device=x.device)
        ws_bytes = (lib.mxp_mx_mlp_ex_workspace_bytes if ex else lib.mxp_mx_mlp_workspace_bytes)(M, K, N1, N2)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=x.device)
        f32 = _lib.MXP_DT_F32
        args = (_ptr(x2), DTYPE_CODES[x.dtype], x2.stride(0), M, K, _ptr(w1_op), N1, _ptr(b1),
                DTYPE_CODES[b1.dtype] if b1 is not None else f32, code, _ptr(w2_op), N2, _ptr(b2),
                DTYPE_CODES[b2.dtype] if b2 is not None else f32, sp.bfloat_bits, int(sp.flush),
                _ptr(out), out.stride(0))
        if ex:
            rc = lib.mxp_mx_mlp_ex_dt(*args, *ad, _ptr(ws), ws_bytes, _stream())
        elif adaln:
            rc = lib.mxp_mx_mlp_adaln_dt(*args, *ad, _ptr(ws), ws_bytes, _stream())
        else:
            rc = lib.mxp_mx_mlp_dt(*args, _ptr(ws), ws_bytes, _stream())
    _lib.check(rc, "mxp_mx_mlp")
    return out.reshape(*x.shape[:-1], N2)


def activation(x: torch.Tensor, act: str = "gelu") -> torch.Tensor:
    """The fused MLP's activation applied elementwise (parity aid): equals ``torch.nn.functional.gelu(x, approximate=...)``
    on CUDA bit for bit.  ``x``: a contiguous CUDA float32, bfloat16 or float16 tensor; the result has its dtype."""
    code = _act_code(act)
    if not isinstance(x, torch.Tensor) or not x.is_cuda or x.dtype not in DTYPE_CODES or not x.is_contiguous():
        raise ValueError("x must be a contiguous CUDA float32, bfloat16 or float16 tensor")
    with torch.cuda.device(x.device):
        out = torch.empty_like(x)
        rc = _lib.load().mxp_activation_dt(_ptr(x), DTYPE_CODES[x.dtype], x.numel(), code, _ptr(out), _stream())
    _lib.check(rc, "mxp_activation_dt")
    return out
