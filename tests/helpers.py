"""Shared helpers for the parity tests."""
import math
import os

import numpy as np
import torch

from oracle import mxint8_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def mx_specs(bfloat=32, flush=False):
    """The dict the reference's scripts build (workloads/deit/scripts/main.py:719-735)."""
    return {
        'w_elem_format': 'int8', 'a_elem_format': 'int8', 'scale_bits': 8,
        'shared_exp_method': 'max', 'block_size': 32, 'bfloat': bfloat, 'fp': 0,
        'bfloat_subnorms': True, 'round': 'nearest', 'round_mx_output': 'nearest',
        'round_output': 'nearest', 'round_weight': 'nearest',
        'mx_flush_fp32_subnorms': flush, 'custom_cuda': False, 'quantize_backprop': False,
    }


def make_qkv(B, H, N, hd, seed=0, kind="randn", Nk=None):
    """Synthetic activations (SURVEY 8d): randn, per-token log-normal scale spread, edge rows."""
    Nk = N if Nk is None else Nk
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, H, N, hd, generator=g)
    k = torch.randn(B, H, Nk, hd, generator=g)
    v = torch.randn(B, H, Nk, hd, generator=g)
    if kind == "lognormal":
        q = q * torch.exp(1.5 * torch.randn(B, H, N, 1, generator=g))
        k = k * torch.exp(1.5 * torch.randn(B, H, Nk, 1, generator=g))
        v = v * torch.exp(0.5 * torch.randn(B, H, Nk, 1, generator=g))
    if kind == "lognormal05":           # moderate per-token scale spread: key windows of 16-21 bits at long N
        q = q * torch.exp(0.5 * torch.randn(B, H, N, 1, generator=g))
        k = k * torch.exp(0.5 * torch.randn(B, H, Nk, 1, generator=g))
    if kind == "edges":
        q[0, 0, 3 % N] = 0.0
        k[0, 0, 5 % Nk] = 0.0
        if hd > 32:
            q[0, 0, 7 % N, 32:min(64, hd)] = 0.0
        k[0, -1, 2 % Nk, :32] = 0.0
        q[0, -1, 4 % N, :8] = -1e-6
        k[0, -1, 9 % Nk, hd // 2:hd // 2 + 8] = -1e-7
        k[0, 0, 11 % Nk] = k[0, 0, 10 % Nk]
        k[0, 0, 12 % Nk] = k[0, 0, 10 % Nk]
        v[0, 0, 6 % Nk] = 0.0
        # block maxima just below a power of two (fp32 log2 rounds up in the reference)
        q[0, 0, 1 % N, 0] = float(np.nextafter(np.float32(8.0), np.float32(0)))
        k[0, 0, 1 % Nk, 1] = -float(np.nextafter(np.float32(16.0), np.float32(0)))
    return q, k, v


def long_inputs(kind, H, N, hd, seed):
    """q, k (1, H, N, hd) for the long-sequence selection: kinds that stress its sampled window and its key windows."""
    g = torch.Generator().manual_seed(seed)
    q, k = torch.randn(1, H, N, hd, generator=g), torch.randn(1, H, N, hd, generator=g)
    if kind.startswith("lognormal"):
        s = float(kind[len("lognormal"):])
        q = q * torch.exp(s * torch.randn(1, H, N, 1, generator=g))
        k = k * torch.exp(s * torch.randn(1, H, N, 1, generator=g))
    elif kind == "ties":                # few distinct key rows: long runs of equal scores
        k = k[:, :, :7].repeat(1, 1, (N + 6) // 7, 1)[:, :, :N].contiguous()
    elif kind == "constant":            # every key row the same: all scores of a row tie
        k = k[:, :, :1].expand(1, H, N, hd).contiguous()
    elif kind == "zeros":               # zero keys in the second half, zero query rows here and there
        k[:, :, N // 2:] = 0.0
        q[:, :, ::17] = 0.0
    elif kind == "skewed":              # the sampled first keys misrepresent the rest of the row
        k[:, :, :256] *= 0.05
        k[:, :, 256:] += 0.5
    elif kind == "outliers":            # a few huge keys widen the static key window
        k[:, :, 5::511] *= 40.0
        q[:, :, 3::97, :32] *= 0.01
    return q, k


def fused_qkv_views(q, k, v):
    """Re-create the reference's layout: one (B,N,3,H,hd) buffer, q/k/v = permuted views
    (workloads/deit/scripts/main.py:87-88).  Requires Nq == Nk."""
    B, H, N, hd = q.shape
    buf = torch.stack([q, k, v], dim=0).permute(1, 3, 0, 2, 4).contiguous()   # (B,N,3,H,hd)
    qkv = buf.permute(2, 0, 3, 1, 4)
    return qkv[0], qkv[1], qkv[2]


def unpack_mask(mask_i32, n_keys):
    return O.mask_words_to_dense(mask_i32.cpu().to(torch.int64) & 0xFFFFFFFF, n_keys)


def canonical_idx_from_mask(dense, top_k):
    """Kept-key indices (ascending) of a dense bool mask with exactly top_k kept keys per row."""
    return torch.sort(dense.to(torch.int8), dim=-1, descending=True, stable=True).indices[..., :top_k].contiguous()


def load_golden(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    d = {k: torch.from_numpy(z[k].astype(np.int64) if z[k].dtype == np.int16 else z[k]) for k in z.files}
    B, H, N, hd, top_k, bfloat, flush = (int(x) for x in z["meta"])
    return d, dict(B=B, H=H, N=N, hd=hd, top_k=top_k, bfloat=bfloat, flush=bool(flush))


def out_error_budget(ref, v, n_keys, bfloat=32, out_tol=1e-3, rel_window=1e-6):
    """Per-row absolute error budget for the fp32 attention output.

    Base: out_tol * max|ref out| (the stated tolerance).  The reference's P quantizer
    (mx.matmul on the softmax matrix, workloads/deit/scripts/main.py:152) is DISCONTINUOUS in p:
    where p*64/2^e sits within a few ulps of a rounding tie, or a window's max p within a few
    ulps of a power of two (e.g. one-hot rows with p = 1 - 2^-24 vs 1.0), a 1-ulp difference in
    exp()/sum order moves the dequantised P by one code step 2^(e-6).  Any two implementations
    (including the reference's own CPU and CUDA runs) disagree there, so such entries add one
    code step * max|V row| to the row's budget.  Everything else must meet the base tolerance.
    """
    vals, idx, out_ref = ref["true_vals"], ref["idx"], ref["out"]
    p64 = torch.softmax(vals.double(), dim=-1)
    attn = torch.zeros(*vals.shape[:-1], n_keys, dtype=torch.float64)
    attn.scatter_(-1, idx, p64)
    nw = (n_keys + 31) // 32
    pad = nw * 32 - n_keys
    a = torch.nn.functional.pad(attn, (0, pad)).reshape(*attn.shape[:-1], nw, 32)
    amax = a.amax(-1, keepdim=True)
    mant, ex = torch.frexp(amax)                     # amax = mant * 2^ex, mant in [0.5, 1)
    e = (ex - 1).clamp(min=-127)                     # floor(log2(amax))
    step = torch.ldexp(torch.ones_like(amax), e - 6)
    t = a / step                                     # code-domain value
    frac = t - torch.floor(t)
    tie = ((frac - 0.5).abs() <= rel_window * t.clamp(min=1.0)) & (a > 0)
    exp_edge = ((mant > 1 - rel_window) | (mant < 0.5 + rel_window)) & (amax > 0)
    risky = tie | (exp_edge & (a > 0))
    if bfloat == 16:      # A1 rounds P to bf16 first: ties of that rounding are risk points too
        m8, _ = torch.frexp(a)
        f8 = m8 * 256.0 - torch.floor(m8 * 256.0)
        risky = risky | (((f8 - 0.5).abs() <= rel_window * 256.0) & (a > 0))
    vrow = v.abs().amax(-1)                          # (B,H,Nk)
    vrow = torch.nn.functional.pad(vrow, (0, pad)).reshape(*vrow.shape[:-1], nw, 32).unsqueeze(-3)
    extra = (risky.double() * (2 * step) * vrow.double()).sum(dim=(-1, -2))     # (B,H,Nq)
    base = out_tol * float(out_ref.abs().max())
    if bfloat == 16:
        # the output itself is rounded to bf16 (A1, matmul.py:89-91): an fp32 sum within an ulp of a
        # rounding tie lands on either neighbour depending on the summation order - one bf16 ulp of
        # the row's largest output
        extra = extra + 2.0 ** -8 * out_ref.abs().amax(-1).double()
    return base + extra.float()


def assert_out_close(out, ref, v, n_keys, bfloat=32, out_tol=1e-3, max_relaxed_frac=None):
    budget = out_error_budget(ref, v, n_keys, bfloat, out_tol)
    err = (out - ref["out"]).abs().amax(-1)
    bad = err > budget
    base = out_tol * float(ref["out"].abs().max())
    frac_relaxed = float((budget > base * 1.0001).float().mean())
    assert not bool(bad.any()), (
        f"{int(bad.sum())} rows exceed their budget; worst err {float(err.max()):.3e}, base tol {base:.3e}")
    if max_relaxed_frac is not None:     # well-conditioned inputs: almost no row may need the allowance
        assert frac_relaxed <= max_relaxed_frac, f"{frac_relaxed:.1%} of rows needed the code-step allowance"
    return float(err.max()), frac_relaxed


def mode_window_ok(qc, qe, kc, ke, hd, mode, bits=20):
    """Rows of the other rankings (partial_Q / partial_K / MXINT4 / two_step / true_ex / exact) whose EVERY (query, key)
    pair keeps all its block terms inside ``bits`` bits: there the tensor core's fp32 accumulation and the reference's
    BLAS agree in any order (DESIGN.md 2, footnote 1), so the selected sets are pinned.  Operand widths: an MXINT8 side
    adds 7 bits below its block exponent, MXINT4 3, the exponent-sign / leading-one sides none; a block sum adds
    ceil(log2(width)) + 1."""
    side = {"partial_Q": (7, 0), "partial_K": (0, 7), "MXINT4": (3, 3), "two_step_leading_ones": (7, 7), "true_ex": (7, 7),
            "exact": (7, 7), "ex_pred": (0, 0)}[mode]
    eq = O.predictor_exponents(qc, qe).to(torch.int64)
    ek = O.predictor_exponents(kc, ke).to(torch.int64)
    s = eq[..., :, None, :] + ek[..., None, :, :]                      # [..., Nq, Nk, nb]
    widths = torch.tensor([math.ceil(math.log2(w)) + 1 for w in O.block_widths(hd)])
    spread = (s + widths).amax(-1) - s.amin(-1) + side[0] + side[1]
    return (spread <= bits).all(-1)


# ---- guard bands -----------------------------------------------------------------------------------------------------
GUARD_BYTES = 256
CANARY_INT = 0x80       # int8 -128: never a code or an exponent; 0x80808080 is no key index
CANARY_FLOAT = 0xFF     # NaN in fp32, bf16 and fp16: an output element left unwritten fails any comparison


class Guarded:
    """A ``shape`` output of ``dtype`` inside a buffer of canary bytes: GUARD_BYTES before and after it, and
    ``row_pad`` elements after each row (a padded row stride, as an ``out=`` view of a larger buffer has)."""

    def __init__(self, shape, dtype, row_pad=0):
        es = torch.empty((), dtype=dtype).element_size()
        g = GUARD_BYTES // es
        inner = shape[-1] + row_pad
        rows = math.prod(shape[:-1])
        total = 2 * g + rows * inner
        strides, s = [], 1
        for n in reversed((*shape[:-1], inner)):
            strides.insert(0, s)
            s *= n
        self.canary = CANARY_FLOAT if dtype.is_floating_point else CANARY_INT
        self.buf = torch.full((total * es,), self.canary, dtype=torch.uint8, device="cuda")
        self.t = self.buf.view(dtype).as_strided(shape, strides, g)
        covered = torch.zeros(total, dtype=torch.bool, device="cuda")
        covered.as_strided(shape, strides, g).fill_(True)
        self.outside = ~covered.repeat_interleave(es)

    def assert_intact(self, what):
        hit = ((self.buf != self.canary) & self.outside).nonzero().flatten()
        assert hit.numel() == 0, (f"{what}: {hit.numel()} bytes outside the output were written, the first at byte "
                                  f"{int(hit[0]) - GUARD_BYTES} from the output's start")

    def assert_untouched(self, what):
        """Nothing at all was written: every byte, inside the output too, still holds the canary."""
        hit = (self.buf != self.canary).nonzero().flatten()
        assert hit.numel() == 0, f"{what}: {hit.numel()} bytes were written by a call that failed"


def select_guarded(q, k, top_k, bfloat=32):
    """mxp_predict_topk_dt with mask, idx and both code / exponent outputs in guarded buffers.  The guards are checked
    before the return code: a call that fails must not have written past its outputs either.  Returns the outputs on
    the CPU."""
    from mx_quantization_b200 import _lib, ops
    lib = _lib.load()
    B, H, Nq, hd = q.shape
    Nk = k.shape[2]
    nb, nw = (hd + 31) // 32, (Nk + 31) // 32
    g = {"mask": Guarded((B, H, Nq, nw), torch.int32), "idx": Guarded((B, H, Nq, top_k), torch.int32),
         "q_codes": Guarded((B, H, Nq, hd), torch.int8), "q_exps": Guarded((B, H, Nq, nb), torch.int8),
         "k_codes": Guarded((B, H, Nk, hd), torch.int8), "k_exps": Guarded((B, H, Nk, nb), torch.int8)}
    ws_bytes = lib.mxp_predict_topk_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device="cuda")
    p = ops._ptr
    rc = lib.mxp_predict_topk_dt(p(q), *q.stride()[:3], p(k), *k.stride()[:3], ops.DTYPE_CODES[q.dtype], B, H, Nq, Nk,
                                 hd, top_k, bfloat, 0, p(g["mask"].t), p(g["idx"].t), p(g["q_codes"].t),
                                 p(g["q_exps"].t), p(g["k_codes"].t), p(g["k_exps"].t), p(ws), ws_bytes, ops._stream())
    for name, b in g.items():
        b.assert_intact(name)
    _lib.check(rc, "mxp_predict_topk_dt")
    return {name: b.t.cpu() for name, b in g.items()}
