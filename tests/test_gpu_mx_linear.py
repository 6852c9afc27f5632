"""MX Linear (``mx_linear`` / ``MxLinear``: ``k_quantize_gemm_operand``, ``k_round_bias``, ``k_mx_linear_umma``) against
a float64 reference of the same operation, per element, across the persistent tile schedule, the operand layout, the
C ABI's strides and the rounding edges.

Reference.  The operands are the oracle's ``fake_quant_mxint8`` of x and W (quantized on the CPU, then widened to
float64 on the device).  They are exact in bf16, so every product is exact in float64 and ``s = Xq @ Wq^T`` is the
exact dot product.  The kernel accumulates in fp32 on the tensor cores, one ``tcgen05.mma`` of K = 16 after another,
and that accumulation is not round-to-nearest outside a 20-bit window (profiles/r01_umma_exactness_b200.txt).  The
model bounds its error by two fp32 ulps of the magnitude each K = 16 step handles:

    |acc - s| <= beta = 2^-22 * sum_j (|S_(j-1)| + sum_(i in step j) |a_i b_i|)      S_j: exact partial sum after step j

(a global ``(K/16 + 2) * 2^-22 * sum|p|`` is as sound but 40-50x wider at K >= 768, too wide to pin bfloat 16).  The
epilogue ``f(acc) = A1(fl32(A1(acc) + A1(b)))`` (A1 = bf16 round-half-away under bfloat 16, the identity under
bfloat 32) and the 16-bit store (round to nearest even) are monotone, so y must lie in
``[f(rd32(s - beta)), f(ru32(s + beta))]`` element by element.  Away from rounding ties that bracket is one value.
Measured on an NVIDIA B200 at its 1000 W power limit (bfloat 32, no bias, fp32 output, where y is the accumulator
itself): with randn activations every accumulator equals s exactly (block exponents stay close enough for the sums to
fit fp32), up to K = 4096 and at 50 432 x 3 072 -> 768.  With block exponents spread over +-10 (the ``_wide`` cases)
the largest ``|acc - s| / sum|p|`` is 1.7e-6 (2^-19.2, K = 1152) and the largest ``|acc - s| / beta`` is 0.26, a
3.9x headroom under the model.

Exact-sum inputs (values already MXINT8, every block holding a code >= 64, exponents in a narrow window, sum|p| below
2^24 quanta) have an exact fp32 accumulator in any summation order, so there the output must equal ``f(s)`` exactly.
"""
import ctypes
import math

import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import make_qkv, mx_specs

A1 = O.bf16_round_half_away
STEP_ULPS = 2.0 ** -22         # beta per K = 16 step, relative to the magnitude the step handles
DEGENERATE_MIN = 0.94          # bfloat 16: share of single-valued brackets (the test stays effectively bit-exact)


def _m():
    import mx_quantization_b200 as m
    return m


# ------------------------------------------------------------------------------------------------ reference helpers
def quant_ref(t, bfloat, flush, device):
    """The oracle's MX operand of ``t`` (quantized on the CPU: the shared-exponent table is a CPU tensor) as float64."""
    return O.fake_quant_mxint8(t.float().cpu(), bfloat=bfloat, flush_subnorms=flush).to(device=device,
                                                                                         dtype=torch.float64)


def _rd32(v):
    r = v.float()
    return torch.where(r.double() > v, torch.nextafter(r, torch.full_like(r, -math.inf)), r)


def _ru32(v):
    r = v.float()
    return torch.where(r.double() < v, torch.nextafter(r, torch.full_like(r, math.inf)), r)


def epilogue(acc, bias, bfloat):
    """f: fp32 accumulator -> fp32 output, with the oracle's roundings (linear.py:85-93)."""
    y = A1(acc) if bfloat == 16 else acc
    if bias is not None:
        b = bias.float().to(y.device)
        y = y + (A1(b) if bfloat == 16 else b)
        if bfloat == 16:
            y = A1(y)
    return y


def exact_and_bound(xq, wq):
    """s = Xq Wq^T and the step magnitude sum_j (|S_(j-1)| + sum_step |p|), float64, in K = 16 steps."""
    M, K = xq.shape
    s = torch.zeros(M, wq.shape[0], dtype=torch.float64, device=xq.device)
    t = torch.zeros_like(s)
    xa, wa = xq.abs(), wq.abs()
    for k0 in range(0, K, 16):
        t.add_(s.abs())
        t.addmm_(xa[:, k0:k0 + 16], wa[:, k0:k0 + 16].t())
        s.addmm_(xq[:, k0:k0 + 16], wq[:, k0:k0 + 16].t())
    return s, t


def bracket(x, w, bias, bfloat, flush, out_dtype=torch.float32):
    """(lo, hi, s, beta, sum|p|): the elementwise bounds on mx_linear(x, w, bias) in ``out_dtype``, on x's device."""
    dev = x.device
    xq, wq = quant_ref(x, bfloat, flush, dev), quant_ref(w, bfloat, flush, dev)
    s, t = exact_and_bound(xq, wq)
    beta = STEP_ULPS * t
    lo = epilogue(_rd32(s - beta), bias, bfloat).to(out_dtype)
    hi = epilogue(_ru32(s + beta), bias, bfloat).to(out_dtype)
    return lo, hi, s, beta, xq.abs() @ wq.abs().t()


def assert_in_bracket(y, lo, hi, what=""):
    yf, lof, hif = y.float(), lo.float(), hi.float()
    bad = ~((yf >= lof) & (yf <= hif))                      # NaN fails both comparisons
    if bool(bad.any()):
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} outputs outside the bracket; first {i}: y={float(yf[i])!r} "
                             f"bracket [{float(lof[i])!r}, {float(hif[i])!r}]")
    return float((lo == hi).float().mean())


def check_global(y, ref, bfloat):
    """The suite's earlier global statement (tests/test_gpu_parity.py::_check_linear), on an fp32 output."""
    err = (y - ref).abs()
    scale = float(ref.abs().max())
    if bfloat == 32:
        assert float(err.max()) <= 2e-5 * scale, float(err.max()) / scale
    else:
        assert float(err.max()) <= 2.0 ** -7 * scale
        assert float((err > 0).float().mean()) <= 0.02


def random_inputs(M, K, N, bias, seed, x_dtype=torch.float32, device="cuda", spread=0):
    """randn with a log-normal row scale (the activations of a real layer), weights ~ K^-1/2.  ``spread`` > 0 also
    scales each 32-block of x by 2^u, u uniform in [-spread, spread]: with block exponents that far apart the exact
    sums no longer fit in fp32 and the tensor core's accumulation rounding shows."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g) * torch.exp(0.5 * torch.randn(M, 1, generator=g))
    if spread:
        u = torch.randint(-spread, spread + 1, (M, K // 32, 1), generator=g).float()
        x = (x.reshape(M, K // 32, 32) * torch.exp2(u)).reshape(M, K)
    w = torch.randn(N, K, generator=g) * K ** -0.5
    b = torch.randn(N, generator=g) * 0.1 if bias else None
    return x.to(device=device, dtype=x_dtype), w.to(device), (b.to(device) if bias else None)


# ------------------------------------------------------------------------------------------------ exact-sum inputs
EXACT_EXP = (-2, 1)            # block exponents of the exact-sum generator
EXACT_SMALL = 7                # |code| of the elements other than each block's leading one


def exact_operand(rows, K, seed, exp_lo=EXACT_EXP[0], exp_hi=EXACT_EXP[1], small=EXACT_SMALL):
    """(rows, K) fp32 values c * 2^(e-6) that MX-quantize to themselves: every 32-block holds one code of magnitude
    64..127 (so its shared exponent is e) and codes |c| <= ``small`` elsewhere; e in [exp_lo, exp_hi] per block."""
    g = torch.Generator().manual_seed(seed)
    nb = K // 32
    c = torch.randint(-small, small + 1, (rows, nb, 32), generator=g)
    lead = torch.randint(64, 128, (rows, nb, 1), generator=g) * (2 * torch.randint(0, 2, (rows, nb, 1), generator=g) - 1)
    c.scatter_(2, torch.randint(0, 32, (rows, nb, 1), generator=g), lead)
    e = torch.randint(exp_lo, exp_hi + 1, (rows, nb, 1), generator=g)
    return torch.ldexp(c.float(), (e - 6).expand(rows, nb, 32).int()).reshape(rows, K)


def assert_exact_sums(x, w):
    """Every partial sum of every (m, n) dot product is an fp32 value: sum|p| < 2^24 quanta, the quantum being the
    smallest product step 2^(min e_x + min e_w - 12) (e: the block exponents)."""
    def quantum(t):
        amax = t.float().cpu().abs().reshape(t.shape[0], -1, 32).amax(-1)
        return int(O.shared_exponent_from_absmax(amax).min()) - 6
    qx, qw = quantum(x), quantum(w)
    quanta = (x.double().abs() * 2.0 ** -qx) @ (w.double().abs() * 2.0 ** -qw).to(x.device).t()
    assert float(quanta.max()) < 2.0 ** 24, math.log2(float(quanta.max()))


# Rows built to land on rounding ties.  x holds t1 at column 0 and t2 at column 32 (different MX blocks, each value
# its block's only element and an exact MXINT8 value); feature f of W has weights (w0, w1) at those columns and
# bias b.  s = w0 t1 + w1 t2 is exact in fp32.
TIE_ROWS = [(4.0, 2 ** -6),            # 4 (1 + 2^-8): A1 gives 4.03125, round-to-nearest-even 4.0
            (-4.0, -2 ** -6),          # the same value negated
            (4.0, 3 * 2 ** -6),        # 4.046875: a bf16 tie whose even neighbour is above (RNE != truncation)
            (4.0, 2 ** -7),            # with bias 2^-7: 4.0 after the first A1, 4.03125 if the bias came before it
            (4.0, 2 ** -9),            # fp16 tie, even neighbour below
            (4.0, 3 * 2 ** -9),        # fp16 tie, even neighbour above
            (4.0, 3 * 2 ** -7),        # 4.0234375: above the bf16 midpoint (RN up, truncation down)
            (2.0 ** -10, 2.0 ** -18)]  # a tie in another binade (fp16-representable)
TIE_FEATURES = [(1.0, 1.0, 0.0),       # (w0, w1, bias)
                (1.0, 0.0, 2 ** -6),   # A1(4) + 2^-6: a tie in the bias addition
                (1.0, 1.0, 2 ** -7),
                (-1.0, -1.0, -2 ** -6)]


def tie_problem(M=300, N=260, K=64):
    """x (M, K), W (N, K), bias (N): TIE_ROWS cycled over the rows, TIE_FEATURES over the features."""
    x = torch.zeros(M, K)
    for r in range(M):
        x[r, 0], x[r, 32] = TIE_ROWS[r % len(TIE_ROWS)]
    w, b = torch.zeros(N, K), torch.zeros(N)
    for n in range(N):
        w[n, 0], w[n, 32], b[n] = TIE_FEATURES[n % len(TIE_FEATURES)]
    return x, w, b


# ------------------------------------------------------------------------------------------------ CPU
def test_exact_inputs_and_bracket_cpu():
    # the exact-sum generator's values are their own MX quantization, under both bfloat settings and flush
    x, w = exact_operand(300, 4096, 1), exact_operand(64, 4096, 2)
    for bfloat in (16, 32):
        for flush in (False, True):
            assert torch.equal(O.fake_quant_mxint8(x, bfloat=bfloat, flush_subnorms=flush), x)
    assert_exact_sums(x, w)
    # the tie rows give the oracle values the epilogue must reproduce
    xt, wt, bt = tie_problem(M=8, N=4)
    y16 = O.mx_linear(xt, wt, None, bfloat=16)
    assert float(y16[0, 0]) == 4.03125 and float(y16[1, 0]) == -4.03125            # round half away, not RNE (4.0)
    assert float(O.mx_linear(xt, wt, None, bfloat=32)[0, 0]) == 4.015625
    yb = O.mx_linear(xt, wt, bt, bfloat=16)
    assert float(yb[0, 1]) == 4.03125                                               # A1(4 + 2^-6) in the bias add
    assert float(yb[3, 2]) == 4.0                                                    # bias after the first A1
    assert float(yb[1, 3]) == 4.03125                                               # 4.03125 - 2^-6: a tie again
    y32 = O.mx_linear(xt, wt, None, bfloat=32)
    assert y32[2, 0].to(torch.bfloat16).item() == 4.0625                             # fp32 -> bf16 store ties: RNE
    assert y32[4, 0].to(torch.float16).item() == 4.0 and y32[5, 0].to(torch.float16).item() == 4.0 + 2 ** -7
    # the bracket contains the oracle's own CPU mx_linear output (a BLAS summation order)
    for (M, K, N, bias, bfloat, flush) in [(33, 64, 36, True, 16, False), (70, 768, 260, True, 32, False),
                                           (40, 1152, 128, False, 16, True)]:
        xr, wr, br = random_inputs(M, K, N, bias, seed=M, device="cpu")
        lo, hi, *_ = bracket(xr, wr, br, bfloat, flush)
        assert_in_bracket(O.mx_linear(xr, wr, br, bfloat=bfloat, flush=flush), lo, hi, "oracle")


# ------------------------------------------------------------------------------------------------ GPU: shape matrix
def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def tile_shape(tiles, exact=True):
    """(M, N) with ragged last row and feature tiles and ``tiles`` 128 x 256 output tiles (the first count at or above
    ``tiles`` with a feature-tile divisor in 2..12 when not ``exact``); N = 4 mod 32."""
    t = tiles
    while True:
        tn = max([d for d in range(1, 13) if t % d == 0])
        if exact or tn > 1:
            break
        t += 1
    tm = t // tn
    M, N = tm * 128 - 37 if tm > 1 else 91, tn * 256 - 28
    assert (-(-M // 128)) * (-(-N // 256)) == t
    return M, N


def _resolve(M, N):
    """Shape entries "S-1" / "S" / "S+1" / "7S+3": tile counts around the SM count S (M and N are then derived)."""
    if isinstance(M, str):
        S = _sms()
        t = {"S-1": S - 1, "S": S, "S+1": S + 1, "7S+3": 7 * S + 3}[M]
        return tile_shape(t, exact=M != "7S+3")
    return M, N


F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
# M, K, N, x dtype, bfloat, bias, flush
RANDOM_CASES = [
    (1, 64, 4, F32, 32, False, False),          # M = 1; one k step (fewer than the 4 stages)
    (127, 192, 252, BF16, 16, True, False),     # 3 k steps
    (128, 256, 256, F32, 32, True, True),       # 4 k steps, flush
    (129, 320, 260, F16, 32, True, False),      # 5 k steps, N = 4 mod 32, a 1-row second row tile
    (257, 768, 1020, F32, 16, False, False),
    (300, 4096, 2304, F32, 32, False, False),   # 64 k steps
    ("S-1", 1152, None, F32, 32, False, False),  # 18 k steps (not a multiple of the 4 stages)
    ("S", 320, None, BF16, 16, True, True),
    ("S+1", 768, None, F16, 32, True, False),   # one CTA takes two tiles
    ("7S+3", 3072, None, F32, 32, False, False),  # about 7 tiles per CTA: accumulator parity and stage ring wrap
    ("7S+3", 1152, None, BF16, 16, True, False),
    (300, 3072, 2304, F32, 32, False, False, 10),   # block exponents 20 bits apart: inexact fp32 accumulation
    ("S+1", 1152, None, F32, 32, False, False, 10),
    ("7S+3", 768, None, BF16, 16, True, False, 10),
]


def _case_id(c):
    return (f"{c[0]}x{c[1]}to{c[2] or 'N'}_{str(c[3])[6:]}_bf{c[4]}{'_bias' if c[5] else ''}{'_flush' if c[6] else ''}"
            f"{'_wide' if len(c) > 7 else ''}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", RANDOM_CASES, ids=_case_id)
def test_random_inputs_in_bracket(case):
    m = _m()
    M, K, N, dt, bfloat, bias, flush = case[:7]
    M, N = _resolve(M, N)
    x, w, b = random_inputs(M, K, N, bias, seed=K + N, x_dtype=dt, spread=case[7] if len(case) > 7 else 0)
    sp = mx_specs(bfloat, flush)
    y = m.mx_linear(x, w, b, sp)
    assert y.dtype == dt and y.shape == (M, N)
    lo, hi, s, beta, sump = bracket(x, w, b, bfloat, flush, dt)
    deg = assert_in_bracket(y, lo, hi, _case_id(case))
    if dt == F32:
        check_global(y, epilogue(s.float(), b, bfloat), bfloat)
    else:
        y32 = m.mx_linear(x.float(), w, b, sp)                 # the 16-bit output is the fp32 call rounded
        assert torch.equal(y, y32.to(dt))
        check_global(y32, epilogue(s.float(), b, bfloat), bfloat)
    if bfloat == 16 and M * N >= 4096:
        assert deg >= DEGENERATE_MIN, f"only {deg:.1%} of the brackets are single values"
    if bfloat == 32 and b is None and dt == F32:            # y is the fp32 accumulator itself
        _record_ratio(_case_id(case), K, y, s, beta, sump)


def _record_ratio(name, K, y, s, beta, sump):
    """Print the accumulation error of an output that is the fp32 accumulator itself, against sum|p| and the model."""
    err = (y.double() - s).abs()
    nz = sump > 0
    r_sum = float((err[nz] / sump[nz]).max())
    r_beta = float((err[nz] / beta[nz]).max())
    print(f"\n[mx_linear accumulation] {name} K={K}: max |acc-s|/sum|p| = {r_sum:.3e} "
          f"(2^{math.log2(r_sum) if r_sum > 0 else -math.inf:.1f}), max |acc-s|/beta = {r_beta:.3e}")


# ------------------------------------------------------------------------------------------------ GPU: exact sums
# M, K, N, x dtype, bfloat, bias, flush
EXACT_CASES = [
    (1, 64, 4, BF16, 16, True, False),
    (129, 192, 260, F32, 32, True, False),
    (257, 4096, 1020, F16, 32, False, True),
    ("S+1", 1152, None, F32, 16, True, False),
    ("7S+3", 320, None, BF16, 32, True, False),
    (50432, 768, 2304, F32, 32, True, False),      # DeiT-base qkv
    (65536, 1152, 1152, BF16, 16, True, False),    # DiT-XL/2 projection
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EXACT_CASES, ids=_case_id)
def test_exact_sums_bit_exact(case):
    m = _m()
    M, K, N, dt, bfloat, bias, flush = case
    M, N = _resolve(M, N)
    x = exact_operand(M, K, seed=M + K).cuda()
    w = exact_operand(N, K, seed=N + K + 1).cuda()
    b = (torch.randn(N, generator=torch.Generator().manual_seed(N)) * 0.1).cuda() if bias else None
    assert torch.equal(O.fake_quant_mxint8(x[:64].cpu(), bfloat=bfloat, flush_subnorms=flush), x[:64].cpu())
    assert_exact_sums(x, w)
    s = x.double() @ w.double().t()
    want = epilogue(s.float(), b, bfloat).to(dt)
    xin = x.to(dt)
    assert torch.equal(xin.float(), x)                     # the exact values are bf16 / fp16 values too
    y = m.mx_linear(xin, w, b, mx_specs(bfloat, flush))
    assert torch.equal(y, want), f"{int((y != want).sum())} of {y.numel()} outputs differ"


@pytest.mark.gpu
@pytest.mark.parametrize("bfloat", [16, 32])
def test_rounding_ties(bfloat):
    """Ties of A1 after the accumulator, of A1 after the bias addition, and of the fp32 -> bf16 / fp16 store, over
    three row tiles and two feature tiles, in every output type."""
    m = _m()
    x, w, b = tie_problem()
    s = x.double() @ w.double().t()
    sp = mx_specs(bfloat)
    for dt in (F32, BF16, F16):
        assert torch.equal(x.to(dt).float(), x)                     # the tie rows are exact in every input type
    for bias in (None, b):
        want = epilogue(s.float(), bias, bfloat)
        for dt in (F32, BF16, F16):
            y = m.mx_linear(x.to(dt).cuda(), w.cuda(), None if bias is None else bias.cuda(), sp)
            assert torch.equal(y.cpu(), want.to(dt)), (dt, bias is not None, (y.cpu() != want.to(dt)).nonzero()[:4])
    assert float(epilogue(s.float(), None, 16)[0, 0]) == 4.03125


@pytest.mark.gpu
@pytest.mark.parametrize("bfloat", [16, 32])
def test_permutation_weight(bfloat):
    """W a row-selection of the identity, no bias: y is the oracle's dequantized x with its columns permuted, bit for
    bit (the activation operand and the epilogue's column mapping)."""
    m = _m()
    M, K, N = 300, 768, 260
    g = torch.Generator().manual_seed(5)
    x = torch.randn(M, K, generator=g) * torch.exp(1.5 * torch.randn(M, 1, generator=g))
    perm = torch.randperm(K, generator=g)[:N]
    w = torch.zeros(N, K)
    w[torch.arange(N), perm] = 1.0
    y = m.mx_linear(x.cuda(), w.cuda(), None, mx_specs(bfloat))
    want = O.fake_quant_mxint8(x, bfloat=bfloat)[:, perm]
    assert torch.equal(y.cpu(), want)


# ------------------------------------------------------------------------------------------------ GPU: production shapes
PRODUCTION = [  # M, K, N, bfloat, bias
    (50432, 768, 2304, 32, True),      # DeiT-base qkv
    (50432, 3072, 768, 32, False),     # DeiT-base fc2
    (65536, 1152, 1152, 16, True),     # DiT-XL/2
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PRODUCTION, ids=lambda s: f"{s[0]}x{s[1]}to{s[2]}_bf{s[3]}")
def test_production_shapes(shape):
    m = _m()
    M, K, N, bfloat, bias = shape
    sp = mx_specs(bfloat)
    x, w, b = random_inputs(M, K, N, bias, seed=K)
    y = m.mx_linear(x, w, b, sp)
    lo, hi, s, beta, sump = bracket(x, w, b, bfloat, False)
    deg = assert_in_bracket(y, lo, hi, f"production {shape}")
    check_global(y, epilogue(s.float(), b, bfloat), bfloat)
    if bfloat == 16:
        assert deg >= DEGENERATE_MIN
    if b is None:
        _record_ratio(f"{M}x{K}to{N}", K, y, s, beta, sump)
    del lo, hi, s, beta, sump
    assert torch.equal(m.mx_linear(x, w, b, sp), y)                                   # repeated calls
    # row independence: an element's MMA sequence does not depend on its output tile
    assert torch.equal(m.mx_linear(x[12345:12645], w, b, sp), y[12345:12645])
    bs = None if b is None else b[100:400]
    assert torch.equal(m.mx_linear(x, w[100:400], bs, sp), y[:, 100:400])
    for dt in (BF16, F16):
        xh = x.to(dt)
        assert torch.equal(m.mx_linear(xh, w, b, sp), m.mx_linear(xh.float(), w, b, sp).to(dt))


# ------------------------------------------------------------------------------------------------ GPU: operand layout
def decode_operand(op, rows, K, rows_tile):
    """[row tile][k step of 64][8 chunks][tile rows][8 bf16] bytes -> (rows_pad, K) bf16 bit patterns (int16), with
    -0 read as +0 (the quantizer keeps the input's sign on a zero code; the oracle's zero is +0)."""
    tiles = -(-rows // rows_tile)
    v = op[: tiles * rows_tile * K * 2].view(torch.int16).reshape(tiles, K // 64, 8, rows_tile, 8)
    bits = v.permute(0, 3, 1, 2, 4).reshape(tiles * rows_tile, K)
    return torch.where(bits == -32768, torch.zeros_like(bits), bits)


def _oracle_bits(t, bfloat, flush, rows_pad):
    q = O.fake_quant_mxint8(t.float().cpu(), bfloat=bfloat, flush_subnorms=flush).to(torch.bfloat16)
    assert torch.equal(q.float(), O.fake_quant_mxint8(t.float().cpu(), bfloat=bfloat, flush_subnorms=flush))
    out = torch.zeros(rows_pad, t.shape[1], dtype=torch.int16)
    out[: t.shape[0]] = q.view(torch.int16)
    return out


def _edge_weight():
    """Rows with zero blocks, -1e-7 blocks, block maxima just below a power of two, and fp32-subnormal blocks."""
    q, k, _ = make_qkv(1, 2, 130, 128, seed=3, kind="edges")
    w = torch.cat([q.reshape(-1, 128), k.reshape(-1, 128)])                 # 520 x 128
    g = torch.Generator().manual_seed(4)
    w[17, :32] = torch.randint(-127, 128, (32,), generator=g).float() * 2.0 ** -133    # block exponent -127
    w[18, 32:64] = torch.randint(-63, 64, (32,), generator=g).float() * 2.0 ** -132    # bf16-subnormal codes
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, BF16, F16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("bfloat,flush", [(32, False), (16, False), (32, True)])
def test_prepared_weight_decodes_to_oracle(dt, bfloat, flush):
    m = _m()
    sp = mx_specs(bfloat, flush)
    for w in (_edge_weight(), random_inputs(1, 320, 1020, False, seed=9, device="cpu")[1] * 37.0):
        wd = w.to(dt)
        N, K = w.shape
        op = m.mx_linear_prepare_weight(wd.cuda(), sp).cpu()
        npad = -(-N // 256) * 256
        assert op.numel() == npad * K * 2
        assert torch.equal(decode_operand(op, N, K, 256), _oracle_bits(wd, bfloat, flush, npad))   # rows >= N: zero


# ------------------------------------------------------------------------------------------------ GPU: C ABI guard bands
SENT32, SENT16, SENT8 = 0x7FA5A5A5, 0x7E5A, 0xA5


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, BF16, F16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("M,K,N,bias,bfloat", [(129, 192, 260, True, 16), (300, 320, 1020, False, 32),
                                               (1, 64, 4, True, 32)])
def test_c_abi_strides_and_guard_bands(dt, M, K, N, bias, bfloat):
    """ldx > K and ldw > K with NaN in the pad columns and in extra rows; ldo > N and extra output rows holding a
    sentinel; the weight operand and the workspace exactly their *_bytes sizes followed by sentinel bytes.  Nothing
    is read past K or M, nothing written past N or M, and the activation operand in the workspace is the oracle's."""
    m = _m()
    from mx_quantization_b200 import _lib
    from mx_quantization_b200.ops import DTYPE_CODES
    lib = _lib.load()
    sp = mx_specs(bfloat)
    x, w, b = random_inputs(M, K, N, bias, seed=M + N, x_dtype=dt)
    w = w.to(dt)
    code = DTYPE_CODES[dt]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    ldx, ldw, ldo = K + 24, K + 40, N + 12
    xb = torch.full((M + 3, ldx), math.nan, dtype=dt, device="cuda")
    xb[:M, :K] = x
    wb = torch.full((N + 5, ldw), math.nan, dtype=dt, device="cuda")
    wb[:N, :K] = w
    wbytes, wsbytes = lib.mxp_mx_linear_weight_bytes(N, K), lib.mxp_mx_linear_workspace_bytes(M, N, K)
    w_op = torch.full((wbytes + 512,), SENT8, dtype=torch.uint8, device="cuda")
    ws = torch.full((wsbytes + 512,), SENT8, dtype=torch.uint8, device="cuda")
    ob = torch.empty((M + 2, ldo), dtype=dt, device="cuda")
    ob.view(torch.int32 if dt == F32 else torch.int16).fill_(SENT32 if dt == F32 else SENT16)
    sent = ob.clone()

    rc = lib.mxp_mx_linear_prepare_weight_dt(ctypes.c_void_p(wb.data_ptr()), code, ldw, N, K, bfloat, 0,
                                             ctypes.c_void_p(w_op.data_ptr()), stream)
    _lib.check(rc, "prepare")
    rc = lib.mxp_mx_linear_dt(ctypes.c_void_p(xb.data_ptr()), code, ldx, M, K, ctypes.c_void_p(w_op.data_ptr()), N,
                              ctypes.c_void_p(0 if b is None else b.data_ptr()), _lib.MXP_DT_F32, bfloat, 0,
                              ctypes.c_void_p(ob.data_ptr()), ldo, ctypes.c_void_p(ws.data_ptr()), wsbytes, stream)
    _lib.check(rc, "mx_linear")
    torch.cuda.synchronize()

    y = ob[:M, :N]
    assert torch.isfinite(y).all()
    assert torch.equal(y, m.mx_linear(x, w, b, sp))
    assert torch.equal(w_op[:wbytes], m.mx_linear_prepare_weight(w, sp))
    inside = torch.zeros_like(ob, dtype=torch.bool)
    inside[:M, :N] = True
    iv = (lambda t: t.view(torch.int32 if dt == F32 else torch.int16))
    assert torch.equal(iv(ob)[~inside], iv(sent)[~inside]), "a store landed outside the M x N output"
    assert bool((w_op[wbytes:] == SENT8).all()), "the weight quantizer wrote past mxp_mx_linear_weight_bytes"
    assert bool((ws[wsbytes:] == SENT8).all()), "mx_linear wrote past mxp_mx_linear_workspace_bytes"
    mpad = -(-M // 128) * 128
    assert torch.equal(decode_operand(ws.cpu(), M, K, 128), _oracle_bits(x, bfloat, False, mpad))


# ------------------------------------------------------------------------------------------------ GPU: weight cache
@pytest.mark.gpu
def test_weight_cache_follows_in_place_updates():
    from mx_quantization_b200.modules import MxLinear
    M, K, N, bfloat = 300, 768, 1020, 16
    sp = mx_specs(bfloat)
    x, w, b = random_inputs(M, K, N, True, seed=21)
    lin = MxLinear(K, N, mx_specs=sp).cuda()
    with torch.no_grad():
        lin.weight.copy_(w)
        lin.bias.copy_(b)
        lin(x)
        lin.weight.mul_(0.5)
        y_mul = lin(x)
        w2 = random_inputs(1, K, N, False, seed=22)[1]
        lin.weight.copy_(w2)
        y_copy = lin(x)
    for y, wn in ((y_mul, w * 0.5), (y_copy, w2)):
        lo, hi, *_ = bracket(x, wn, b, bfloat, False)
        assert_in_bracket(y, lo, hi, "cache")
        assert torch.equal(y, _m().mx_linear(x, wn, b, sp))


# ------------------------------------------------------------------------------------------------ GPU: subnormal operands
@pytest.mark.gpu
@pytest.mark.parametrize("flush", [False, True])
@pytest.mark.parametrize("bfloat", [32, 16])
def test_subnormal_operands(bfloat, flush):
    """The reference's behaviour (bfloat_subnorms=True): blocks with exponents -127..-124 give bf16-subnormal
    operands (every code at e = -127, codes below 64 at e = -126) and, times weights near 1, fp32-subnormal products
    and sums.  The kernel's output equals f(s) of the oracle's operands exactly (every partial sum is an fp32 value)."""
    m = _m()
    M, K, N = 256, 256, 260
    g = torch.Generator().manual_seed(11)
    c = torch.randint(-127, 128, (M, K), generator=g).float()
    e = torch.tensor([-127, -126, -125, -124]).repeat(2).repeat_interleave(32)        # block exponents
    x = c * torch.pow(2.0, (e - 6).float())
    x[:, 32:64] = torch.randint(-63, 64, (M, 32), generator=g).float() * 2.0 ** -132  # all codes < 64 at e = -126
    w = exact_operand(N, K, seed=12, exp_lo=0, exp_hi=0)
    w[N // 2:] *= 2.0 ** 60                                                   # normal products for these features
    xq = quant_ref(x, bfloat, flush, "cpu")
    wq = quant_ref(w, bfloat, flush, "cpu")
    assert_exact_sums(xq, wq[: N // 2])
    assert_exact_sums(xq, wq[N // 2:])
    want = epilogue((xq @ wq.t()).float(), None, bfloat)
    assert bool((want[:, N // 2:] != 0).all())
    if not flush:
        assert bool((want[:, : N // 2].abs() < 2.0 ** -126).any())           # fp32-subnormal outputs
    y = m.mx_linear(x.cuda(), w.cuda(), None, mx_specs(bfloat, flush)).cpu()
    bad = y != want
    assert not bool(bad.any()), (f"{int(bad.sum())} of {y.numel()} outputs differ; first "
                                 f"{[(tuple(i.tolist()), float(y[tuple(i)]), float(want[tuple(i)])) for i in bad.nonzero()[:3]]}")

