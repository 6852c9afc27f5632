"""LayerNorm inside the MX Linear operand quantizer: ``ops.layer_norm`` (the row statistics kernel's parity aid) against
``torch.native_layer_norm`` bit for bit, ``mx_linear`` / ``mx_mlp`` with ``ln_eps`` / ``ln_weight`` / ``ln_bias`` and
``add`` against the torch composition with torch.equal, guard bytes around the output and the workspace, the launches,
and the rejections of malformed arguments."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import mx_specs

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["fp32", "bf16", "fp16"]
KS = [64, 96, 100, 768, 1152, 2048, 4096]       # multiples of 4: the rows torch's vectorized kernel takes
MS = [1, 127, 128, 129, 4096]
ROW_KINDS = ["randn", "offset", "constant", "outlier", "tiny"]


def _m():
    import mx_quantization_b200 as m
    return m


def _rows(kind, M, K, g):
    x = torch.randn(M, K, generator=g, dtype=torch.float64)
    if kind == "offset":            # Welford's update order decides the low bits of the mean and the variance
        x = 1e3 + x
    elif kind == "constant":
        x = torch.randn(M, 1, generator=g, dtype=torch.float64).expand(M, K).clone()
    elif kind == "outlier":
        x[torch.arange(M), torch.randint(0, K, (M,), generator=g)] = 1e4
    elif kind == "tiny":
        x = x * 1e-20
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("kind", ROW_KINDS)
def test_layer_norm_equals_torch(dt, K, kind):
    """y, mean and rstd against torch.native_layer_norm, every M, eps 1e-5 and 1e-6, affine (random weight and bias)
    and not."""
    m = _m()
    g = torch.Generator().manual_seed(K)
    for M in MS:
        x = _rows(kind, M, K, g).to(dt).cuda()
        w = (1 + 0.5 * torch.randn(K, generator=g)).to(dt).cuda()
        b = (0.5 * torch.randn(K, generator=g)).to(dt).cuda()
        for eps in (1e-5, 1e-6):
            for weight, bias in ((w, b), (None, None)):
                want = torch.native_layer_norm(x, (K,), weight, bias, eps)
                got = m.layer_norm(x, weight, bias, eps)
                for gt, wt, name in zip(got, want, ("y", "mean", "rstd")):
                    assert gt.dtype == wt.dtype and gt.shape == wt.shape, name
                    assert torch.equal(gt, wt), (name, M, eps, weight is not None)


# ---------------------------------------------------------------------------------------------- mx_linear / mx_mlp
def _norm_params(K, dt, seed):
    g = torch.Generator().manual_seed(seed)
    return (1 + 0.5 * torch.randn(K, generator=g)).to(dt).cuda(), (0.5 * torch.randn(K, generator=g)).to(dt).cuda()


def _block_inputs(B, T, K, N, dt, seed):
    """x (B, T, K) with a per-row offset and scale; shift / scale / gate column slices; residual and add (B, T, N)."""
    g = torch.Generator().manual_seed(seed)
    x = 3 + torch.randn(B, T, K, generator=g) * torch.exp(torch.randn(B, T, 1, generator=g))
    table = torch.randn(B, 6 * K, generator=g) * 0.5
    gtab = torch.randn(B, 2 * N, generator=g)
    residual, add = torch.randn(B, T, N, generator=g), torch.randn(B, T, N, generator=g)
    x, table, gtab, residual, add = (t.cuda().to(dt) for t in (x, table, gtab, residual, add))
    shift, scale = table.chunk(6, dim=1)[:2]
    return x, shift, scale, residual, gtab[:, N:], add


def _modulate(x, shift, scale):
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)


def _cases(x, shift, scale, residual, gate, add, K, w, b):
    """(kwargs, the input the plain call takes, the torch expression applied to its output) for every combination of
    the norm (affine or not) with the modulation and with add or the gated residual."""
    for ln in (dict(ln_eps=1e-5, ln_weight=w, ln_bias=b), dict(ln_eps=1e-6)):
        xn = F.layer_norm(x, (K,), ln.get("ln_weight"), ln.get("ln_bias"), ln["ln_eps"])
        for mod in (False, True):
            kw_mod = dict(shift=shift, scale=scale) if mod else {}
            xin = _modulate(xn, shift, scale) if mod else xn
            yield dict(ln, **kw_mod), xin, (lambda y: y)
            yield dict(ln, **kw_mod, add=add), xin, (lambda y: add + y)
            yield dict(ln, **kw_mod, residual=residual, gate=gate), xin, (lambda y: residual + gate.unsqueeze(1) * y)
    yield dict(add=add), x, (lambda y: add + y)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
def test_mx_linear_layer_norm_equals_composition(dt, bfloat, flush):
    """K = 192, N = 260 (a partial column tile), T = 100 (a partial last row tile); raw and prepared weights, with and
    without a bias."""
    m = _m()
    sp = mx_specs(bfloat, flush)
    B, T, K, N = 3, 100, 192, 260
    x, shift, scale, residual, gate, add = _block_inputs(B, T, K, N, dt, seed=bfloat + int(flush))
    lw, lb = _norm_params(K, dt, seed=1)
    g = torch.Generator().manual_seed(2)
    w = (torch.randn(N, K, generator=g) * K ** -0.5).cuda()
    bias = (torch.randn(N, generator=g) * 0.5).cuda()
    w_op = m.mx_linear_prepare_weight(w, sp)
    for weight, bb, nf in ((w, bias.to(dt), None), (w_op, None, N)):
        for kw, xin, post in _cases(x, shift, scale, residual, gate, add, K, lw, lb):
            want = post(m.mx_linear(xin, weight, bb, sp, out_features=nf))
            got = m.mx_linear(x, weight, bb, sp, out_features=nf, **kw)
            assert got.dtype == dt and got.shape == (B, T, N)
            assert torch.equal(got, want), sorted(kw)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
def test_mx_mlp_layer_norm_equals_composition(dt, bfloat, flush):
    """K = 192, N1 = 320, N2 = 260, T = 100; raw and prepared weights, with and without biases."""
    m = _m()
    sp = mx_specs(bfloat, flush)
    B, T, K, N1, N2 = 3, 100, 192, 320, 260
    x, shift, scale, residual, gate, add = _block_inputs(B, T, K, N2, dt, seed=7 + bfloat + int(flush))
    lw, lb = _norm_params(K, dt, seed=3)
    g = torch.Generator().manual_seed(4)
    w1, w2 = (torch.randn(N1, K, generator=g) * K ** -0.5).cuda(), (torch.randn(N2, N1, generator=g) * N1 ** -0.5).cuda()
    b1, b2 = (torch.randn(N1, generator=g) * 0.5).cuda(), (torch.randn(N2, generator=g) * 0.5).cuda()
    ops1 = (w1, b1.to(dt), w2, b2, {})
    ops2 = (m.mx_linear_prepare_weight(w1, sp), None, m.mx_linear_prepare_weight(w2, sp), None,
            dict(hidden_features=N1, out_features=N2))
    for a1, bb1, a2, bb2, fkw in (ops1, ops2):
        for kw, xin, post in _cases(x, shift, scale, residual, gate, add, K, lw, lb):
            want = post(m.mx_mlp(xin, a1, bb1, a2, bb2, sp, act="gelu", **fkw))
            got = m.mx_mlp(x, a1, bb1, a2, bb2, sp, act="gelu", **fkw, **kw)
            assert got.dtype == dt and got.shape == (B, T, N2)
            assert torch.equal(got, want), sorted(kw)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_layer_norm_on_row_strided_2d_x(dt):
    """A 2-D x whose rows are a column slice of a wider tensor (row stride 2K), 2-D add."""
    m = _m()
    sp = mx_specs(32)
    M, K, N = 300, 128, 96
    g = torch.Generator().manual_seed(5)
    wide = (2 + torch.randn(M, 2 * K, generator=g)).to(dt).cuda()
    x = wide[:, K:]
    assert x.stride() == (2 * K, 1)
    lw, lb = _norm_params(K, dt, seed=6)
    add = torch.randn(M, N, generator=g).to(dt).cuda()
    w = (torch.randn(N, K, generator=g) * K ** -0.5).cuda()
    want = add + m.mx_linear(F.layer_norm(x, (K,), lw, lb, 1e-5), w, None, sp)
    assert torch.equal(m.mx_linear(x, w, None, sp, ln_eps=1e-5, ln_weight=lw, ln_bias=lb, add=add), want)
    y, mean, rstd = m.layer_norm(x, lw, lb, 1e-5)
    want = torch.native_layer_norm(x, (K,), lw, lb, 1e-5)
    assert all(torch.equal(a, b) for a, b in zip((y, mean, rstd), want))


# ---------------------------------------------------------------------------------------------- guards and launches
def _guarded(n_bytes, dev):
    """A byte buffer with 256 guard bytes of 0xA5 either side; returns (whole, interior)."""
    whole = torch.full((n_bytes + 512,), 0xA5, dtype=torch.uint8, device=dev)
    return whole, whole[256:256 + n_bytes]


def _lib_call(name, *args):
    from mx_quantization_b200 import _lib
    lib = _lib.load()
    rc = getattr(lib, name)(*args)
    _lib.check(rc, name)
    return lib.mxp_last_launch_count()


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
def test_ex_calls_keep_guard_bytes_and_count_launches(dt):
    """The C entry points on guarded output and workspace buffers: the bytes around them survive, the output equals
    ops', and the launches are the plain call's plus one for the norm."""
    from mx_quantization_b200 import _lib
    from mx_quantization_b200.ops import DTYPE_CODES
    m = _m()
    sp = mx_specs(16)
    dev = torch.device("cuda")
    M, K, N1, N2 = 200, 192, 320, 260
    esz = torch.empty((), dtype=dt).element_size()
    g = torch.Generator().manual_seed(8)
    x = (1 + torch.randn(M, K, generator=g)).to(dt).cuda()
    add = torch.randn(M, N2, generator=g).to(dt).cuda()
    lw, lb = _norm_params(K, dt, seed=9)
    w1, w2 = (torch.randn(N1, K, generator=g) * 0.1).cuda(), (torch.randn(N2, N1, generator=g) * 0.1).cuda()
    w1_op, w2_op = m.mx_linear_prepare_weight(w1, sp), m.mx_linear_prepare_weight(w2, sp)
    lib = _lib.load()
    dtc, f32 = DTYPE_CODES[dt], _lib.MXP_DT_F32
    no_adaln = [M] + [None, 0] * 4
    for name, ws_fn, ws_args, head, N in (
            ("mxp_mx_linear_ex_dt", lib.mxp_mx_linear_ex_workspace_bytes, (M, N1, K),
             lambda out: [_p(x), dtc, K, M, K, _p(w1_op), N1, None, f32, 16, 0, _p(out), N1], N1),
            ("mxp_mx_mlp_ex_dt", lib.mxp_mx_mlp_ex_workspace_bytes, (M, K, N1, N2),
             lambda out: [_p(x), dtc, K, M, K, _p(w1_op), N1, None, f32, _lib.MXP_ACT_GELU, _p(w2_op), N2, None, f32,
                          16, 0, _p(out), N2], N2)):
        ws_bytes = ws_fn(*ws_args)
        ws_whole, ws = _guarded(ws_bytes, dev)
        assert ws.data_ptr() % 256 == 0             # the allocation is; 256 guard bytes keep the interior so
        out_whole, out_b = _guarded(M * N * esz, dev)
        out = out_b.view(dt).view(M, N)
        adaln = list(no_adaln)
        if name == "mxp_mx_mlp_ex_dt":
            adaln[5:7] = [_p(add), N2]
        launches = _lib_call(name, *head(out), 1, _p(lw), _p(lb), ctypes.c_float(1e-5), *adaln, _p(ws), ws_bytes, None)
        torch.cuda.synchronize()
        for whole, n in ((ws_whole, ws_bytes), (out_whole, M * N * esz)):
            assert bool((whole[:256] == 0xA5).all()) and bool((whole[256 + n:] == 0xA5).all()), name
        if name == "mxp_mx_linear_ex_dt":
            want = m.mx_linear(x, w1_op, None, sp, out_features=N1, ln_eps=1e-5, ln_weight=lw, ln_bias=lb)
            assert launches == 3                    # statistics, quantizer, GEMM
        else:
            want = m.mx_mlp(x, w1_op, None, w2_op, None, sp, hidden_features=N1, out_features=N2, ln_eps=1e-5,
                            ln_weight=lw, ln_bias=lb, add=add)
            assert launches == 4                    # statistics, quantizer, fc1, fc2
        assert torch.equal(out, want)
    # ops: one launch more than the plain call with the norm, none more for add
    m.mx_linear(x, w1_op, None, sp, out_features=N1)
    plain = m.last_launch_count()
    m.mx_linear(x, w1_op, None, sp, out_features=N1, ln_eps=1e-5)
    assert m.last_launch_count() == plain + 1
    m.mx_mlp(x, w1_op, None, w2_op, None, sp, hidden_features=N1, out_features=N2, add=add)
    assert m.last_launch_count() == 3
    m.layer_norm(x, lw, lb)
    assert m.last_launch_count() == 1


@pytest.mark.gpu
def test_layer_norm_arguments_rejections_leave_no_cuda_error():
    m = _m()
    sp = mx_specs(32)
    B, T, K, N = 2, 64, 128, 64
    x, shift, scale, residual, gate, add = _block_inputs(B, T, K, N, torch.float32, seed=11)
    lw, lb = _norm_params(K, torch.float32, seed=12)
    w = (torch.randn(N, K) * 0.1).cuda()
    bad = [
        dict(ln_eps=1e-5, ln_weight=lw),                                    # weight without bias
        dict(ln_eps=1e-5, ln_bias=lb),                                      # bias without weight
        dict(ln_weight=lw, ln_bias=lb),                                     # affine parameters without eps
        dict(ln_eps=-1.0),
        dict(ln_eps=float("nan")),
        dict(ln_eps=1e-5, ln_weight=lw.half(), ln_bias=lb.half()),          # not x's dtype
        dict(ln_eps=1e-5, ln_weight=lw[:K // 2], ln_bias=lb[:K // 2]),      # wrong shape
        dict(ln_eps=1e-5, ln_weight=torch.randn(2 * K, device="cuda")[::2], ln_bias=lb),   # strided
        dict(ln_eps=1e-5, ln_weight=torch.randn(K + 1, device="cuda")[1:], ln_bias=lb),    # misaligned
        dict(add=add, residual=residual, gate=gate),                        # add with the gated residual
        dict(add=add, residual=residual),
        dict(add=add, gate=gate),
        dict(add=add[:, :, :N // 2]),                                       # wrong shape
        dict(add=add.half()),                                               # wrong dtype
        dict(add=add.transpose(0, 1)),                                      # rows that form no 2-D view
        dict(residual=residual),                                            # residual without gate (adaLN rule)
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            m.mx_linear(x, w, None, sp, **kw)
    w1, w2 = torch.randn(128, K, device="cuda"), torch.randn(N, 128, device="cuda")
    for kw in bad[:3] + bad[9:]:
        with pytest.raises(ValueError):
            m.mx_mlp(x, w1, None, w2, None, sp, **kw)
    with pytest.raises(ValueError):
        m.layer_norm(x, lw, None)
    with pytest.raises(ValueError):
        m.layer_norm(torch.randn(4, 6, device="cuda"))                     # K not a multiple of 4
    with pytest.raises(ValueError):
        m.layer_norm(x.transpose(0, 1))
    torch.cuda.synchronize()                                                # no CUDA error was left behind
    assert torch.equal(m.mx_linear(x, w, None, sp, add=add), add + m.mx_linear(x, w, None, sp))
