"""Fused MX MLP (``mx_mlp``: fc1 with the GELU epilogue writing fc2's MXINT8 operand, then fc2) against the composition
``mx_linear(F.gelu(mx_linear(x, w1, b1)), w2, b2)`` with torch.equal, the activation against torch.nn.functional.gelu
over every fp32, bf16 and fp16 input, the launches of the fused call, ``QuantizedMlp``'s choice of path, and the
rejections of mx_mlp."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.helpers import mx_specs

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["fp32", "bf16", "fp16"]
APPROX = {"gelu": "none", "gelu_tanh": "tanh"}


def _m():
    import mx_quantization_b200 as m
    return m


def _inputs(M, K, N1, N2, dt, seed=0, bias=True):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g) * torch.exp(0.5 * torch.randn(M, 1, generator=g))
    w1 = torch.randn(N1, K, generator=g) * K ** -0.5
    w2 = torch.randn(N2, N1, generator=g) * N1 ** -0.5
    b1 = torch.randn(N1, generator=g) * 0.5 if bias else None
    b2 = torch.randn(N2, generator=g) * 0.1 if bias else None
    cuda = lambda t: None if t is None else t.cuda()    # noqa: E731
    return cuda(x).to(dt), cuda(w1), cuda(b1), cuda(w2), cuda(b2)


def _composition(x, w1, b1, w2, b2, sp, act, N1=None, N2=None):
    m = _m()
    h = m.mx_linear(x, w1, b1, sp, out_features=N1)
    return m.mx_linear(F.gelu(h, approximate=APPROX[act]), w2, b2, sp, out_features=N2)


# ---------------------------------------------------------------------------------------------- activation
@pytest.mark.gpu
@pytest.mark.parametrize("act", list(APPROX))
def test_activation_every_fp32_input(act):
    from mx_quantization_b200 import ops
    chunk = 1 << 28
    for start in range(-(1 << 31), 1 << 31, chunk):
        bits = torch.arange(start, start + chunk, dtype=torch.int64, device="cuda").to(torch.int32)
        x = bits.view(torch.float32)
        got, want = ops.activation(x, act), F.gelu(x, approximate=APPROX[act])
        same = got.view(torch.int32) == want.view(torch.int32)
        nan_in, nan_got, nan_want = torch.isnan(x), torch.isnan(got), torch.isnan(want)
        assert bool((same | nan_in | (nan_got & nan_want)).all()), f"bits differ in chunk starting at {start:#x}"
        assert bool(nan_got[nan_in].all())
        del bits, x, got, want, same, nan_in, nan_got, nan_want


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES[1:], ids=DT_IDS[1:])
@pytest.mark.parametrize("act", list(APPROX))
def test_activation_every_16bit_input(dt, act):
    from mx_quantization_b200 import ops
    x = torch.arange(-(1 << 15), 1 << 15, dtype=torch.int32, device="cuda").to(torch.int16).view(dt)
    got, want = ops.activation(x, act), F.gelu(x, approximate=APPROX[act])
    nan_in = torch.isnan(x)
    same = got.view(torch.int16) == want.view(torch.int16)
    assert bool((same | nan_in | (torch.isnan(got) & torch.isnan(want))).all())
    assert bool(torch.isnan(got)[nan_in].all())


# ---------------------------------------------------------------------------------------------- mx_mlp == composition
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("flush", [False, True], ids=["noflush", "flush"])
def test_mx_mlp_equals_composition(dt, bfloat, flush):
    """DeiT-base widths, M = 2 x 197 (a partial row tile): raw and prepared weights, every bias type, no bias, a
    row-strided view of x."""
    m = _m()
    sp = mx_specs(bfloat, flush)
    M, K, N1, N2 = 2 * 197, 768, 3072, 768
    x, w1, b1, w2, b2 = _inputs(M, K, N1, N2, dt, seed=bfloat + int(flush))
    if flush:
        x[5, :64] *= 1e-39                                         # blocks whose shared exponent is subnormal
    y = m.mx_mlp(x, w1, b1.to(dt), w2, b2.to(dt), sp)
    assert y.dtype == dt and y.shape == (M, N2)
    assert torch.equal(y, _composition(x, w1, b1.to(dt), w2, b2.to(dt), sp, "gelu"))
    w1_op, w2_op = m.mx_linear_prepare_weight(w1.to(dt), sp), m.mx_linear_prepare_weight(w2, sp)
    for bd1, bd2 in ((torch.float32, torch.bfloat16), (torch.float16, torch.float32)):
        got = m.mx_mlp(x, w1_op, b1.to(bd1), w2_op, b2.to(bd2), sp, hidden_features=N1, out_features=N2)
        assert torch.equal(got, _composition(x, w1_op, b1.to(bd1), w2_op, b2.to(bd2), sp, "gelu", N1, N2))
    assert torch.equal(m.mx_mlp(x, w1, None, w2, None, sp), _composition(x, w1, None, w2, None, sp, "gelu"))
    wide = torch.zeros(M, K + 64, dtype=dt, device="cuda")
    wide[:, :K] = x
    xs = wide[:, :K]
    assert torch.equal(m.mx_mlp(xs, w1, b1, w2, b2, sp, act="gelu_tanh"), _composition(xs, w1, b1, w2, b2, sp, "gelu_tanh"))


SHAPES = [  # M, K, N1, N2, act
    (2 * 256, 1152, 4608, 1152, "gelu_tanh"),    # DiT-XL/2 MLP (tanh GELU)
    (300, 128, 320, 64, "gelu"),                  # N1 = 320: a partial 256-column tile of fc1
    (1, 64, 64, 4, "gelu"),                       # one token
    (1, 64, 64, 4, "gelu_tanh"),
    (50432, 768, 3072, 768, "gelu"),              # DeiT-base, 256 images x 197 tokens
]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}to{s[2]}to{s[3]}_{s[4]}")
def test_mx_mlp_shapes(dt, shape):
    m = _m()
    M, K, N1, N2, act = shape
    for bfloat in (16, 32):
        sp = mx_specs(bfloat)
        x, w1, b1, w2, b2 = _inputs(M, K, N1, N2, dt, seed=M + bfloat)
        y = m.mx_mlp(x, w1, b1, w2, b2, sp, act=act)
        assert y.dtype == dt and y.shape == (M, N2)
        assert torch.equal(y, _composition(x, w1, b1, w2, b2, sp, act))
    x3 = x.reshape(1, M, K)
    assert m.mx_mlp(x3, w1, b1, w2, b2, sp, act=act).shape == (1, M, N2)


# ---------------------------------------------------------------------------------------------- launches
@pytest.mark.gpu
def test_mx_mlp_launches_only_library_kernels():
    from torch.profiler import ProfilerActivity, profile
    m = _m()
    sp = mx_specs(16)
    M, K, N1, N2 = 394, 768, 3072, 768
    x, w1, b1, w2, b2 = _inputs(M, K, N1, N2, torch.bfloat16)
    w1_op, w2_op = m.mx_linear_prepare_weight(w1, sp), m.mx_linear_prepare_weight(w2, sp)
    # x's quantizer, the rounding of b1 and of b2 (each only when present), fc1 with the GELU epilogue, fc2
    for bb1, bb2, n in ((b1, b2, 5), (None, b2, 4), (b1, None, 4), (None, None, 3)):
        m.mx_mlp(x, w1_op, bb1, w2_op, bb2, sp, hidden_features=N1, out_features=N2)
        assert m.last_launch_count() == n
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.mx_mlp(x, w1_op, b1, w2_op, b2, sp, hidden_features=N1, out_features=N2)
        torch.cuda.synchronize()
    kernels = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
    kernels = [k for k in kernels if not k.startswith("Memset") and not k.startswith("Memcpy")]
    assert len(kernels) == 5 and all("mxp::" in k for k in kernels), kernels
    assert sum("k_mx_linear_umma" in k for k in kernels) == 2


# ---------------------------------------------------------------------------------------------- QuantizedMlp
class _TimmMlp(nn.Module):
    def __init__(self, dim, act):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), act, nn.Linear(4 * dim, dim), nn.Dropout(0.0)


class _GeluSubclass(nn.GELU):
    pass


def _mlp_ref(mlp, x):
    """QuantizedMlp layer by layer: MxLinear fc1 -> the module's activation -> MxLinear fc2."""
    return mlp.fc2(mlp.act(mlp.fc1(x)))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("act", [nn.GELU(), nn.GELU("tanh"), nn.SiLU(), _GeluSubclass()],
                         ids=["gelu", "gelu_tanh", "silu", "gelu_subclass"])
def test_quantized_mlp_path(dt, act, monkeypatch):
    from mx_quantization_b200 import ops
    from mx_quantization_b200.modules import QuantizedMlp
    torch.manual_seed(5)
    mlp = QuantizedMlp(_TimmMlp(128, act), mx_specs=mx_specs(16)).cuda().to(dt)
    x = torch.randn(2, 197, 128, device="cuda").to(dt)
    calls = []
    real = ops.mx_mlp
    monkeypatch.setattr(ops, "mx_mlp", lambda *a, **k: calls.append(k.get("act")) or real(*a, **k))
    with torch.no_grad():
        z = mlp(x)
        want = _mlp_ref(mlp, x)
    fused = type(act) is nn.GELU
    assert calls == ([{"none": "gelu", "tanh": "gelu_tanh"}[act.approximate]] if fused else [])
    assert z.dtype == dt and z.shape == x.shape and torch.equal(z, want)
    with pytest.raises(RuntimeError, match="inference"):
        mlp(x)                                                    # grad mode with trainable weights: refused


# ---------------------------------------------------------------------------------------------- rejections
@pytest.mark.gpu
def test_mx_mlp_rejections_leave_no_cuda_error():
    m = _m()
    sp = mx_specs()
    x, w1, b1, w2, b2 = _inputs(64, 128, 256, 64, torch.float32)
    with pytest.raises(ValueError, match="act"):
        m.mx_mlp(x, w1, b1, w2, b2, sp, act="relu")
    with pytest.raises(ValueError, match="multiple of 64"):
        m.mx_mlp(x, w1[:96], b1[:96], w2[:, :96].contiguous(), b2, sp)          # N1 = 96
    with pytest.raises(ValueError, match="float64"):
        m.mx_mlp(x.double(), w1, b1, w2, b2, sp)
    with pytest.raises(ValueError, match="CUDA"):
        m.mx_mlp(x.cpu(), w1, b1, w2, b2, sp)
    with pytest.raises(ValueError):
        m.mx_mlp(x, w1, b1, w2[:, :128].contiguous(), b2, sp)                  # w2 does not take N1 inputs
    with pytest.raises(ValueError, match="hidden_features"):
        m.mx_mlp(x, m.mx_linear_prepare_weight(w1, sp), b1, w2, b2, sp)
    from mx_quantization_b200 import ops
    with pytest.raises(ValueError, match="act"):
        ops.activation(x, act="gelu_erf")
    torch.cuda.synchronize()
    y = m.mx_mlp(x, w1, b1, w2, b2, sp)                                         # a valid call still runs
    torch.cuda.synchronize()
    assert torch.equal(y, _composition(x, w1, b1, w2, b2, sp, "gelu"))
