"""Second, independent oracle for the quantizer (stage A2): the reference's OWN C++ device
functions (microxscaling/mx/cpp/{shared_exp,quantize}.cuh) compiled into oracle/_ref/libmxref.so
by oracle/ref_build/Makefile.  Checks the Python-path restatement (oracle/mxint8_oracle.py)
against it; skipped when the .so was not built.  The .so is not part of the repository: it can only be
built where the reference's sources are at hand (oracle/ref_build/Makefile, REF = their mx/cpp directory)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import mxint8_oracle as O

SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libmxref.so")
needs_so = pytest.mark.skipif(not os.path.exists(SO), reason="oracle/_ref/libmxref.so not built")


def ref_quantize(x: torch.Tensor, flush=False):
    lib = ctypes.CDLL(SO)
    x = x.contiguous().float()
    rows, hd = x.reshape(-1, x.shape[-1]).shape
    nb = (hd + 31) // 32
    out = np.empty((rows, hd), dtype=np.float32)
    exps = np.empty((rows, nb), dtype=np.int32)
    rc = lib.ref_quantize_mxint8(ctypes.c_void_p(x.data_ptr()), ctypes.c_long(rows), hd, 32, int(flush),
                                 out.ctypes.data_as(ctypes.c_void_p), exps.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0
    return torch.from_numpy(out).reshape(x.shape), torch.from_numpy(exps).reshape(*x.shape[:-1], nb)


@needs_so
@pytest.mark.parametrize("hd", [64, 72, 32, 128])
@pytest.mark.parametrize("kind", ["randn", "lognormal"])
def test_restatement_matches_reference_cpp(hd, kind):
    g = torch.Generator().manual_seed(hd)
    x = torch.randn(4, 197, hd, generator=g)
    if kind == "lognormal":
        x = x * torch.exp(2.0 * torch.randn(4, 197, 1, generator=g))
    x[0, 3] = 0.0                      # all-zero row
    x[1, 5, :32] = 0.0                 # all-zero block
    x[2, 7, :8] = -1e-7                # tiny negatives -> -0
    ref, ref_e = ref_quantize(x)
    c, e = O.quantize_mxint8(x)
    assert torch.equal(O.dequantize_mxint8(c, e), ref)          # value-equal (+-0 compare equal)
    nz = x.reshape(4, 197, -1, min(32, hd)).abs().amax(-1) > 0 if hd % 32 == 0 else None
    if nz is not None:                 # exponents agree on every non-zero block
        assert torch.equal(e.to(torch.int32)[nz], ref_e[nz])


@needs_so
def test_cpp_path_differs_only_at_log2_boundary():
    """The C++ path reads the exponent bits; the Python golden path uses fp32 floor(log2(.)) and
    rounds up just below a power of two (oracle LOG2_BUMP).  Document the one known divergence."""
    x = torch.zeros(1, 32)
    x[0, 0] = float(np.nextafter(np.float32(8.0), np.float32(0)))
    x[0, 1] = 1.0
    ref, ref_e = ref_quantize(x)
    c, e = O.quantize_mxint8(x)
    assert int(ref_e[0, 0]) == 2 and int(e[0, 0]) == 3
