"""The cost-follows-k epilogue on either side of its register bound: rows of up to 2 * K2S_KMAX = 32 kept keys keep
their list entries in registers after the compaction, longer rows run on the shared-memory list
(csrc/mxprune_attend_sparse.cuh).  At 197 tokens, top_k 32 and 33 through the fused launch (72 / 96 heads, fused path 2)
and through the three kernels with the stand-alone k_attend_sparse (18 / 24 heads: below the fused launch's 64-head
minimum, default path): the instantiation each launcher picks, masks bit-exact against the oracle, outputs within the oracle
budget, repeat calls identical, and 16-bit q / k / v equal to the call on the widened fp32 tensors."""
import re

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import mxint8_oracle as O
from tests.helpers import assert_out_close, fused_qkv_views, make_qkv, mx_specs, unpack_mask

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-3
KMAX = 16               # K2S_KMAX: rows of up to 2 * KMAX kept keys take the register path


@pytest.fixture(scope="module")
def mxq():
    import mx_quantization_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


def _kernels(fn, reps=3):
    """Names of the CUDA kernels fn launches, over reps calls (a profiling session late in a long run can miss its first
    kernel, which for a one-launch call is all of them)."""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


def _last_template_int(name):
    """Last template argument of a kernel name, demangled ('k<false, 0, 16>(...)') or mangled ('...ELi16EEEv...')."""
    m = re.search(r",\s*(\d+)>\s*\(", name) or re.search(r"Li(\d+)EEEv", name)
    assert m, name
    return int(m.group(1))


CASES = [  # B, H, hd, kind, bfloat, flush   (197 tokens)
    (8, 12, 64, "randn", 32, False),        # DeiT-base heads: the head_dim 64 instantiations
    (8, 12, 64, "lognormal", 16, True),     # wide score ranges: windows on the slow exponent path; bfloat 16, flush
    (8, 9, 32, "edges", 32, False),         # run-time head_dim instantiations, edge rows
]


@pytest.mark.parametrize("top_k", [2 * KMAX, 2 * KMAX + 1], ids=["registers", "list"])
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "three_kernels"])
@pytest.mark.parametrize("B,H,hd,kind,bfloat,flush", CASES)
def test_sparse_epilogue_register_bound(mxq, B, H, hd, kind, bfloat, flush, fused, top_k):
    N = 197
    assert top_k * 100 <= 35 * N                  # both sides of the bound take the cost-follows-k epilogue
    if not fused:
        B = 2                                     # B * H < 64: the default plan is the three kernels
    q, k, v = make_qkv(B, H, N, hd, seed=31, kind=kind)
    specs = mx_specs(bfloat, flush)
    qv, kv, vv = fused_qkv_views(q.cuda(), k.cuda(), v.cuda())
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    kmax = KMAX if top_k <= 2 * KMAX else 0
    try:
        mxq.set_fused_path(2 if fused else 1)
        res = {}
        names = _kernels(lambda: res.update(r=mxq.pruned_attention(qv, kv, vv, specs, top_k, return_mask=True)))
        out, mask = res["r"]
        assert mxq.last_launch_count() == (1 if fused else 3)
        # the launcher's choice of the register bound: the kernel's last template argument
        kname = "k_fused_pruned_attention" if fused else "k_attend_sparse"
        ours = [n for n in names if kname in n]
        assert ours and all(_last_template_int(n) == kmax for n in ours), names
        assert torch.equal(unpack_mask(mask, N), want), "masks differ from the oracle"
        assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL, 0.02 if (kind == "randn" and bfloat == 32) else None)
        assert torch.equal(mxq.pruned_attention(qv, kv, vv, specs, top_k), out), "not deterministic"
        for dt in (torch.bfloat16, torch.float16):
            hq, hk, hv = (x.to(dt) for x in (qv, kv, vv))
            out16 = mxq.pruned_attention(hq, hk, hv, specs, top_k)
            out32 = mxq.pruned_attention(hq.float(), hk.float(), hv.float(), specs, top_k)
            assert torch.equal(out16, out32.to(dt)), f"{dt}: differs from the widened fp32 call"
    finally:
        mxq.set_fused_path(True)
