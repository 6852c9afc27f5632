"""GPU parity: libmxprune (through the C ABI) against the CPU oracle and the reference's golden
vectors.  Integer stages bit-exact; fp32 attention output within 1e-3 of the reference's max-abs."""
import os

import numpy as np
import pytest
import torch

from oracle import mxint8_oracle as O
from tests.helpers import (assert_out_close, canonical_idx_from_mask, fused_qkv_views, load_golden, long_inputs,
                           make_qkv, mode_window_ok, mx_specs, unpack_mask)

pytestmark = pytest.mark.gpu

OUT_TOL = 1e-3     # max|out - ref| <= OUT_TOL * max|ref|   (north star: "max-abs 1e-3 relative")


@pytest.fixture(scope="module")
def mxq():
    import mx_quantization_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return m


SHAPES = [  # B, H, N, hd, kind, bfloat, flush
    (1, 2, 32, 64, "randn", 32, False),
    (2, 3, 197, 64, "randn", 32, False),       # C1 / C2 shape
    (1, 2, 256, 72, "lognormal", 32, False),   # C3 / C4 shape
    (1, 2, 256, 72, "randn", 16, False),       # DiT bfloat 16
    (1, 2, 120, 72, "edges", 32, True),        # PixArt flush + edge rows
    (1, 2, 37, 64, "edges", 32, False),
    (1, 1, 64, 32, "randn", 32, False),
    (1, 1, 100, 128, "lognormal", 32, False),
    (1, 2, 50, 96, "edges", 16, False),
    (1, 1, 8, 40, "randn", 32, False),
]


@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES)
def test_quantizer_bit_exact(mxq, B, H, N, hd, kind, bfloat, flush):
    q, k, v = make_qkv(B, H, N, hd, seed=1, kind=kind)
    specs = mx_specs(bfloat, flush)
    for x in (q, k):
        codes, exps, signs = mxq.quantize_mxint8(x.cuda(), specs, with_signs=True)
        oc, oe = O.quantize_mxint8(x, 32, bfloat, flush)
        assert torch.equal(codes.cpu(), oc)
        assert torch.equal(exps.cpu(), oe)
        assert torch.equal(signs.cpu().to(torch.int64) & 0xFFFFFFFF, O.sign_words(oc))
        approx = mxq.exp_sign_approx(x.cuda(), specs)
        assert torch.equal(approx.cpu(), O.exponent_based_sign(oc, oe))


def test_quantizer_log2_boundary(mxq):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "quantizer_log2_boundary.npz"))
    x = torch.from_numpy(z["x"])                    # (rows, 32)
    ref = torch.from_numpy(z["MX"])                 # reference fake-quant output
    codes, exps = mxq.quantize_mxint8(x.reshape(1, 1, -1, 32).cuda(), mx_specs())
    deq = O.dequantize_mxint8(codes.cpu().reshape(-1, 32), exps.cpu().reshape(-1, 1))
    assert torch.equal(deq, ref)


@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES)
def test_pred_scores_bit_exact(mxq, B, H, N, hd, kind, bfloat, flush):
    q, k, _ = make_qkv(B, H, N, hd, seed=2, kind=kind)
    s = mxq.predict_scores(q.cuda(), k.cuda(), mx_specs(bfloat, flush)).cpu()
    qc, qe = O.quantize_mxint8(q, 32, bfloat, flush)
    kc, ke = O.quantize_mxint8(k, 32, bfloat, flush)
    assert torch.equal(s, O.pred_scores_integer(qc, qe, kc, ke))


@pytest.mark.parametrize("pred_path", ["tcgen05", "cuda_core"])
@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES)
@pytest.mark.parametrize("kfrac", [0.0, 0.15, 0.6, 1.0])
def test_topk_mask_bit_exact(mxq, B, H, N, hd, kind, bfloat, flush, kfrac, pred_path):
    """Both predictor kernels (tensor-core scoring / CUDA-core XOR+POPC) against the oracle."""
    top_k = max(1, min(N, int(round(kfrac * N))))
    q, k, _ = make_qkv(B, H, N, hd, seed=3, kind=kind)
    specs = mx_specs(bfloat, flush)
    mxq.set_predict_path(pred_path)
    try:
        r = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True, return_codes=True)
        r_nocodes = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k)
    finally:
        mxq.set_predict_path("tcgen05")
    assert torch.equal(r_nocodes["mask"], r["mask"])
    qc, qe = O.quantize_mxint8(q, 32, bfloat, flush)
    kc, ke = O.quantize_mxint8(k, 32, bfloat, flush)
    idx = O.canonical_topk(O.pred_scores_integer(qc, qe, kc, ke), top_k)
    want = O.mask_words_to_dense(O.idx_to_mask_words(idx, N), N)
    got = unpack_mask(r["mask"], N)
    assert torch.equal(got, want)
    assert torch.equal(r["idx"].cpu().to(torch.int64), torch.sort(idx, dim=-1).values)
    assert torch.equal(r["q_codes"].cpu(), qc) and torch.equal(r["q_exps"].cpu(), qe)
    assert torch.equal(r["k_codes"].cpu(), kc) and torch.equal(r["k_exps"].cpu(), ke)


@pytest.mark.parametrize("path", ["tcgen05", "cuda_core"])
@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES)
def test_sparse_attention_same_index_set(mxq, B, H, N, hd, kind, bfloat, flush, path):
    mxq.set_attention_path(path)
    top_k = max(1, int(0.3 * N))
    q, k, v = make_qkv(B, H, N, hd, seed=4, kind=kind)
    specs = mx_specs(bfloat, flush)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    mask = O.idx_to_mask_words(ref["idx"], N)
    mask_i32 = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask).to(torch.int32)
    out = mxq.sparse_attention(ref["q_codes"].cuda(), ref["q_exps"].cuda(), ref["k_codes"].cuda(),
                               ref["k_exps"].cuda(), v.cuda(), mask_i32.cuda(), specs,
                               scale=O.default_scale(hd)).cpu()
    mxq.set_attention_path("tcgen05")
    assert_out_close(out, ref, v, N, bfloat, OUT_TOL, 0.02 if (kind == "randn" and bfloat == 32) else None)


@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES)
def test_pruned_attention_end_to_end(mxq, B, H, N, hd, kind, bfloat, flush):
    top_k = max(1, int(0.4 * N))
    q, k, v = make_qkv(B, H, N, hd, seed=5, kind=kind)
    specs = mx_specs(bfloat, flush)
    qv, kv, vv = fused_qkv_views(q.cuda(), k.cuda(), v.cuda())    # strided views, as in the modules
    assert not qv.is_contiguous()
    out, mask = mxq.pruned_attention(qv, kv, vv, specs, top_k, return_mask=True)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    assert torch.equal(unpack_mask(mask, N), want)
    assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL, 0.02 if (kind == "randn" and bfloat == 32) else None)
    # writing into a (B,N,H,hd) buffer through a permuted view == the module's transpose(1,2)
    buf = torch.empty(B, N, H, hd, device="cuda")
    mxq.pruned_attention(qv, kv, vv, specs, top_k, out=buf.permute(0, 2, 1, 3))
    assert torch.equal(buf.permute(0, 2, 1, 3), out)


@pytest.mark.parametrize("ratio", [0.04, 0.15, 0.34])
@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,flush", SHAPES + [(2, 12, 197, 64, "randn", 32, False),
                                                                 (2, 4, 256, 72, "lognormal", 16, True)])
def test_pruned_attention_cost_follows_k(mxq, B, H, N, hd, kind, bfloat, flush, ratio):
    """Small top_k / Nk: the exact stage runs on the compacted row lists (k_attend_sparse, cost ~ k) - same masks,
    outputs within the same budget as the dense-epilogue kernel it replaces (workloads/deit/scripts/main.py:124,147-152:
    only the k gathered entries are ever used)."""
    top_k = max(1, int(ratio * N))
    q, k, v = make_qkv(B, H, N, hd, seed=11, kind=kind)
    specs = mx_specs(bfloat, flush)
    qv, kv, vv = fused_qkv_views(q.cuda(), k.cuda(), v.cuda())
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    outs = {}
    try:
        for on in (True, False):
            mxq.set_fused_path(on)
            out, mask = mxq.pruned_attention(qv, kv, vv, specs, top_k, return_mask=True)
            assert torch.equal(unpack_mask(mask, N), want)
            # (top_k < 4: p sits at / next to a power of two in most rows - one-hot rows - so the allowance is the norm)
            assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL,
                             0.02 if (kind == "randn" and bfloat == 32 and top_k >= 4) else None)
            outs[on] = out.cpu()
    finally:
        mxq.set_fused_path(True)
    # the two epilogues differ only in the order of the row sum (a few ulps of p)
    scale = float(ref["out"].abs().max())
    assert float((outs[True] - outs[False]).abs().max()) <= 2 * OUT_TOL * scale


@pytest.mark.parametrize("name", ["predictor_methods_deit", "predictor_methods_dit_bf16", "predictor_methods_pixart"])
def test_predictor_class_methods(mxq, name):
    """``exponent_approximation`` - the one name the reference exports (funcs/__init__.py:11) - built from STRIDED views
    of a fused qkv buffer as the modules pass them (workloads/deit/scripts/main.py:87-88,107): every method's dense
    return against the unmodified reference's (tests/golden/make_golden_methods.py), bit for bit, plus the compact
    accessors against the oracle."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    B, H, N, hd, _, bfloat, flush = (int(x) for x in z["meta"])
    q, k = torch.from_numpy(z["q"]), torch.from_numpy(z["k"])
    qv, kv, _ = fused_qkv_views(q.cuda(), k.cuda(), k.cuda())
    assert not qv.is_contiguous()
    specs = mx_specs(bfloat, bool(flush))
    obj = mxq.exponent_approximation(Q=qv, K=kv, mx_specs=specs)
    for method in ("exponent_based_sign", "partial_Q", "partial_K", "MXINT4", "two_step_leading_ones",
                   "exponent_based_sign_leading_ones"):
        aq, ak = getattr(obj, method)()
        assert aq.shape == q.shape and ak.shape == k.shape and aq.dtype == torch.float32
        assert torch.equal(aq.cpu(), torch.from_numpy(z[method + ".Q"])), f"{method}: Q operand differs from the reference"
        assert torch.equal(ak.cpu(), torch.from_numpy(z[method + ".K"])), f"{method}: K operand differs from the reference"
    oqc, oqe = O.quantize_mxint8(q, 32, bfloat, bool(flush))
    okc, oke = O.quantize_mxint8(k, 32, bfloat, bool(flush))
    (qc, kc), (qe, ke), (qs, ks) = obj.codes, obj.exps, obj.signbits
    assert torch.equal(qc.cpu(), oqc) and torch.equal(kc.cpu(), okc)
    assert torch.equal(qe.cpu(), oqe) and torch.equal(ke.cpu(), oke)
    assert torch.equal(qs.cpu().to(torch.int64) & 0xFFFFFFFF, O.sign_words(oqc))
    assert torch.equal(ks.cpu().to(torch.int64) & 0xFFFFFFFF, O.sign_words(okc))
    # the fused replacement of `method() -> @ -> topk` selects what the dense route selects (canonical tie rule)
    top_k = max(1, N // 4)
    aq, ak = obj.exponent_based_sign()
    want = O.canonical_topk((aq @ ak.transpose(-2, -1)).cpu(), top_k)
    sel = obj.predict_topk(top_k, return_idx=True)
    pinned = O.pred_window_ok(O.predictor_exponents(oqc, oqe), O.predictor_exponents(okc, oke), O.block_widths(hd)).all(-1)
    assert torch.equal(sel["idx"].cpu().to(torch.int64)[pinned], torch.sort(want, dim=-1).values[pinned])


def test_analysis_outputs_reference_fixture(mxq):
    """--anal figures from the GPU masks: diff_idx_analysis (funcs/analysis.py:136-157) against the value the reference
    function returned for the same index sets, with the predicted set coming from the selection kernel."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "analysis_overlap.npz"))
    B, H, N, hd, k_true, k_pred = (int(x) for x in z["meta"])
    q, k = torch.from_numpy(z["q"]).cuda(), torch.from_numpy(z["k"]).cuda()
    specs = mx_specs()
    pred = mxq.predict_topk(q, k, specs, k_pred, return_idx=True)
    true = mxq.predict_topk(q, k, specs, k_true, return_idx=True, pred_mode="exact")
    assert torch.equal(torch.sort(torch.from_numpy(z["pred_idx"]), dim=-1).values, pred["idx"].cpu().to(torch.int64))
    assert torch.equal(torch.sort(torch.from_numpy(z["true_idx"]), dim=-1).values, true["idx"].cpu().to(torch.int64))
    got = mxq.diff_idx_analysis(true["idx"].to(torch.int64), pred["idx"].to(torch.int64))
    assert abs(got - float(z["diff_idx_analysis"][0])) < 1e-12
    # the per-row intersection ratio from the bitmask agrees with a set intersection on the index lists
    ov = mxq.topk_overlap(pred["mask"], true["idx"].to(torch.int64)).cpu()
    ti, pi = true["idx"].cpu(), pred["idx"].cpu()
    brute = torch.tensor([[[len(set(ti[b, h, r].tolist()) & set(pi[b, h, r].tolist())) / k_true for r in range(N)]
                           for h in range(H)] for b in range(B)], dtype=torch.float64)
    assert torch.equal(ov, brute)


FUSED_SHAPES = [  # B, H, N, hd, top_k, kind, bfloat, flush   (B * H >= 64: the domain of the fused kernel)
    (8, 12, 197, 64, 30, "randn", 32, False),       # C2 slice: tight 104-column split, cost-follows-k epilogue
    (6, 12, 197, 64, 80, "lognormal", 32, False),   # dense epilogue (k / N = 0.41)
    (4, 16, 256, 72, 154, "randn", 16, False),      # C3 slice: bfloat 16, dense epilogue
    (4, 16, 256, 72, 77, "lognormal", 32, True),    # C4 slice: flush
    (4, 16, 256, 72, 26, "edges", 32, True),        # C5 ratio 0.1: sparse epilogue at head_dim 72, edge rows
    (8, 8, 160, 64, 40, "edges", 32, False),        # NC = 7 without the tight split, generic rows
    (8, 8, 220, 64, 50, "randn", 16, False),        # 112-column split
    (8, 9, 130, 32, 13, "randn", 32, False),        # head_dim 32
    (33, 2, 250, 72, 60, "lognormal", 16, False),   # odd head count: the last group of the last CTA idles
    (20, 16, 197, 64, 30, "randn", 32, False),      # 320 heads on 296 groups: the shared last round (one query tile per group)
]


@pytest.mark.parametrize("B,H,N,hd,top_k,kind,bfloat,flush", FUSED_SHAPES)
def test_fused_kernel(mxq, B, H, N, hd, top_k, kind, bfloat, flush):
    """The whole path as ONE persistent launch (k_fused_pruned_attention): bit-exact masks, outputs within the
    budget, against the oracle and against the three-kernel path it replaces (workloads/deit/scripts/main.py:101-152)."""
    q, k, v = make_qkv(B, H, N, hd, seed=21, kind=kind)
    specs = mx_specs(bfloat, flush)
    qv, kv, vv = fused_qkv_views(q.cuda(), k.cuda(), v.cuda())
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    outs, launches = {}, {}
    try:
        for on in (True, False):
            mxq.set_fused_path(2 if on else 0)          # 2: also where the default policy prefers the three kernels
            out, mask = mxq.pruned_attention(qv, kv, vv, specs, top_k, return_mask=True)
            launches[on] = mxq.last_launch_count()
            assert torch.equal(unpack_mask(mask, N), want), f"fused={on}: masks differ from the oracle"
            assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL, 0.02 if (kind == "randn" and bfloat == 32) else None)
            outs[on] = out.cpu()
            # without a mask output (the default call): the masks stay in the kernel's workspace slots
            out2 = mxq.pruned_attention(qv, kv, vv, specs, top_k)
            assert torch.equal(out2.cpu(), outs[on])
    finally:
        mxq.set_fused_path(True)
    assert launches[True] == 1 and launches[False] == 3, launches
    scale = float(ref["out"].abs().max())
    assert float((outs[True] - outs[False]).abs().max()) <= 2 * OUT_TOL * scale


@pytest.mark.parametrize("B,H,N,hd,top_k,launches", [
    (6, 12, 197, 64, 30, 1),       # DeiT-shaped: one fused persistent launch
    (2, 3, 197, 64, 30, 3),        # too few heads for a persistent launch (C1)
    (8, 16, 256, 72, 26, 3),       # head_dim 72: 64-row staging steps - the three kernels (K2 = the cost-follows-k kernel)
    (8, 16, 256, 72, 154, 3),      # DiT's k: dense epilogue
    (2, 4, 512, 72, 128, -6),      # streamed key blocks: operand pre-passes + selection + V prep + two-lanes-per-row attention (at most 6)
])
def test_default_launch_plan(mxq, B, H, N, hd, top_k, launches):
    """The launch plan mxp_pruned_attention picks by default (DESIGN.md 5): results are checked elsewhere; here only that the
    shapes of the workloads take the plan that was measured faster, and that the call stays a fixed, small number of launches."""
    q, k, v = make_qkv(B, H, N, hd, seed=2)
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), mx_specs(), top_k, return_mask=True)
    n = mxq.last_launch_count()
    assert (n == launches) if launches > 0 else (3 < n <= -launches), n
    words = mask.to(torch.int64) & 0xFFFFFFFF
    pop = sum(((words >> b) & 1) for b in range(32)).sum(-1)
    assert bool((pop == top_k).all()) and bool(torch.isfinite(out).all())


def test_fused_kernel_full_c2_properties(mxq):
    """DeiT-base layer at its full size (B=256, H=12, N=197, hd=64, k=30): the fused launch against the three-kernel
    path on all 3072 heads - identical masks, every row keeps exactly k keys, outputs agree."""
    B, H, N, hd, top_k = 256, 12, 197, 64, 30
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn(B, N, 3, H, hd, device="cuda", generator=g).permute(2, 0, 3, 1, 4)
    specs = mx_specs()
    res = {}
    try:
        for on in (True, False):
            mxq.set_fused_path(on)
            res[on] = mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k, return_mask=True)
    finally:
        mxq.set_fused_path(True)
    torch.cuda.synchronize()
    assert torch.equal(res[True][1], res[False][1])
    words = res[True][1].to(torch.int64) & 0xFFFFFFFF
    pop = sum(((words >> b) & 1) for b in range(32)).sum(-1)
    assert bool((pop == top_k).all())
    # the two exact stages sum the row's exponentials in different orders: a p within an ulp of a rounding tie of the
    # P quantizer lands on the other code in a handful of the 605 184 rows (one code step of one key, see
    # helpers.out_error_budget); everything else agrees to the tolerance
    scale = float(res[False][0].abs().max())
    diff = (res[True][0] - res[False][0]).abs().amax(-1)
    assert float((diff > 2 * OUT_TOL * scale).float().mean()) < 2e-4
    assert float(diff.max()) <= 2.0 ** -6 * float(qkv[2].abs().max()) * 1.01
    # determinism of the persistent schedule
    again = mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k)
    assert torch.equal(again, res[True][0])


def test_two_devices_one_process(mxq):
    """SURVEY 8(b): the library must be callable on several devices of one process (per-device shared-memory
    opt-in, no process-global device state)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    specs = mx_specs()
    outs = []
    q, k, v = make_qkv(8, 12, 197, 64, seed=5)
    for dev in ("cuda:0", "cuda:1", "cuda:0"):
        for on in (True, False):
            mxq.set_fused_path(on)
            out, mask = mxq.pruned_attention(q.to(dev), k.to(dev), v.to(dev), specs, 30, return_mask=True)
            outs.append((out.cpu(), mask.cpu()))
    mxq.set_fused_path(True)
    for o, m in outs[2:]:
        assert torch.equal(m, outs[0][1])
    assert torch.equal(outs[2][0], outs[0][0]) and torch.equal(outs[4][0], outs[0][0])
    assert torch.equal(outs[3][0], outs[1][0]) and torch.equal(outs[5][0], outs[1][0])


@pytest.mark.parametrize("name", ["deit_small", "dit_small", "dit_bf16", "pixart_flush", "deit_edges",
                                  "deit_tiny_c1"])
def test_against_reference_golden(mxq, name):
    """Outputs of the unmodified reference (tests/golden/make_golden.py)."""
    d, m = load_golden(name)
    specs = mx_specs(m["bfloat"], m["flush"])
    q, k, v = d["q"].cuda(), d["k"].cuda(), d["v"].cuda()
    codes, exps = mxq.quantize_mxint8(q, specs)
    assert torch.equal(O.dequantize_mxint8(codes.cpu(), exps.cpu()), d["MX_Q"])
    if "approx_Q" in d:
        assert torch.equal(mxq.exp_sign_approx(q, specs).cpu(), d["approx_Q"])
        assert torch.equal(mxq.exp_sign_approx(k, specs).cpu(), d["approx_K"])
    out, mask = mxq.pruned_attention(q, k, v, specs, m["top_k"], return_mask=True)
    got = unpack_mask(mask, m["N"])
    want = torch.zeros_like(got)
    want.scatter_(-1, d["idx"], True)
    if name in ("pixart_flush", "deit_edges"):
        # all-zero blocks: where the block terms of a (query, key) pair spread past one 24-bit window the reference's
        # fp32 matmul is summation-order dependent (parity unpinned, DESIGN.md).  Rows whose EVERY pair is inside the
        # window are pinned and must be bit-equal; only the others are exempt
        qc, qe = O.quantize_mxint8(d["q"], 32, m["bfloat"], m["flush"])
        kc, ke = O.quantize_mxint8(d["k"], 32, m["bfloat"], m["flush"])
        pinned = O.pred_window_ok(O.predictor_exponents(qc, qe), O.predictor_exponents(kc, ke),
                                  O.block_widths(m["hd"])).all(-1)
        assert torch.equal(got[pinned], want[pinned])
        print(f"{name}: {int((~pinned).sum())} of {pinned.numel()} rows exempt (a pair outside the 24-bit window)")
        # (one all-zero key block un-pins every query row of its head: about half the rows of these two fixtures)
        assert float(pinned.float().mean()) > 0.3
        assert float((got == want).all(-1).float().mean()) > 0.9
        assert bool((got.sum(-1) == m["top_k"]).all())
    else:
        assert torch.equal(got, want)
        ref = {"true_vals": d["true_vals"], "idx": d["idx"], "out": d["out"]}
        assert_out_close(out.cpu(), ref, d["v"], m["N"], m["bfloat"], OUT_TOL)


def test_full_size_properties(mxq):
    """C3/C4 full shape (B=256,H=16,N=256,hd=72,k=154): size-independent properties + exact
    comparison with the oracle on a sample of heads (heads are independent)."""
    B, H, N, hd, top_k = 256, 16, 256, 72, 154
    g = torch.Generator(device="cuda").manual_seed(7)
    qkv = torch.randn(B, N, 3, H, hd, device="cuda", generator=g).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    specs = mx_specs()
    out, mask = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
    torch.cuda.synchronize()
    # every row keeps exactly top_k keys
    m64 = mask.to(torch.int64) & 0xFFFFFFFF
    pop = torch.zeros_like(m64)
    for s in range(32):
        pop += (m64 >> s) & 1
    assert bool((pop.sum(-1) == top_k).all())
    # deterministic
    out2, mask2 = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
    assert torch.equal(out, out2) and torch.equal(mask, mask2)
    # the CUDA-core predictor kernel selects the same sets on all 4096 heads
    mxq.set_predict_path("cuda_core")
    try:
        _, mask3 = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
    finally:
        mxq.set_predict_path("tcgen05")
    assert torch.equal(mask, mask3)
    # head independence: a (batch, head) slice computed alone gives the same bits
    sl = (slice(17, 19), slice(5, 8))
    out_s, mask_s = mxq.pruned_attention(q[sl], k[sl], v[sl], specs, top_k, return_mask=True)
    assert torch.equal(out_s, out[sl]) and torch.equal(mask_s, mask[sl])
    # softmax.V is a convex combination of (quantised) V rows
    vmax = v.abs().amax(dim=2, keepdim=True)
    assert bool((out.abs() <= vmax * 1.02 + 1e-6).all())
    # exact check on sampled heads
    for (b, h) in [(0, 0), (100, 7), (255, 15)]:
        qs, ks, vs = (t[b:b + 1, h:h + 1].cpu() for t in (q, k, v))
        ref = O.pruned_attention(qs, ks, vs, top_k, integer_scores=True)
        want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
        assert torch.equal(unpack_mask(mask[b:b + 1, h:h + 1], N), want)
        assert_out_close(out[b:b + 1, h:h + 1].cpu(), ref, vs, N, 32, OUT_TOL)


def test_error_behaviour(mxq):
    q, k, v = make_qkv(1, 1, 32, 64)
    specs = mx_specs()
    with pytest.raises(ValueError):
        mxq.pruned_attention(q, k, v, specs, 8)                        # CPU tensors: no fallback
    with pytest.raises(ValueError):
        mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, 33)  # top_k > Nk
    bad = dict(specs); bad["a_elem_format"] = "fp8_e4m3"
    with pytest.raises(ValueError):
        mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), bad, 8)
    with pytest.raises(ValueError):
        mxq.pruned_attention(q.cuda().double(), k.cuda(), v.cuda(), specs, 8)


LONG_SHAPES = [  # B, H, N, hd, bfloat  -- key counts beyond one key block (Nk > 256): online softmax path
    (1, 2, 512, 72, 32),
    (1, 1, 1000, 64, 32),
    (1, 2, 300, 72, 16),
    (1, 1, 2048, 72, 32),
    (1, 1, 600, 128, 32),      # head_dim 128: the largest shared-memory layout of the long-sequence kernel
    (1, 2, 400, 40, 16),       # head_dim 40: operands padded to 48
]


@pytest.mark.parametrize("B,H,N,hd,bfloat", LONG_SHAPES)
def test_exact_attention_long_sequences(mxq, B, H, N, hd, bfloat):
    """Exact stage on key counts above 256 (C5 sweep territory), kept set taken from the oracle."""
    top_k = max(1, int(0.25 * N))
    q, k, v = make_qkv(B, H, N, hd, seed=6, kind="randn")
    specs = mx_specs(bfloat, False)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, integer_scores=True)
    mask = O.idx_to_mask_words(ref["idx"], N)
    mask_i32 = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask).to(torch.int32)
    out = mxq.sparse_attention(ref["q_codes"].cuda(), ref["q_exps"].cuda(), ref["k_codes"].cuda(),
                               ref["k_exps"].cuda(), v.cuda(), mask_i32.cuda(), specs,
                               scale=O.default_scale(hd)).cpu()
    assert_out_close(out, ref, v, N, bfloat, OUT_TOL)


@pytest.mark.parametrize("kfrac", [0.1, 0.5])
@pytest.mark.parametrize("bfloat", [16, 32])
@pytest.mark.parametrize("hd", [64, 72, 128])
@pytest.mark.parametrize("N", [300, 1000])
def test_long_attention_same_in_every_fused_mode(mxq, N, hd, bfloat, kfrac):
    """Nk > 256: fused path 0 changes only how the selection finds a row's threshold (same masks), not the attention
    kernel - masks and outputs are bit-identical to the default's."""
    top_k = max(1, int(kfrac * N))
    q, k, v = (t.cuda() for t in make_qkv(1, 2, N, hd, seed=9))
    specs = mx_specs(bfloat, False)
    res = {}
    try:
        for mode in (0, 1):
            mxq.set_fused_path(mode)
            res[mode] = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
    finally:
        mxq.set_fused_path(True)
    assert torch.equal(res[0][1], res[1][1])
    assert torch.equal(res[0][0], res[1][0])


@pytest.mark.parametrize("B,H,N,hd,kind,bfloat,kfrac", [
    (1, 2, 512, 72, "randn", 32, 0.1),
    (1, 1, 1000, 64, "lognormal", 32, 0.25),
    (1, 2, 300, 64, "edges", 32, 0.5),
    (1, 1, 1024, 72, "randn", 16, 0.5),
    (1, 1, 2048, 72, "randn", 32, 0.1),
    (2, 2, 700, 96, "randn", 32, 0.3),
    (1, 3, 333, 64, "randn", 16, 0.2),
    (1, 1, 4096, 72, "randn", 32, 0.1),            # C5's largest point (BASELINE.json configs[4]), both ends of the ratio range
    (1, 1, 4096, 72, "randn", 32, 0.5),
    (1, 2, 1536, 72, "lognormal05", 32, 0.25),     # keys wider than 15 bits stay on the tensor-core selection; bins of 2^fs keys
    (1, 1, 2304, 64, "lognormal05", 16, 0.1),
])
@pytest.mark.parametrize("pred_path", ["tcgen05", "cuda_core"])
def test_long_sequence_end_to_end(mxq, B, H, N, hd, kind, bfloat, kfrac, pred_path):
    """Config C5 territory (Nk > 256): long-sequence predictor (tensor-core radix select with the
    CUDA-core kernel for rows outside the integer window / CUDA-core kernel alone) + key-blocked
    exact attention."""
    top_k = max(1, int(kfrac * N))
    q, k, v = make_qkv(B, H, N, hd, seed=8, kind=kind)
    specs = mx_specs(bfloat, False)
    mxq.set_predict_path(pred_path)
    try:
        _long_e2e(mxq, q, k, v, specs, top_k, N, bfloat)
    finally:
        mxq.set_predict_path("tcgen05")


@pytest.mark.parametrize("kind", ["randn", "lognormal0.25", "lognormal0.5", "lognormal1.5", "ties", "constant", "zeros",
                                  "skewed", "outliers"])
@pytest.mark.parametrize("N,hd,kfrac", [(640, 72, 0.25), (1100, 64, 0.1), (2048, 72, 0.5)])
def test_long_selection_paths_agree(mxq, kind, N, hd, kfrac):
    """The long-sequence selection (k_select_long_tc) resolves a row's threshold three ways - sampled fine window (bins of one
    or of 2^fs key values), the radix levels alone (fused path 0), and, outside the tensor-core window, the CUDA-core integer
    kernel: masks AND index lists must be identical, whatever the input does to the sample (funcs: main.py:118-123 top-k of
    the predicted scores; the canonical tie rule of SURVEY 8a)."""
    q, k = long_inputs(kind, 2, N, hd, seed=N + hd)
    specs = mx_specs(32, False)
    top_k = max(1, int(kfrac * N))
    res = {}
    try:
        for name, fused, pred in (("fine", 1, "tcgen05"), ("radix", 0, "tcgen05"), ("core", 1, "cuda_core")):
            mxq.set_fused_path(fused)
            mxq.set_predict_path(pred)
            res[name] = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True)
    finally:
        mxq.set_fused_path(True)
        mxq.set_predict_path("tcgen05")
    for name in ("radix", "core"):
        assert torch.equal(res["fine"]["mask"], res[name]["mask"]), f"fine window vs {name}: masks differ"
        assert torch.equal(res["fine"]["idx"], res[name]["idx"]), f"fine window vs {name}: index lists differ"


def _long_e2e(mxq, q, k, v, specs, top_k, N, bfloat):
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
    assert torch.equal(unpack_mask(mask, N), want)
    assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL)
    r = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True, return_codes=True)
    assert torch.equal(r["idx"].cpu().to(torch.int64), torch.sort(ref["idx"], dim=-1).values)
    assert torch.equal(r["k_codes"].cpu(), ref["k_codes"]) and torch.equal(r["q_exps"].cpu(), ref["q_exps"])


# ---- SURVEY 8 f1: cross-attention (Nq != Nk) with PixArt's additive text mask ----------------------

def _load_cross(name):
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    d = {k: torch.from_numpy(z[k]) for k in z.files}
    B, H, Nq, S, hd, top_k, bfloat, flush = (int(x) for x in z["meta"])
    return d, dict(B=B, H=H, Nq=Nq, S=S, hd=hd, top_k=top_k, bfloat=bfloat, flush=bool(flush))


@pytest.mark.parametrize("pred_path", ["tcgen05", "cuda_core"])
@pytest.mark.parametrize("name", ["pixart_cross", "pixart_cross_k77", "pixart_cross_all"])
def test_cross_attention_reference_golden(mxq, name, pred_path):
    """Outputs of the unmodified reference functions in the order of PixArt's MXCrossAttention.forward
    (workloads/PixArt/models/MX_transformer_block.py:791-859; tests/golden/make_golden_cross.py)."""
    d, m = _load_cross(name)
    specs = mx_specs(m["bfloat"], m["flush"])
    bias = d["key_bias"].reshape(m["B"], 1, 1, m["S"]).cuda()
    mxq.set_predict_path(pred_path)
    try:
        out, mask = mxq.pruned_attention(d["q"].cuda(), d["k"].cuda(), d["v"].cuda(), specs, m["top_k"],
                                         scale=1.0 / (m["hd"] ** 0.5), return_mask=True, key_bias=bias)
    finally:
        mxq.set_predict_path("tcgen05")
    got = unpack_mask(mask, m["S"])
    want = torch.zeros_like(got)
    want.scatter_(-1, d["idx"], True)
    assert torch.equal(got, want)
    ref = {"true_vals": d["true_vals"], "idx": d["idx"], "out": d["out"]}
    assert_out_close(out.cpu(), ref, d["v"], m["S"], m["bfloat"], OUT_TOL)


@pytest.mark.parametrize("B,H,Nq,Nk,hd,top_k,bfloat", [
    (2, 3, 256, 120, 72, 77, 32),      # PixArt cross-attention shape, no mask
    (1, 2, 100, 197, 64, 30, 16),
    (1, 1, 300, 64, 64, 16, 32),
    (1, 2, 64, 1000, 72, 100, 32),     # long key side
])
def test_rectangular_attention(mxq, B, H, Nq, Nk, hd, top_k, bfloat):
    """Nq != Nk through the whole path, against the oracle."""
    g = torch.Generator().manual_seed(31)
    q = torch.randn(B, H, Nq, hd, generator=g)
    k = torch.randn(B, H, Nk, hd, generator=g)
    v = torch.randn(B, H, Nk, hd, generator=g)
    specs = mx_specs(bfloat, False)
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], Nk), Nk)
    assert torch.equal(unpack_mask(mask, Nk), want)
    assert_out_close(out.cpu(), ref, v, Nk, bfloat, OUT_TOL)


def test_cross_attention_module_shim(mxq):
    """MXCrossAttention shim == pruned_attention on its own projections."""
    from mx_quantization_b200.modules import MXCrossAttention
    torch.manual_seed(0)
    dim, heads, B, N, S = 128, 2, 2, 64, 40
    m = MXCrossAttention(dim, heads).cuda().set_config(mx_quant=True, mx_specs=mx_specs(32, True), top_k=True, k=20,
                                                       ex_pred=True, pred_mode="ex_pred")
    x = torch.randn(B, N, dim, device="cuda")
    enc = torch.randn(B, S, dim, device="cuda")
    keep = torch.zeros(B, S, device="cuda"); keep[0, :13] = 1; keep[1, :27] = 1
    amask = ((1 - keep) * -10000.0).reshape(B, 1, S)
    with torch.no_grad():
        y = m(x, encoder_hidden_states=enc, attention_mask=amask)
    with torch.no_grad():
        q = m.to_q(x).view(B, N, heads, dim // heads).transpose(1, 2)
        k = m.to_k(enc).view(B, S, heads, dim // heads).transpose(1, 2)
        v = m.to_v(enc).view(B, S, heads, dim // heads).transpose(1, 2)
    from mx_quantization_b200.modules import MxLinear
    assert isinstance(m.to_q, MxLinear) and isinstance(m.to_out[0], MxLinear)      # set_config swapped the projections
    ref = O.pruned_attention(q.cpu(), k.cpu(), v.cpu(), 20, scale=1.0 / ((dim // heads) ** 0.5), flush=True,
                             integer_scores=True, key_bias=amask.reshape(B, 1, 1, S).cpu())
    with torch.no_grad():
        want = m.to_out(ref["out"].transpose(1, 2).reshape(B, N, dim).cuda())
    assert float((y - want).abs().max()) <= 2e-3 * float(want.abs().max())


@pytest.mark.parametrize("B,H,N,hd,bfloat", [(2, 3, 197, 64, 32), (1, 2, 256, 72, 16), (1, 1, 50, 96, 32)])
def test_dense_attention_top_k_false(mxq, B, H, N, hd, bfloat):
    """The reference's top_k=False blocks (last block of each model, deit main.py:282-296): dense MXINT8
    attention == every key kept.  Checked against the oracle and through the DeiT shim."""
    q, k, v = make_qkv(B, H, N, hd, seed=9, kind="randn")
    specs = mx_specs(bfloat, False)
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, N, return_mask=True)
    assert bool(unpack_mask(mask, N).all())
    ref = O.pruned_attention(q, k, v, N, bfloat=bfloat, integer_scores=True)
    assert_out_close(out.cpu(), ref, v, N, bfloat, OUT_TOL)
    r = mxq.predict_topk(q.cuda(), k.cuda(), specs, N, return_idx=True)
    assert torch.equal(r["idx"].cpu().to(torch.int64), torch.arange(N).expand(B, H, N, N))

    from mx_quantization_b200.modules import PrunedAttentionCore
    core = PrunedAttentionCore(specs, 0)           # k = 0 <=> top_k=False
    y = core(q.cuda(), k.cuda(), v.cuda())
    assert torch.equal(y, out.permute(0, 2, 1, 3).reshape(B, N, H * hd))


# ---- SURVEY 8 f2: MX Linear (mx.Linear forward, MXINT8 activations and weights) ----------------------

def _check_linear(y, ref, bfloat):
    err = (y - ref).abs()
    scale = float(ref.abs().max())
    if bfloat == 32:
        # exact products, fp32 accumulation in a different order from the reference's BLAS
        assert float(err.max()) <= 2e-5 * scale, float(err.max()) / scale
    else:
        # the two bf16 roundings of the output flip where the fp32 sums straddle a rounding tie
        assert float(err.max()) <= 2.0 ** -7 * scale
        assert float((err > 0).float().mean()) <= 0.02


@pytest.mark.parametrize("name", ["mx_linear_qkv", "mx_linear_bf16", "mx_linear_nobias"])
def test_mx_linear_reference_golden(mxq, name):
    """Outputs of the unmodified reference mx.Linear forward (tests/golden/make_golden_linear.py)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    M, K, N, has_bias, bfloat, flush = (int(v) for v in z["meta"])
    x, w = torch.from_numpy(z["x"]).cuda(), torch.from_numpy(z["w"]).cuda()
    b = torch.from_numpy(z["b"]).cuda() if has_bias else None
    y = mxq.mx_linear(x, w, b, mx_specs(bfloat, bool(flush)))
    _check_linear(y.cpu(), torch.from_numpy(z["y"]), bfloat)


@pytest.mark.parametrize("M,K,N,bias,bfloat", [
    (300, 768, 2304, True, 32),        # DeiT-base qkv projection
    (257, 1152, 1152, True, 16),       # DiT / PixArt output projection, bfloat 16
    (64, 64, 4, False, 32),
    (1000, 3072, 768, True, 32),       # DeiT-base MLP fc2
])
def test_mx_linear_vs_oracle(mxq, M, K, N, bias, bfloat):
    g = torch.Generator().manual_seed(51)
    x = torch.randn(2, M // 2 if M % 2 == 0 else M, K, generator=g)[: 2 if M % 2 == 0 else 1]
    x = x * torch.exp(0.5 * torch.randn(*x.shape[:-1], 1, generator=g))
    w = torch.randn(N, K, generator=g) * K ** -0.5
    b = torch.randn(N, generator=g) * 0.1 if bias else None
    specs = mx_specs(bfloat, False)
    from mx_quantization_b200.modules import MxLinear
    lin = MxLinear(K, N, bias=bias, mx_specs=specs).cuda()
    with torch.no_grad():
        lin.weight.copy_(w)
        if bias:
            lin.bias.copy_(b)
        y = lin(x.cuda())
        y2 = lin(x.cuda())                                   # cached weight operand
    assert torch.equal(y, y2)
    ref = O.mx_linear(x, w, b, bfloat=bfloat)
    assert y.shape == ref.shape
    _check_linear(y.cpu(), ref, bfloat)


@pytest.mark.parametrize("bias_kind", ["mask_-10000", "arbitrary_fp32", "dyadic_small", "half_masked_-1e4_hd64"])
def test_key_bias_variants(mxq, bias_kind):
    """Additive key bias: the integer-key fast path (bias carried through the MMA, exact) and the fp32
    fallback (bias with more than 16 significant bits / not a multiple of the row's 2^(g+1)) must both
    reproduce the oracle's sets."""
    B, H, Nq, S, hd, top_k = 2, 2, 96, 120, (64 if "hd64" in bias_kind else 72), 50
    g = torch.Generator().manual_seed(77)
    q = torch.randn(B, H, Nq, hd, generator=g)
    k = torch.randn(B, H, S, hd, generator=g)
    v = torch.randn(B, H, S, hd, generator=g)
    if bias_kind.startswith("mask") or bias_kind.startswith("half"):
        keep = torch.zeros(B, S); keep[0, :31] = 1; keep[1, :60] = 1
        bias = (1 - keep) * -10000.0
    elif bias_kind == "arbitrary_fp32":
        bias = torch.randn(B, S, generator=g) * 3.0
    else:
        bias = torch.randint(-8, 9, (B, S), generator=g).float() * 0.5
    specs = mx_specs(32, True)
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True,
                                     key_bias=bias.reshape(B, 1, 1, S).cuda())
    ref = O.pruned_attention(q, k, v, top_k, flush=True, integer_scores=True, key_bias=bias.reshape(B, 1, 1, S))
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], S), S)
    assert torch.equal(unpack_mask(mask, S), want)
    assert_out_close(out.cpu(), ref, v, S, 32, OUT_TOL)


@pytest.mark.parametrize("B,H,Nq,Nk,hd,top_k,bfloat,flush", [
    (1, 1, 1, 1, 32, 1, 32, False),        # single query, single key
    (1, 2, 5, 3, 40, 2, 32, True),
    (2, 1, 17, 256, 48, 1, 32, False),     # k = 1
    (1, 3, 130, 33, 80, 33, 32, False),    # k = Nk (dense), two tiles
    (1, 1, 257, 129, 104, 64, 32, True),   # three tiles, NC = 7 path with Nk = 129
    (1, 2, 64, 225, 128, 100, 32, False),  # NC = 8 with padding columns, head_dim 128
    (2, 2, 300, 257, 64, 77, 32, False),   # just past the single-key-block limit
    (1, 1, 40, 300, 36, 30, 32, False),    # head_dim % 8 != 0 -> CUDA-core predictor; Nk > 256 unsupported for attention
])
def test_odd_shapes(mxq, B, H, Nq, Nk, hd, top_k, bfloat, flush):
    """Corner shapes found useful by tools/fuzz_parity.py (which runs ~1000 random ones)."""
    g = torch.Generator().manual_seed(123)
    q = torch.randn(B, H, Nq, hd, generator=g)
    k = torch.randn(B, H, Nk, hd, generator=g)
    v = torch.randn(B, H, Nk, hd, generator=g)
    specs = mx_specs(bfloat, flush)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, flush=flush, integer_scores=True)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], Nk), Nk)
    r = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True)
    assert torch.equal(unpack_mask(r["mask"], Nk), want)
    assert torch.equal(r["idx"].cpu().to(torch.int64), torch.sort(ref["idx"], dim=-1).values)
    if hd % 8 == 0:
        out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True)
        assert torch.equal(mask, r["mask"])
        assert_out_close(out.cpu(), ref, v, Nk, bfloat, OUT_TOL)
    else:
        with pytest.raises(ValueError):             # unsupported combination: loud, no fallback
            mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k)


def test_cuda_graph_capture_and_replay(mxq):
    """The library allocates nothing, never synchronises and enqueues on the caller's stream, so a
    whole call (three kernels, tensor maps baked into the launch parameters) captures into a CUDA
    graph; replaying it on new input values in the same buffers gives the eager result."""
    B, H, N, hd, top_k = 2, 3, 197, 64, 30
    specs = mx_specs(32, False)
    g = torch.Generator(device="cuda").manual_seed(3)
    buf = torch.randn(B, N, 3, H, hd, device="cuda", generator=g)
    qkv = buf.permute(2, 0, 3, 1, 4)
    out = torch.empty(B, N, H, hd, device="cuda")
    mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k, out=out.permute(0, 2, 1, 3))      # warm-up (attributes set)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k, out=out.permute(0, 2, 1, 3))
    buf.copy_(torch.randn(B, N, 3, H, hd, device="cuda", generator=g))                              # new activations
    graph.replay()
    torch.cuda.synchronize()
    got = out.clone()
    want = mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k).permute(0, 2, 1, 3)
    assert torch.equal(got, want.contiguous())


# ---- the reference's other rankings (SURVEY 8 f3): partial_Q / partial_K / top-k of the true scores ----
MODES = ["partial_Q", "partial_K", "MXINT4", "two_step_leading_ones", "true_ex", "exact"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["modes_deit", "modes_dit_bf16", "modes_pixart", "modes_deit_197"])
def test_other_rankings_reference_golden(mxq, name, mode):
    """Masks and outputs of the unmodified reference (tests/golden/make_golden_modes.py)."""
    d, m = load_golden(name)
    specs = mx_specs(m["bfloat"], m["flush"])
    q, k, v = d["q"].cuda(), d["k"].cuda(), d["v"].cuda()
    out, mask = mxq.pruned_attention(q, k, v, specs, m["top_k"], return_mask=True, pred_mode=mode)
    got = unpack_mask(mask, m["N"])
    want = torch.zeros_like(got)
    want.scatter_(-1, d[f"{mode}.idx"], True)
    assert torch.equal(got, want)
    r = O.pruned_attention(d["q"], d["k"], d["v"], m["top_k"], bfloat=m["bfloat"], flush=m["flush"],
                           idx=d[f"{mode}.idx"])
    ref = {"true_vals": r["true_vals"], "idx": d[f"{mode}.idx"], "out": d[f"{mode}.out"]}
    assert_out_close(out.cpu(), ref, d["v"], m["N"], m["bfloat"], OUT_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B,H,Nq,Nk,hd,kfrac,bfloat,kind", [
    (2, 3, 197, 197, 64, 0.15, 32, "randn"),
    (1, 2, 256, 256, 72, 0.6, 16, "randn"),
    (1, 2, 130, 77, 72, 0.3, 32, "edges"),          # rectangular, two query tiles, ragged key chunk
    (1, 1, 64, 32, 32, 0.5, 32, "randn"),
    (2, 2, 100, 224, 128, 0.05, 32, "randn"),
    (1, 2, 197, 197, 64, 0.2, 32, "lognormal"),     # wide exponent spread: ranks on the ordered fp32 key
    (1, 1, 40, 40, 64, 1.0, 32, "randn"),           # every key kept
])
def test_other_rankings_vs_oracle(mxq, B, H, Nq, Nk, hd, kfrac, bfloat, kind, mode):
    top_k = max(1, min(Nk, int(round(kfrac * Nk))))
    q, k, v = make_qkv(B, H, Nq, hd, seed=31, kind=kind, Nk=Nk)
    specs = mx_specs(bfloat, False)
    res = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True, pred_mode=mode)
    ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, pred_mode=mode)
    want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], Nk), Nk)
    got = unpack_mask(res["mask"], Nk)
    if kind == "lognormal":
        # terms of one pair can spread past the tensor core's exact window (and past fp32's 24 bits, where
        # the reference's own BLAS order decides): near-ties may flip there.  Rows whose every pair keeps its
        # block terms (operand widths included) inside 20 bits are pinned and must be bit-equal
        pinned = mode_window_ok(ref["q_codes"], ref["q_exps"], ref["k_codes"], ref["k_exps"], hd, mode)
        assert torch.equal(got[pinned], want[pinned])
        print(f"{mode} lognormal: {int((~pinned).sum())} of {pinned.numel()} rows exempt")
        assert float((got == want).all(-1).float().mean()) > 0.97
        assert bool((got.sum(-1) == top_k).all())
    else:
        assert torch.equal(got, want)
        assert torch.equal(res["idx"].cpu().to(torch.int64), torch.sort(ref["idx"], dim=-1).values)
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True, pred_mode=mode)
    assert torch.equal(mask, res["mask"])
    ref2 = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, idx=canonical_idx_from_mask(unpack_mask(mask, Nk), top_k))
    assert_out_close(out.cpu(), ref2, v, Nk, bfloat, OUT_TOL)


@pytest.mark.gpu
def test_other_rankings_full_size_properties(mxq):
    """DeiT-base layer shape (B=256,H=12,N=197,hd=64,k=30): every row keeps exactly k keys; the 'exact' ranking
    keeps, per row, a set whose smallest true score is >= every dropped key's (checked on a head sample)."""
    B, H, N, hd, top_k = 256, 12, 197, 64, 30
    g = torch.Generator(device="cuda").manual_seed(3)
    q = torch.randn(B, H, N, hd, device="cuda", generator=g)
    k = torch.randn(B, H, N, hd, device="cuda", generator=g)
    specs = mx_specs(32, False)
    for mode in MODES:
        mask = mxq.predict_topk(q, k, specs, top_k, pred_mode=mode)["mask"]
        bits = (mask.to(torch.int64) & 0xFFFFFFFF)
        cnt = sum(((bits >> s) & 1) for s in range(32)).sum(-1)
        assert bool((cnt == top_k).all()), mode
        sl = (slice(0, 256, 97), slice(0, 12, 5))
        ref = O.pruned_attention(q[sl].cpu(), k[sl].cpu(), k[sl].cpu(), top_k, pred_mode=mode)
        want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], N), N)
        assert torch.equal(unpack_mask(mask[sl], N), want), mode


@pytest.mark.gpu
@torch.no_grad()
def test_other_rankings_module_and_errors(mxq):
    from mx_quantization_b200.modules import Attention
    torch.manual_seed(0)
    specs = mx_specs(16, False)
    x = torch.randn(2, 64, 128, device="cuda")
    outs = {}
    for name, kw in {"ex": dict(ex_pred=True, pred_mode="ex_pred"), "pq": dict(ex_pred=True, pred_mode="partial_Q"),
                     "exact": dict(ex_pred=False)}.items():
        torch.manual_seed(1)
        m = Attention(128, num_heads=2, qkv_bias=True, mx_quant=True, mx_specs=specs, top_k=True, k=16, **kw).cuda()
        outs[name] = m(x)
        assert outs[name].shape == x.shape and bool(torch.isfinite(outs[name]).all())
    assert not torch.equal(outs["ex"], outs["exact"])
    with pytest.raises(NotImplementedError):
        Attention(128, num_heads=2, mx_quant=True, mx_specs=specs, top_k=True, k=16, ex_pred=True, pred_mode="sanger")
    q = torch.randn(1, 1, 300, 64, device="cuda")
    with pytest.raises(ValueError):                      # modes 1-3: Nk <= 256
        mxq.predict_topk(q, q, specs, 10, pred_mode="partial_K")
    with pytest.raises(NotImplementedError):
        mxq.predict_topk(q, q, specs, 10, pred_mode="sanger")
    big = torch.randn(1, 1, 256, 128, device="cuda")       # two-part operands: head_dim 128 x 256 keys do not fit
    with pytest.raises(ValueError, match="shared memory"):
        mxq.predict_topk(big, big, specs, 10, pred_mode="two_step_leading_ones")


@pytest.mark.parametrize("mode", MODES)
def test_cross_attention_other_rankings_golden(mxq, mode):
    """Cross-attention (Nq != Nk) with the additive text mask in the other ranking modes; "exact" is what an
    excluded timestep runs (MX_transformer_block.py:806,833-834).  Reference-generated fixture."""
    d, m = _load_cross("modes_pixart_cross")
    specs = mx_specs(m["bfloat"], m["flush"])
    bias = d["key_bias"].reshape(m["B"], 1, 1, m["S"]).cuda()
    out, mask = mxq.pruned_attention(d["q"].cuda(), d["k"].cuda(), d["v"].cuda(), specs, m["top_k"],
                                     scale=1.0 / (m["hd"] ** 0.5), return_mask=True, key_bias=bias, pred_mode=mode)
    got = unpack_mask(mask, m["S"])
    idx = d[f"{mode}.idx"].to(torch.int64)
    want = torch.zeros_like(got)
    want.scatter_(-1, idx, True)
    assert torch.equal(got, want)
    r = O.pruned_attention(d["q"], d["k"], d["v"], m["top_k"], scale=1.0 / (m["hd"] ** 0.5), bfloat=m["bfloat"],
                           flush=m["flush"], key_bias=d["key_bias"].reshape(m["B"], 1, 1, m["S"]), idx=idx)
    ref = {"true_vals": r["true_vals"], "idx": idx, "out": d[f"{mode}.out"]}
    assert_out_close(out.cpu(), ref, d["v"], m["S"], m["bfloat"], OUT_TOL)
    sel = mxq.predict_topk(d["q"].cuda(), d["k"].cuda(), specs, m["top_k"], pred_mode=mode,
                           scale=1.0 / (m["hd"] ** 0.5), key_bias=bias)
    assert torch.equal(sel["mask"], mask)


@torch.no_grad()
def test_exclude_timesteps_in_shims(mxq):
    """DiT / PixArt self-attention run dense attention on the listed steps (models.py:172,
    MX_transformer_block.py:656); PixArt cross-attention ranks on the true scores there (:806,833-834)."""
    from mx_quantization_b200.modules import Attention, MXCrossAttention
    specs = mx_specs(16, False)
    torch.manual_seed(0)
    x = torch.randn(2, 64, 128, device="cuda")
    torch.manual_seed(1)
    a = Attention(128, num_heads=2, qkv_bias=True, mx_quant=True, mx_specs=specs, top_k=True, k=16, ex_pred=True,
                  exclude_timesteps=[1]).cuda()
    torch.manual_seed(1)
    dense = Attention(128, num_heads=2, qkv_bias=True, mx_quant=True, mx_specs=specs, top_k=False).cuda()
    y0, y1, y2 = a(x), a(x), a(x)
    assert torch.equal(y0, y2) and not torch.equal(y0, y1)
    assert torch.equal(y1, dense(x))
    torch.manual_seed(2)
    c = MXCrossAttention(128, 2).cuda().set_config(mx_quant=True, mx_specs=specs, top_k=True, k=8, ex_pred=True,
                                                    exclude_timesteps=[0])
    enc = torch.randn(2, 40, 128, device="cuda")
    am = torch.zeros(2, 1, 40, device="cuda")
    am[0, 0, 25:] = -10000.0
    z0, z1 = c(x, encoder_hidden_states=enc, attention_mask=am), c(x, encoder_hidden_states=enc, attention_mask=am)
    assert z0.shape == x.shape and bool(torch.isfinite(z0).all()) and not torch.equal(z0, z1)


@pytest.mark.parametrize("name", ["elsa_deit", "elsa_dit", "elsa_edges"])
def test_elsa_reference_golden(mxq, name):
    """ELSA ranking (funcs/elsa_approximation.py): masks against the unmodified reference.  A hash bit is the sign of
    an fp32 projection; the fixture records how close the closest one comes to 0 (relative to its row) - above a few
    fp32 rounding errors every mask must match, below that a row may differ where its hash flipped."""
    d, m = load_golden(name)
    specs = mx_specs(m["bfloat"], m["flush"])
    q, k, v, P = d["q"].cuda(), d["k"].cuda(), d["v"].cuda(), d["P"].cuda()
    out, mask = mxq.pruned_attention(q, k, v, specs, m["top_k"], return_mask=True, pred_mode="ELSA", orthogonal_matrix=P)
    got = unpack_mask(mask, m["N"])
    want = torch.zeros_like(got)
    want.scatter_(-1, d["idx"], True)
    assert bool((got.sum(-1) == m["top_k"]).all())
    rows_equal = float((got == want).all(-1).float().mean())
    if float(d["hash_margin"][0]) > 5e-6:
        assert rows_equal == 1.0
        r = O.pruned_attention(d["q"], d["k"], d["v"], m["top_k"], bfloat=m["bfloat"], flush=m["flush"], idx=d["idx"])
        ref = {"true_vals": r["true_vals"], "idx": d["idx"], "out": d["out"]}
        assert_out_close(out.cpu(), ref, d["v"], m["N"], m["bfloat"], OUT_TOL)
    else:
        assert rows_equal > 0.98
    sel = mxq.predict_topk(q, k, specs, m["top_k"], pred_mode="ELSA", orthogonal_matrix=P, return_idx=True)
    assert torch.equal(sel["mask"], mask)


@torch.no_grad()
def test_elsa_module_and_errors(mxq):
    from mx_quantization_b200.modules import Attention
    specs = mx_specs(16, False)
    torch.manual_seed(0)
    x = torch.randn(2, 64, 128, device="cuda")
    P = torch.linalg.qr(torch.randn(64, 64))[0].cuda()
    m = Attention(128, num_heads=2, qkv_bias=True, mx_quant=True, mx_specs=specs, top_k=True, k=16, ex_pred=True,
                  pred_mode="ELSA", orthogonal_matrix=P).cuda()
    y = m(x)
    assert y.shape == x.shape and bool(torch.isfinite(y).all())
    with pytest.raises(ValueError):
        Attention(128, num_heads=2, mx_quant=True, mx_specs=specs, top_k=True, k=16, ex_pred=True, pred_mode="ELSA")
    q = torch.randn(1, 1, 64, 64, device="cuda")
    with pytest.raises(ValueError):                      # Nq != Nk
        mxq.predict_topk(q, q[:, :, :32], specs, 8, pred_mode="ELSA", orthogonal_matrix=P)
    with pytest.raises(ValueError):                      # matrix shape
        mxq.predict_topk(q, q, specs, 8, pred_mode="ELSA", orthogonal_matrix=P[:32])


@torch.no_grad()
def test_anal_flag_reports_coverage(mxq, capsys):
    """--anal (main.py:134-136): the shims print / keep "Average chosen k" = funcs/analysis.py total_chosen_k,
    computed from the kept-key bitmask."""
    from mx_quantization_b200.modules import Attention
    specs = mx_specs(32, False)
    torch.manual_seed(0)
    x = torch.randn(2, 48, 128, device="cuda")
    torch.manual_seed(1)
    a = Attention(128, num_heads=2, qkv_bias=True, mx_quant=True, mx_specs=specs, top_k=True, k=12, ex_pred=True,
                  anal=True).cuda()
    y = a(x)
    assert "Average chosen k:" in capsys.readouterr().out
    qkv = a.qkv(x).reshape(2, 48, 3, 2, 64).permute(2, 0, 3, 1, 4)
    _, mask = mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, 12, return_mask=True)
    idx = canonical_idx_from_mask(unpack_mask(mask, 48), 12)
    want = np.mean([len(torch.unique(idx[b, h])) / 48 for b in range(2) for h in range(2)])   # total_chosen_k
    assert abs(a.core.avg_chosen_k - want) < 1e-12 and y.shape == x.shape


def test_apply_quantization_to_deit(mxq):
    """The model-patching helper with the reference's block policy (workloads/deit/scripts/main.py:231-318) on a
    timm-shaped toy model: last block dense, excluded blocks on another ranking, MLPs on MX Linear."""
    import torch.nn as nn
    from mx_quantization_b200.modules import (MxLinear, QuantizedAttention, QuantizedMlp, apply_quantization_to_deit)

    class _Attn(nn.Module):
        def __init__(self, dim, heads):
            super().__init__()
            self.num_heads, self.scale = heads, (dim // heads) ** -0.5
            self.qkv, self.proj, self.proj_drop = nn.Linear(dim, 3 * dim), nn.Linear(dim, dim), nn.Dropout(0.0)

    class _Mlp(nn.Module):
        def __init__(self, dim):
            super().__init__()
            self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), nn.GELU(), nn.Linear(4 * dim, dim), nn.Dropout(0.0)

    class _Block(nn.Module):
        def __init__(self, dim, heads):
            super().__init__()
            self.norm1, self.attn, self.norm2, self.mlp = nn.LayerNorm(dim), _Attn(dim, heads), nn.LayerNorm(dim), _Mlp(dim)

        def forward(self, x):
            x = x + self.attn(self.norm1(x))
            return x + self.mlp(self.norm2(x))

    torch.manual_seed(0)
    model = nn.Module()
    model.blocks = nn.ModuleList([_Block(128, 2) for _ in range(3)])
    cfg = {"blocks": [0, 1, 2], "components": ["attn", "ffn"], "mx_specs": mx_specs(32, False)}
    apply_quantization_to_deit(model, cfg, top_k=True, k=10, approx_flag=True, pred_mode="ex_pred",
                               exclude_blocks=[1], exclude_block_type="partial_Q", dense_blocks=(2,))
    model.cuda()
    assert all(isinstance(b.attn, QuantizedAttention) and isinstance(b.mlp, QuantizedMlp) for b in model.blocks)
    assert isinstance(model.blocks[0].mlp.fc1, MxLinear)
    assert [b.attn.core.pred_mode for b in model.blocks] == ["ex_pred", "partial_Q", "ex_pred"]
    assert [b.attn.core.k for b in model.blocks] == [10, 10, 0]          # last block: every key kept
    x = torch.randn(2, 50, 128, device="cuda")
    with pytest.raises(RuntimeError):            # inference forward only: grad mode with trainable weights is refused
        model.blocks[0](x)
    with torch.no_grad():
        for b in model.blocks:
            x = b(x)
    assert x.shape == (2, 50, 128) and bool(torch.isfinite(x).all())
    # the reference hard-codes block 11 as the dense one (main.py:266,281,296): the default leaves a 3-block model pruned
    model2 = nn.Module()
    model2.blocks = nn.ModuleList([_Block(128, 2) for _ in range(3)])
    apply_quantization_to_deit(model2, cfg, top_k=True, k=10)
    assert [b.attn.core.k for b in model2.blocks] == [10, 10, 10]


@pytest.mark.parametrize("Nk", [193, 197, 200, 207, 208, 209, 216, 223, 224])
@pytest.mark.parametrize("kind,hd,bfloat", [("randn", 64, 32), ("edges", 72, 16), ("lognormal", 64, 32)])
def test_tight_lane_split_key_counts(mxq, Nk, kind, hd, bfloat):
    """193 .. 224 keys: the selection splits a row's key columns between its two lanes at 104 / 112 instead of 128
    and writes the row mask byte-wise (k_predict_topk_tc<7, .., HG = 13 / 14>); masks, indices and outputs against
    the oracle, square and rectangular, several k (ties included through the 'edges' rows)."""
    for Nq, top_k in ((Nk, 30), (Nk, 1), (Nk, Nk - 1), (150, 77), (260, max(2, Nk // 2))):
        q, k, v = make_qkv(2, 2, Nq, hd, seed=Nk + top_k, kind=kind if Nq == Nk else "randn", Nk=Nk)
        specs = mx_specs(bfloat, False)
        res = mxq.predict_topk(q.cuda(), k.cuda(), specs, top_k, return_idx=True)
        ref = O.pruned_attention(q, k, v, top_k, bfloat=bfloat, integer_scores=True)
        want = O.mask_words_to_dense(O.idx_to_mask_words(ref["idx"], Nk), Nk)
        assert torch.equal(unpack_mask(res["mask"], Nk), want), (Nq, top_k)
        assert torch.equal(res["idx"].cpu().to(torch.int64), torch.sort(ref["idx"], dim=-1).values), (Nq, top_k)
        # bits past Nk in the last mask word stay clear
        last = res["mask"][..., -1].cpu().to(torch.int64) & 0xFFFFFFFF
        assert int((last >> (Nk - 32 * ((Nk - 1) // 32))).max()) == 0 or Nk % 32 == 0
    out, mask = mxq.pruned_attention(q.cuda(), k.cuda(), v.cuda(), specs, top_k, return_mask=True)
    assert torch.equal(mask, res["mask"])
    assert_out_close(out.cpu(), ref, v, Nk, bfloat, OUT_TOL)
