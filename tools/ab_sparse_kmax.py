#!/usr/bin/env python
"""A/B aid for the cost-follows-k epilogue's register path (csrc/mxprune_attend_sparse.cuh): two builds of libmxprune
(MXPRUNE_LIB selects the library) compared output for output and timed against each other.

    MXPRUNE_LIB=A.so python tools/ab_sparse_kmax.py dump A.pt      outputs + masks of CASES, both launch plans
    python tools/ab_sparse_kmax.py compare A.pt B.pt                byte-for-byte comparison of two dumps
    python tools/ab_sparse_kmax.py alternate A.so B.so [...]        three rounds, the builds in rotated order, each:
                                                                    bench.py --no-e2e --no-cpu-baseline and the
                                                                    stand-alone k_attend_sparse time; one JSON line each

The stand-alone kernel is timed at 192 DeiT-base heads (16 x 12, k = 30), where the default policy takes the three
kernels (between 1 and 1.7 heads per SM; see fused_try); bench.py's three_kernel_path runs the dense epilogue
(fused path 0) and does not reach it."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [  # fused path, B, H, N, hd, top_k, kind, bfloat, flush, dtype
    (1, 24, 12, 197, 64, 30, "randn", 32, False, "float32"),       # fused launch
    (1, 24, 12, 197, 64, 32, "randn", 32, False, "float32"),
    (1, 24, 12, 197, 64, 33, "randn", 32, False, "float32"),
    (1, 24, 12, 197, 64, 30, "lognormal", 16, True, "float32"),    # slow exponent path
    (1, 24, 12, 197, 64, 12, "lognormal", 32, False, "float32"),
    (1, 8, 9, 197, 32, 30, "edges", 32, False, "float32"),         # run-time head_dim
    (1, 24, 12, 197, 64, 30, "randn", 32, False, "bfloat16"),
    (1, 16, 12, 197, 64, 30, "randn", 32, False, "float32"),       # 192 heads: three kernels, k_attend_sparse
    (1, 2, 12, 197, 64, 32, "randn", 32, False, "float32"),        # 24 heads: three kernels, k_attend_sparse
    (1, 2, 12, 197, 64, 33, "randn", 32, False, "float32"),
    (1, 2, 12, 197, 64, 30, "lognormal", 16, True, "float32"),
    (1, 2, 9, 197, 32, 30, "edges", 32, False, "float32"),
    (1, 2, 12, 197, 64, 30, "randn", 32, False, "bfloat16"),
    (1, 8, 12, 256, 72, 26, "edges", 32, True, "float32"),         # head_dim 72: three kernels, k_attend_sparse
    (2, 8, 12, 256, 72, 26, "edges", 32, True, "float32"),         # the same forced into the fused launch
]


def dump(path):
    import torch
    import mx_quantization_b200 as m
    from tests.helpers import fused_qkv_views, make_qkv, mx_specs
    res = {}
    try:
        for mode, B, H, N, hd, top_k, kind, bf, fl, dt in CASES:
            m.set_fused_path(mode)
            q, k, v = make_qkv(B, H, N, hd, seed=7, kind=kind)
            tdt = getattr(torch, dt)
            qv, kv, vv = fused_qkv_views(q.to(tdt).cuda(), k.to(tdt).cuda(), v.to(tdt).cuda())
            out, mask = m.pruned_attention(qv, kv, vv, mx_specs(bf, fl), top_k, return_mask=True)
            key = f"path{mode}_{B}x{H}x{N}_hd{hd}_k{top_k}_{kind}_bf{bf}_fl{int(fl)}_{dt}"
            res[key] = (out.cpu(), mask.cpu(), m.last_launch_count())
    finally:
        m.set_fused_path(1)
    torch.save(res, path)
    print(f"{len(res)} cases from {m._lib.LIB_PATH} -> {path}")


def compare(pa, pb):
    import torch
    a, b = torch.load(pa), torch.load(pb)
    bits = lambda t: t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)
    ok = True
    for key in a:
        (oa, ma, la), (ob, mb, lb) = a[key], b[key]
        same = oa.dtype == ob.dtype and torch.equal(bits(oa), bits(ob)) and torch.equal(ma, mb) and la == lb
        ok &= same
        print(f"{key}: {'identical' if same else 'DIFFERENT'} ({la} / {lb} launches)")
    print("all identical" if ok else "OUTPUTS DIFFER")
    return 0 if ok else 1


def time_sparse(iters=50):
    """Mean device time of k_attend_sparse at 192 DeiT-base heads (torch.profiler, after a warm-up)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    import mx_quantization_b200 as m
    from tests.helpers import fused_qkv_views, make_qkv, mx_specs
    q, k, v = make_qkv(16, 12, 197, 64, seed=3)
    qv, kv, vv = fused_qkv_views(q.cuda(), k.cuda(), v.cuda())
    for _ in range(10):
        m.pruned_attention(qv, kv, vv, mx_specs(), 30)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            m.pruned_attention(qv, kv, vv, mx_specs(), 30)
        torch.cuda.synchronize()
    ts = [ev.time_range.elapsed_us() for ev in prof.events()
          if ev.device_type == torch.autograd.DeviceType.CUDA and "k_attend_sparse" in ev.name]
    assert len(ts) == iters, f"expected {iters} k_attend_sparse launches, saw {len(ts)}"
    print(json.dumps({"k_attend_sparse_ms": sum(ts) / len(ts) / 1e3}))


def alternate(libs, rounds=3):
    for r in range(rounds):
        order = libs[r % len(libs):] + libs[:r % len(libs)]
        for lib in order:
            env = dict(os.environ, MXPRUNE_LIB=os.path.abspath(lib))
            line = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-e2e", "--no-cpu-baseline"],
                                  env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
            d = json.loads(line)
            ks = json.loads(subprocess.run([sys.executable, __file__, "time"], env=env, capture_output=True, text=True,
                                           check=True).stdout.strip().splitlines()[-1])
            print(json.dumps({"kind": "result", "round": r + 1, "lib": lib, "ms_per_step": d["ms_per_step"],
                              "fused_ms": d["roofline"]["avg_ms"], **ks,
                              "dense_exact_attention_ms": d["roofline"]["three_kernel_path"]["kernels"]["exact_attention"]["avg_ms"],
                              "other_ms_per_step": {k: v["ms_per_step"] for k, v in d.get("other_workloads", {}).items()}}),
                  flush=True)


if __name__ == "__main__":
    cmd = sys.argv[1] if len(sys.argv) > 1 else ""
    if cmd == "dump":
        dump(sys.argv[2])
    elif cmd == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    elif cmd == "time":
        time_sparse()
    elif cmd == "alternate":
        alternate(sys.argv[2:])
    else:
        sys.exit(__doc__)
