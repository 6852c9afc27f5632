#!/usr/bin/env python
"""bf16 activations on the exponent-sign path: what a bf16 user gains from passing q, k, v natively.

Three arms per workload, run alternating in one process (round-robin over --rounds, each round timing --steps steps
of every arm after the warm-up):
  fp32      q, k, v fp32 (fused qkv buffer, permuted views), fp32 output
  bf16      the same values in bf16, read natively, bf16 output
  bf16_cvt  the bf16 buffer converted with .float() every step, then the fp32 path (what a bf16 user did before)
Workloads: C2 DeiT-base (256 x 12 heads, 197 tokens, head_dim 64, k 30, 12 layers), C3 DiT-XL/2 (256 x 16, 256, 72,
k 154, bfloat 16, 28 layers), C5 (16 x 16, N 4096, 72, k 1024, timed as 4 layers).  Every layer has its own qkv buffer,
so no layer finds its inputs in the 126 MB L2: the smallest buffer, one C5 layer in bf16, is 113 MB, and the 3 other
buffers of the step pass through L2 before the same layer comes round again.  Device time from CUDA events around
whole steps.  Bytes are the algorithmic q/k/v reads plus the output write: 16 N hd per head in fp32, 8 N hd in bf16,
and for bf16_cvt the conversion pass (read 2 + write 4 bytes per q/k/v element) on top of the fp32 bytes.  Writes a JSONL file (default
profiles/half_inputs_b200.jsonl) whose first line records the GPU's name and power limit.
    python tools/bench_half_inputs.py [--steps 5] [--rounds 3] [--out profiles/half_inputs_b200.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mx_quantization_b200 as mxq  # noqa: E402
from bench import mx_specs  # noqa: E402

WORKLOADS = {
    "deit_base_c2": dict(B=256, H=12, N=197, hd=64, top_k=30, layers=12, bfloat=32),
    "dit_xl2_c3": dict(B=256, H=16, N=256, hd=72, top_k=154, layers=28, bfloat=16),
    "dit_long_c5": dict(B=16, H=16, N=4096, hd=72, top_k=1024, layers=4, bfloat=32),   # 4 buffers: see the docstring
}
ARMS = ("fp32", "bf16", "bf16_cvt")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clk = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": int(clk), "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "half_inputs_b200.jsonl"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_half_inputs needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for wname in args.workloads.split(","):
        w = WORKLOADS[wname]
        B, H, N, hd, top_k, L = w["B"], w["H"], w["N"], w["hd"], w["top_k"], w["layers"]
        specs = mx_specs(w["bfloat"], False)
        g = torch.Generator(device=dev).manual_seed(0)
        bufs16 = [torch.randn(B, N, 3, H, hd, device=dev, generator=g).to(torch.bfloat16) for _ in range(L)]
        bufs32 = [b.float() for b in bufs16]
        out32 = torch.empty(B, N, H, hd, device=dev).permute(0, 2, 1, 3)
        out16 = torch.empty(B, N, H, hd, device=dev, dtype=torch.bfloat16).permute(0, 2, 1, 3)

        def step(arm):
            for layer in range(L):
                if arm == "fp32":
                    qkv, out = bufs32[layer].permute(2, 0, 3, 1, 4), out32
                elif arm == "bf16":
                    qkv, out = bufs16[layer].permute(2, 0, 3, 1, 4), out16
                else:
                    qkv, out = bufs16[layer].float().permute(2, 0, 3, 1, 4), out32
                mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k, out=out)

        # the arms compute the same thing: outputs of the last layer agree (bf16 = fp32 rounded)
        results = {}
        for arm in ARMS:
            step(arm)
            results[arm] = (out16 if arm == "bf16" else out32).clone()
        exact = bool(torch.equal(results["bf16"], results["fp32"].to(torch.bfloat16))
                     and torch.equal(results["bf16_cvt"], results["fp32"]))
        for arm in ARMS:
            for _ in range(args.warmup):
                step(arm)
        torch.cuda.synchronize()
        times = {arm: [] for arm in ARMS}
        for _ in range(args.rounds):
            for arm in ARMS:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    step(arm)
                e1.record()
                torch.cuda.synchronize()
                times[arm].append(e0.elapsed_time(e1) / args.steps)
        heads = B * H * L
        elems = B * H * N * hd * L                                  # per tensor, all layers
        for arm in ARMS:
            ms = min(times[arm])
            bytes_ = {"fp32": 16 * elems, "bf16": 8 * elems, "bf16_cvt": 16 * elems + 3 * 6 * elems}[arm]
            rec = dict(kind="result", workload=wname, arm=arm, config=w, steps=args.steps, rounds=args.rounds,
                       ms_per_step=ms, ms_per_step_all=times[arm], heads_per_s=heads / (ms * 1e-3),
                       algorithmic_bytes=bytes_, algorithmic_gb_per_s=bytes_ / (ms * 1e-3) / 1e9,
                       outputs_exact=exact)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        del bufs16, bufs32
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
