#!/usr/bin/env python
"""Cost of the additive key bias on the long-sequence path (Nk > 256): pruned_attention with PixArt's padding mask,
with a random fp32 bias, and without a bias, on the same q / k / v.

256 heads (B = 16 x H = 16) at head_dim 72, Nq in {1024, 4096}, Nk in {300, 1024, 4096}, top_k = Nk / 4, fp32.  The
three arms run alternating in one process (round-robin over --rounds, each round timing --steps calls of every arm
after the warm-up); device time from CUDA events around the calls, median over rounds.  The fallback share is the
share of query rows the tensor-core selection (k_select_long_tc) leaves to the CUDA-core kernel (k_predict_topk_long):
rows outside the integer-key window, biases that are no multiple of a row's key unit, and thresholds below the window.
It is read from the per-row flags at the end of the selection's workspace (mxp_predict_topk_mode, pred_mode 0).
Writes a JSONL file (default profiles/long_bias_b200.jsonl) whose first line records the GPU's name and power limit.
    python tools/bench_long_bias.py [--steps 5] [--rounds 3] [--out profiles/long_bias_b200.jsonl]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mx_quantization_b200 as mxq  # noqa: E402
from bench import mx_specs  # noqa: E402

ARMS = ("pixart_mask", "random_bias", "no_bias")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clk = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": int(clk), "torch_name": torch.cuda.get_device_name(0)}


def fallback_share(q, k, bias, top_k):
    from mx_quantization_b200 import _lib, ops
    lib = _lib.load()
    B, H, Nq, hd = q.shape
    Nk = k.shape[2]
    mask = torch.empty((B, H, Nq, (Nk + 31) // 32), dtype=torch.int32, device=q.device)
    ws_bytes = lib.mxp_predict_topk_workspace_bytes(B, H, Nq, Nk, hd)
    ws = torch.zeros((ws_bytes,), dtype=torch.uint8, device=q.device)
    kb = None if bias is None else bias.reshape(B, Nk).contiguous()
    rc = lib.mxp_predict_topk_mode(ops._ptr(q), *q.stride()[:3], ops._ptr(k), *k.stride()[:3], B, H, Nq, Nk, hd, top_k,
                                   0, float(hd) ** -0.5, 32, 0, ops._ptr(kb), Nk, ops._ptr(mask), None, ops._ptr(ws),
                                   ws_bytes, ops._stream())
    _lib.check(rc, "mxp_predict_topk_mode")
    n = B * H * Nq
    start = ws_bytes - (n + 255) // 256 * 256              # the flags are the workspace's last region
    return float((ws[start:start + n] != 0).float().mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--nq", default="1024,4096")
    ap.add_argument("--nk", default="300,1024,4096")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "long_bias_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long_bias needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    B, H, hd = 16, 16, 72
    specs = mx_specs(32, False)
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for Nq in [int(x) for x in args.nq.split(",")]:
        for Nk in [int(x) for x in args.nk.split(",")]:
            top_k = Nk // 4
            g = torch.Generator(device=dev).manual_seed(Nq + Nk)
            q = torch.randn(B, H, Nq, hd, device=dev, generator=g)
            k = torch.randn(B, H, Nk, hd, device=dev, generator=g)
            v = torch.randn(B, H, Nk, hd, device=dev, generator=g)
            keep = torch.zeros(B, Nk, device=dev)
            for b in range(B):                      # valid text lengths spread over the batch
                keep[b, :max(1, (b + 1) * Nk // B)] = 1.0
            biases = {"pixart_mask": ((1 - keep) * -10000.0).reshape(B, 1, 1, Nk),
                      "random_bias": torch.randn(B, 1, 1, Nk, device=dev, generator=g),
                      "no_bias": None}
            out = torch.empty(B, H, Nq, hd, device=dev)

            def call(arm):
                mxq.pruned_attention(q, k, v, specs, top_k, out=out, key_bias=biases[arm])

            for arm in ARMS:
                for _ in range(args.warmup):
                    call(arm)
            torch.cuda.synchronize()
            times = {arm: [] for arm in ARMS}
            for _ in range(args.rounds):
                for arm in ARMS:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(args.steps):
                        call(arm)
                    e1.record()
                    e1.synchronize()
                    times[arm].append(e0.elapsed_time(e1) / args.steps)
            for arm in ARMS:
                rec = dict(kind="point", arm=arm, B=B, H=H, Nq=Nq, Nk=Nk, hd=hd, top_k=top_k,
                           ms_per_call=statistics.median(times[arm]), ms_spread=[min(times[arm]), max(times[arm])],
                           fallback_share=fallback_share(q, k, biases[arm], top_k))
                lines.append(rec)
                print(json.dumps(rec), flush=True)
            del q, k, v, out
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
