#!/usr/bin/env python
"""bf16 activations through whole modules: what a bf16 DiT / DeiT pipeline gains from running the MX Linear
projections and the attention shims natively instead of through an fp32 copy of the model.

Three arms per case, run alternating in one process (round-robin over --rounds, each round timing --steps steps of
every arm after --warmup warm-up steps; the best round is reported):
  a  fp32      the fp32 module on fp32 x
  b  bf16      the same module .to(torch.bfloat16) on bf16 x, read and written natively
  c  bf16_cvt  bf16 x -> .float() -> the fp32 module -> .to(torch.bfloat16) (what a bf16 pipeline had to do before)
The fp32 module holds the widened bf16 parameters (a bf16 model's fp32 copy), so b and c compute from the same values.
Cases:
  deit_base_attention   QuantizedAttention, 256 x 197 tokens, C 768, 12 heads, k 30, bfloat 32
  dit_xl2_attention     DiT Attention, 256 x 256 tokens, C 1152, 16 heads of 72, k 154, bfloat 16, qkv bias
  linear_{qkv,proj,fc1,fc2}   MxLinear alone at DeiT-base's projection shapes (M = 256 x 197 tokens), bfloat 32
Every step runs the module on --inputs distinct input tensors in turn, so that the inputs of one step (at least
310 MB in bf16) do not fit the 126 MB L2.  Device time from CUDA events around whole steps, reported per module call.
outputs_equal_b_c says whether b's and c's outputs are bit-identical on the last input; under bfloat 16 the fp32
module's every layer boundary is a bf16 value, so for dit_xl2_attention they must be.
After the timing, one torch.profiler pass per linear case gives the device time of each kernel of arms a and b
(kernel_us), which compares the GEMM with fp32 output against the GEMM with bf16 output.
Writes a JSONL file (default profiles/half_module_b200.jsonl) whose first line records the GPU's name and power limit.
    python tools/bench_half_module.py [--steps 10] [--rounds 5] [--out profiles/half_module_b200.jsonl]"""
import argparse
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from bench import mx_specs  # noqa: E402
from mx_quantization_b200.modules import Attention, MxLinear, QuantizedAttention  # noqa: E402

ARMS = ("fp32", "bf16", "bf16_cvt")
DEIT_TOKENS = 256 * 197


class _TimmAttention(nn.Module):            # the attributes QuantizedAttention takes from timm's Attention
    def __init__(self, dim, heads):
        super().__init__()
        self.num_heads, self.scale = heads, (dim // heads) ** -0.5
        self.qkv, self.proj = nn.Linear(dim, 3 * dim), nn.Linear(dim, dim)
        self.proj_drop = nn.Identity()


def cases():
    return {
        "deit_base_attention": (lambda: QuantizedAttention(_TimmAttention(768, 12), mx_quant=True,
                                                           mx_specs=mx_specs(32, False), top_k=True, k=30),
                                (256, 197, 768)),
        "dit_xl2_attention": (lambda: Attention(1152, num_heads=16, qkv_bias=True, mx_quant=True,
                                                mx_specs=mx_specs(16, False), top_k=True, k=154, ex_pred=True),
                              (256, 256, 1152)),
        "linear_qkv": (lambda: MxLinear(768, 2304, mx_specs=mx_specs(32, False)), (DEIT_TOKENS, 768)),
        "linear_proj": (lambda: MxLinear(768, 768, mx_specs=mx_specs(32, False)), (DEIT_TOKENS, 768)),
        "linear_fc1": (lambda: MxLinear(768, 3072, mx_specs=mx_specs(32, False)), (DEIT_TOKENS, 768)),
        "linear_fc2": (lambda: MxLinear(3072, 768, mx_specs=mx_specs(32, False)), (DEIT_TOKENS, 3072)),
    }


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout.strip()
    name, power, clk = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": int(clk), "torch_name": torch.cuda.get_device_name(0)}


def kernel_us(fn, reps):
    """Device time per call of each kernel fn launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.count:
            out[ev.key] = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--inputs", type=int, default=4)
    ap.add_argument("--cases", default=",".join(cases()))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "half_module_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_half_module needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    all_cases = cases()
    for cname in args.cases.split(","):
        make, xshape = all_cases[cname]
        torch.manual_seed(0)
        m16 = make().to(dev).eval().to(torch.bfloat16)
        m32 = copy.deepcopy(m16).float()                   # the fp32 copy of the bf16 model: widened parameters
        g = torch.Generator(device=dev).manual_seed(1)
        x16 = [torch.randn(*xshape, device=dev, generator=g).to(torch.bfloat16) for _ in range(args.inputs)]
        x32 = [x.float() for x in x16]
        outs = {}

        def step(arm):
            for i in range(args.inputs):
                if arm == "fp32":
                    y = m32(x32[i])
                elif arm == "bf16":
                    y = m16(x16[i])
                else:
                    y = m32(x16[i].float()).to(torch.bfloat16)
                outs[arm] = y

        with torch.no_grad():
            for arm in ARMS:
                step(arm)
            equal_b_c = bool(torch.equal(outs["bf16"], outs["bf16_cvt"]))
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
                    times[arm].append(e0.elapsed_time(e1) / (args.steps * args.inputs))
            kus = {}
            if cname.startswith("linear_"):
                kus = {"fp32": kernel_us(lambda: m32(x32[0]), 20), "bf16": kernel_us(lambda: m16(x16[0]), 20)}
        tokens = x16[0].numel() // x16[0].shape[-1]
        best = {arm: min(times[arm]) for arm in ARMS}
        rec = dict(kind="result", case=cname, x_shape=list(xshape), inputs=args.inputs, steps=args.steps,
                   rounds=args.rounds, ms_per_call={a: best[a] for a in ARMS},
                   ms_per_call_all={a: times[a] for a in ARMS},
                   tokens_per_s={a: tokens / (best[a] * 1e-3) for a in ARMS},
                   b_over_c=best["bf16"] / best["bf16_cvt"], b_over_a=best["bf16"] / best["fp32"],
                   outputs_equal_b_c=equal_b_c)
        if kus:
            rec["kernel_us"] = kus
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del m16, m32, x16, x32, outs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
