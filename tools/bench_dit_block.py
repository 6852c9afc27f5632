#!/usr/bin/env python
"""DiT block with adaLN inside the MX Linear kernels (modules.QuantizedDiTBlock: the qkv / fc1 quantizers apply the
modulation, the proj / fc2 stores apply the gated residual) against the same modules run through DiTBlock.forward's torch
composition (workloads/DiT/models.py:293-297), and each half alone.

Arms per case, run alternating in one process (round-robin over --rounds, each round timing --steps steps of every arm
after --warmup warm-up steps; best and median round reported):
  fused             QuantizedDiTBlock(x, c)
  composition       the same modules: torch LayerNorm, torch modulate, Attention shim, torch gated residual, LayerNorm,
                    modulate, QuantizedMlp (the fused mx_mlp), gated residual (what a DiT block ran before)
  attn_fused / attn_composition   the attention half alone on a precomputed norm1(x) and adaLN chunks
  mlp_fused / mlp_composition     the MLP half alone on a precomputed norm2(x) and adaLN chunks
Cases: DiT-XL/2 blocks, 256 images x 256 tokens, C = 1152, 16 heads, top-k 154, bfloat 16, tanh GELU, with fp32 x and
with bf16 x.  Every step runs on --inputs distinct x tensors in turn (302 MB each in fp32, 151 MB in bf16: larger than the
126 MB L2).  Device time from CUDA events around whole steps, per call.  outputs_equal says whether the fused and the
composition outputs are bit-identical (they must be).  After the timing, one torch.profiler pass per case gives the device
time of each kernel of the fused block and of the composition (kernel_us).  bytes_elementwise_* are the DRAM bytes, by the
algorithm from shapes (not measured), of the tensors the adaLN steps touch: per half, the composition's operand quantizer
reads the modulated x, the projection writes y, modulate reads and writes two (M, C) tensors, and the gated residual reads
y and writes gate * y, then reads x and gate * y and writes the sum (11 tensors); the fused half reads the normalized x
and the residual and writes the sum (3 tensors).
Writes a JSONL file (default profiles/dit_block_b200.jsonl) whose first line records the GPU's name and power limit
from a read-only nvidia-smi query.
    python tools/bench_dit_block.py [--steps 5] [--rounds 5] [--out profiles/dit_block_b200.jsonl]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from bench import mx_specs  # noqa: E402
from mx_quantization_b200.modules import Attention, QuantizedDiTBlock  # noqa: E402
from tools.bench_half_module import gpu_info, kernel_us  # noqa: E402

ARMS = ("fused", "composition", "attn_fused", "attn_composition", "mlp_fused", "mlp_composition")
CASES = {  # images, tokens, C, heads, top_k, dtype
    "dit_xl2_fp32": (256, 256, 1152, 16, 154, torch.float32),
    "dit_xl2_bf16": (256, 256, 1152, 16, 154, torch.bfloat16),
}


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1, self.act, self.fc2 = nn.Linear(dim, hidden), nn.GELU(approximate="tanh"), nn.Linear(hidden, dim)


class _DiTBlock(nn.Module):
    """DiTBlock.__init__ (workloads/DiT/models.py:276-289) with the Attention shim."""

    def __init__(self, C, heads, top_k, sp):
        super().__init__()
        self.norm1 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn = Attention(C, num_heads=heads, qkv_bias=True, mx_quant=True, mx_specs=sp, top_k=True, k=top_k,
                              ex_pred=True)
        self.norm2 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.mlp = _Mlp(C, 4 * C)
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(C, 6 * C, bias=True))


def _modulate(x, shift, scale):
    return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)


def composition(blk, x, c):
    """DiTBlock.forward (models.py:293-297) on QuantizedDiTBlock's modules."""
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = blk.adaLN_modulation(c).chunk(6, dim=1)
    x = x + gate_msa.unsqueeze(1) * blk.attn(_modulate(blk.norm1(x), shift_msa, scale_msa))
    return x + gate_mlp.unsqueeze(1) * blk.mlp(_modulate(blk.norm2(x), shift_mlp, scale_mlp))


def traffic(M, C, es):
    """DRAM bytes of the (M, C) tensors the adaLN steps touch, by the algorithm (es = bytes per element)."""
    t = M * C * es
    return dict(composition=2 * 11 * t, fused=2 * 3 * t, removed=2 * 8 * t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--inputs", type=int, default=2)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "dit_block_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dit_block needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for cname in args.cases.split(","):
        B, T, C, heads, top_k, dt = CASES[cname]
        sp = mx_specs(16, False)
        torch.manual_seed(0)
        blk = QuantizedDiTBlock(_DiTBlock(C, heads, top_k, sp), mx_specs=sp).to(dev).to(dt).eval()
        with torch.no_grad():                   # adaLN-Zero initialises the modulation to zero: use a trained-like one
            blk.adaLN_modulation[1].weight.normal_(0, 0.02)
            blk.adaLN_modulation[1].bias.normal_(0, 0.2)
        g = torch.Generator(device=dev).manual_seed(1)
        xs = [torch.randn(B, T, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        cs = [torch.randn(B, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        with torch.no_grad():
            chunks = [blk.adaLN_modulation(c).chunk(6, dim=1) for c in cs]
            n1 = [blk.norm1(x) for x in xs]
            n2 = [blk.norm2(x) for x in xs]
            attn, mlp = blk.attn, blk.mlp
            arms = {
                "fused": lambda i: blk(xs[i], cs[i]),
                "composition": lambda i: composition(blk, xs[i], cs[i]),
                "attn_fused": lambda i: attn.forward_adaln(n1[i], chunks[i][0], chunks[i][1], xs[i], chunks[i][2]),
                "attn_composition": lambda i: xs[i] + chunks[i][2].unsqueeze(1) * attn(
                    _modulate(n1[i], chunks[i][0], chunks[i][1])),
                "mlp_fused": lambda i: mlp.forward_adaln(n2[i], chunks[i][3], chunks[i][4], xs[i], chunks[i][5]),
                "mlp_composition": lambda i: xs[i] + chunks[i][5].unsqueeze(1) * mlp(
                    _modulate(n2[i], chunks[i][3], chunks[i][4])),
            }
            equal = {name: bool(torch.equal(arms[p + "fused"](0), arms[p + "composition"](0)))
                     for name, p in (("block", ""), ("attn", "attn_"), ("mlp", "mlp_"))}
            for a in ARMS:
                for _ in range(args.warmup):
                    for i in range(args.inputs):
                        arms[a](i)
            torch.cuda.synchronize()
            times = {a: [] for a in ARMS}
            for _ in range(args.rounds):
                for a in ARMS:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(args.steps):
                        for i in range(args.inputs):
                            arms[a](i)
                    e1.record()
                    torch.cuda.synchronize()
                    times[a].append(e0.elapsed_time(e1) / (args.steps * args.inputs))
            kus = {"fused": kernel_us(lambda: arms["fused"](0), 5),
                   "composition": kernel_us(lambda: arms["composition"](0), 5)}
        best = {a: min(times[a]) for a in ARMS}
        med = {a: sorted(times[a])[len(times[a]) // 2] for a in ARMS}
        by = traffic(B * T, C, 4 if dt == torch.float32 else 2)
        rec = dict(kind="result", case=cname, images=B, tokens=T, dim=C, heads=heads, top_k=top_k,
                   dtype=str(dt).replace("torch.", ""), bfloat=16, approximate="tanh", inputs=args.inputs,
                   steps=args.steps, rounds=args.rounds, ms_per_call=best, ms_per_call_median=med,
                   ms_per_call_all=times, fused_over_composition=best["fused"] / best["composition"],
                   attn_fused_over_composition=best["attn_fused"] / best["attn_composition"],
                   mlp_fused_over_composition=best["mlp_fused"] / best["mlp_composition"],
                   bytes_elementwise_by_algorithm=by, outputs_equal=all(equal.values()), outputs_equal_by_arm=equal,
                   kernel_us=kus)
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del blk, xs, cs, chunks, n1, n2, arms
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
