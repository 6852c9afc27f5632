#!/usr/bin/env python
"""DeiT block with its LayerNorms in the MX Linear operand quantizers and its residual adds in the output stores
(modules.QuantizedDeiTBlock) against the same modules run through timm's Block.forward composition (torch LayerNorm,
the attention and MLP shims, torch adds), and the output projection alone with each store.

Arms per case, run alternating in one process (round-robin over --rounds, each round timing --steps steps of every arm
after --warmup warm-up steps; best and median round reported):
  fused             QuantizedDeiTBlock(x)
  composition       x = x + attn(norm1(x)); x + mlp(norm2(x)) on the same modules (what a DeiT block ran before)
  proj_plain        proj(a)                                      the plain store
  proj_plain_add    x + proj(a)                                  the plain store and the torch add it replaces
  proj_add          proj.forward_adaln(a, add=x)                 the residual store
  proj_gated        proj.forward_adaln(a, residual=x, gate=g)    the gated residual store
Case: DeiT-base C2 blocks, 256 images x 197 tokens, C = 768, 12 heads, top-k 30, bfloat 16, with fp32 x and with bf16 x.
Every step runs on --inputs distinct x tensors in turn (155 MB each in fp32, 77 MB in bf16; with the attention input
a of the same size, each step's working set exceeds the 126 MB L2).  Device time from CUDA events around whole steps, per
call.  outputs_equal says whether the fused and the composition outputs are bit-identical (they must be).  After the
timing, one torch.profiler pass per arm gives the device time of each kernel (kernel_us): the row statistics
(k_layer_norm), the quantizers, and k_mx_linear_umma<dt, EPI> with EPI 0 (plain store), 3 (gated residual) or 4
(residual add).  bytes_removed_by_algorithm: the DRAM bytes (from shapes, not measured) the two torch norms and the two
torch adds move per block (each norm reads x and writes y, each add reads two tensors and writes one) minus the
statistics kernel's read of x.
Writes a JSONL file (default profiles/deit_block_b200.jsonl) whose first line records the GPU's name and power limit
from a read-only nvidia-smi query.
    python tools/bench_deit_block.py [--steps 5] [--rounds 5] [--out profiles/deit_block_b200.jsonl]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from bench import mx_specs  # noqa: E402
from mx_quantization_b200.modules import QuantizedAttention, QuantizedDeiTBlock, QuantizedMlp  # noqa: E402
from tools.bench_half_module import gpu_info, kernel_us  # noqa: E402

ARMS = ("fused", "composition", "proj_plain", "proj_plain_add", "proj_add", "proj_gated")
CASES = {  # images, tokens, C, heads, top_k, dtype
    "deit_base_c2_fp32": (256, 197, 768, 12, 30, torch.float32),
    "deit_base_c2_bf16": (256, 197, 768, 12, 30, torch.bfloat16),
}


class _Attn(nn.Module):                 # the attributes QuantizedAttention takes from timm's Attention
    def __init__(self, dim, heads):
        super().__init__()
        self.num_heads, self.scale = heads, (dim // heads) ** -0.5
        self.qkv, self.proj, self.proj_drop = nn.Linear(dim, 3 * dim), nn.Linear(dim, dim), nn.Dropout(0.0)


class _Mlp(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, 4 * dim), nn.GELU(), nn.Linear(4 * dim, dim), nn.Dropout(0.0)


class _Block(nn.Module):                # timm 0.4.12 vision_transformer.Block, drop_path 0
    def __init__(self, C, heads, top_k, sp):
        super().__init__()
        self.norm1 = nn.LayerNorm(C, eps=1e-6)
        self.attn = QuantizedAttention(_Attn(C, heads), mx_quant=True, mx_specs=sp, top_k=True, k=top_k)
        self.drop_path = nn.Identity()
        self.norm2 = nn.LayerNorm(C, eps=1e-6)
        self.mlp = QuantizedMlp(_Mlp(C), mx_specs=sp)

    def forward(self, x):
        x = x + self.drop_path(self.attn(self.norm1(x)))
        return x + self.drop_path(self.mlp(self.norm2(x)))


def traffic(M, C, es):
    t = M * C * es
    return dict(torch_norms_and_adds=2 * 2 * t + 2 * 3 * t, statistics=2 * t, removed=2 * 2 * t + 2 * 3 * t - 2 * t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--inputs", type=int, default=2)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deit_block_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_deit_block needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for cname in args.cases.split(","):
        B, T, C, heads, top_k, dt = CASES[cname]
        sp = mx_specs(16, False)
        torch.manual_seed(0)
        src = _Block(C, heads, top_k, sp).to(dev).to(dt).eval()
        with torch.no_grad():
            for n in (src.norm1, src.norm2):
                n.weight.normal_(1, 0.2)
                n.bias.normal_(0, 0.2)
        blk = QuantizedDeiTBlock(src)
        g = torch.Generator(device=dev).manual_seed(1)
        xs = [torch.randn(B, T, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        acts = [torch.randn(B, T, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        gate = torch.randn(B, C, device=dev, generator=g).to(dt)
        proj = src.attn.proj
        with torch.no_grad():
            arms = {
                "fused": lambda i: blk(xs[i]),
                "composition": lambda i: src(xs[i]),
                "proj_plain": lambda i: proj(acts[i]),
                "proj_plain_add": lambda i: xs[i] + proj(acts[i]),
                "proj_add": lambda i: proj.forward_adaln(acts[i], add=xs[i]),
                "proj_gated": lambda i: proj.forward_adaln(acts[i], residual=xs[i], gate=gate),
            }
            equal = dict(block=bool(torch.equal(arms["fused"](0), arms["composition"](0))),
                         proj_add=bool(torch.equal(arms["proj_add"](0), arms["proj_plain_add"](0))))
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
            kus = {a: kernel_us(lambda _a=a: arms[_a](0), 5) for a in ARMS}
        best = {a: min(times[a]) for a in ARMS}
        med = {a: sorted(times[a])[len(times[a]) // 2] for a in ARMS}
        rec = dict(kind="result", case=cname, images=B, tokens=T, dim=C, heads=heads, top_k=top_k,
                   dtype=str(dt).replace("torch.", ""), bfloat=16, inputs=args.inputs, steps=args.steps,
                   rounds=args.rounds, ms_per_call=best, ms_per_call_median=med, ms_per_call_all=times,
                   fused_over_composition=best["fused"] / best["composition"],
                   proj_add_over_plain_add=best["proj_add"] / best["proj_plain_add"],
                   bytes_removed_by_algorithm=traffic(B * T, C, 4 if dt == torch.float32 else 2),
                   outputs_equal=all(equal.values()), outputs_equal_by_arm=equal, kernel_us=kus)
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del blk, src, xs, acts, arms
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
