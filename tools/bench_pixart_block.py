#!/usr/bin/env python
"""PixArt-alpha adaLN-single block in the MX kernels (modules.QuantizedPixArtBlock: q, k and v from one GEMM whose
quantizer applies the modulation, to_out / fc2 stores that apply the gated residuals) against the same modules run
through BasicTransformerBlock.forward's torch composition, and each adaLN half alone.

Arms per case, run alternating in one process (round-robin over --rounds, each round timing --steps steps of every arm
after --warmup warm-up steps; best and median round reported):
  fused             QuantizedPixArtBlock(h, encoder_hidden_states, encoder_attention_mask, timestep)
  composition       the same modules: LayerNorm, torch modulate, MXSelfAttention.forward (three projections), torch gated
                    residual, MXCrossAttention + add, LayerNorm, modulate, QuantizedMlp (the fused mx_mlp), gated residual
  attn_fused / attn_composition   the self-attention half alone on a precomputed norm1(h) and adaLN chunks
  ff_fused / ff_composition       the feed-forward half alone on a precomputed norm2(h) and adaLN chunks
Cases: PixArt-alpha 256 x 256 blocks (C4): 256 images x 256 tokens, C = 1152, 16 heads of 72, top-k 77, S = 120 text
tokens with a mask, bfloat 32, flush, tanh GELU, with fp32 x and with fp16 x.  Every step runs on --inputs distinct
hidden-state tensors in turn (302 MB each in fp32, 151 MB in fp16: larger than the 126 MB L2).  Device time from CUDA
events around whole steps, per call.  outputs_equal says whether the fused and the composition outputs are bit-identical
(they must be).  After the timing, one torch.profiler pass per case gives the device time of each kernel of the fused
block and of the composition (kernel_us).  bytes_adaln_* are the DRAM bytes, by the algorithm from shapes (not measured),
of the (M, C) tensors the two adaLN halves touch outside the attention core and the MLP: per half, the composition's
modulate reads and writes two tensors, each operand quantizer reads the modulated x (three in the self-attention half,
one in the feed-forward), the output projection writes y and the gated residual reads y, writes gate * y, reads h and
gate * y and writes the sum; the fused half reads the normalized x and the residual and writes the sum.
Writes a JSONL file (default profiles/pixart_block_b200.jsonl) whose first line records the GPU's name and power limit
from a read-only nvidia-smi query.
    python tools/bench_pixart_block.py [--steps 5] [--rounds 5] [--out profiles/pixart_block_b200.jsonl]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from bench import mx_specs  # noqa: E402
from mx_quantization_b200.modules import MXCrossAttention, MXSelfAttention, QuantizedPixArtBlock  # noqa: E402
from tools.bench_half_module import gpu_info, kernel_us  # noqa: E402

ARMS = ("fused", "composition", "attn_fused", "attn_composition", "ff_fused", "ff_composition")
CASES = {  # images, tokens, C, heads, top_k, text tokens, dtype
    "pixart_c4_fp32": (256, 256, 1152, 16, 77, 120, torch.float32),
    "pixart_c4_fp16": (256, 256, 1152, 16, 77, 120, torch.float16),
}


class _GELU(nn.Module):
    """diffusers.models.activations.GELU (owns the feed-forward's fc1)."""

    def __init__(self, dim_in, dim_out, approximate):
        super().__init__()
        self.proj, self.approximate = nn.Linear(dim_in, dim_out), approximate

    def forward(self, x):
        return F.gelu(self.proj(x), approximate=self.approximate)


class _FeedForward(nn.Module):
    """diffusers.models.attention.FeedForward with activation_fn="gelu-approximate" (PixArt)."""

    def __init__(self, dim):
        super().__init__()
        self.net = nn.ModuleList([_GELU(dim, 4 * dim, "tanh"), nn.Dropout(0.0), nn.Linear(4 * dim, dim)])


class _PixArtBlock(nn.Module):
    """BasicTransformerBlock(norm_type="ada_norm_single", norm_elementwise_affine=False, norm_eps=1e-6) with the shims."""

    def __init__(self, C, heads, top_k, sp):
        super().__init__()
        cfg = dict(mx_quant=True, mx_specs=sp, top_k=True, k=top_k, ex_pred=True)
        self.norm1 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn1 = MXSelfAttention(C, heads).set_config(**cfg)
        self.norm2 = nn.LayerNorm(C, elementwise_affine=False, eps=1e-6)
        self.attn2 = MXCrossAttention(C, heads).set_config(**cfg)
        self.ff = _FeedForward(C)
        self.scale_shift_table = nn.Parameter(torch.randn(6, C) / C ** 0.5)


def _chunks(blk, t):
    return (blk.scale_shift_table[None] + t.reshape(t.shape[0], 6, -1)).chunk(6, dim=1)


def composition(blk, h, enc, mask, t):
    """BasicTransformerBlock.forward (ada_norm_single) on QuantizedPixArtBlock's modules."""
    shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp = _chunks(blk, t)
    h = gate_msa * blk.attn1(blk.norm1(h) * (1 + scale_msa) + shift_msa) + h
    h = blk.attn2(h, enc, attention_mask=mask) + h
    return gate_mlp * blk.ff(blk.norm2(h) * (1 + scale_mlp) + shift_mlp) + h


def traffic(M, C, es):
    """DRAM bytes of the (M, C) tensors the two adaLN halves touch, by the algorithm (es = bytes per element)."""
    t = M * C * es
    comp = (4 + 3 + 1 + 5) + (4 + 1 + 1 + 5)
    return dict(composition=comp * t, fused=2 * 3 * t, removed=(comp - 6) * t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--inputs", type=int, default=2)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pixart_block_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pixart_block needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for cname in args.cases.split(","):
        B, T, C, heads, top_k, S, dt = CASES[cname]
        sp = mx_specs(32, True)
        torch.manual_seed(0)
        blk = QuantizedPixArtBlock(_PixArtBlock(C, heads, top_k, sp), mx_specs=sp).to(dev).to(dt).eval()
        g = torch.Generator(device=dev).manual_seed(1)
        hs = [torch.randn(B, T, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        ts = [(0.5 * torch.randn(B, 6 * C, device=dev, generator=g)).to(dt) for _ in range(args.inputs)]
        encs = [torch.randn(B, S, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        # diffusers' additive text mask (1 - keep) * -10000, (B, 1, S): a prompt of 20-120 tokens per image
        lens = torch.randint(20, S + 1, (B,), device=dev, generator=g)
        mask = ((torch.arange(S, device=dev)[None] >= lens[:, None]).float() * -10000.0).unsqueeze(1)
        with torch.no_grad():
            chunks = [[c.squeeze(1) for c in _chunks(blk, t)] for t in ts]
            n1 = [blk.norm1(h) for h in hs]
            n2 = [blk.norm2(h) for h in hs]
            attn, ff = blk.attn1, blk.ff

            def mod(x, shift, scale):
                return x * (1 + scale.unsqueeze(1)) + shift.unsqueeze(1)

            arms = {
                "fused": lambda i: blk(hs[i], encoder_hidden_states=encs[i], encoder_attention_mask=mask,
                                       timestep=ts[i]),
                "composition": lambda i: composition(blk, hs[i], encs[i], mask, ts[i]),
                "attn_fused": lambda i: attn.forward_adaln(n1[i], chunks[i][0], chunks[i][1], hs[i], chunks[i][2]),
                "attn_composition": lambda i: chunks[i][2].unsqueeze(1) * attn(
                    mod(n1[i], chunks[i][0], chunks[i][1])) + hs[i],
                "ff_fused": lambda i: ff.forward_adaln(n2[i], chunks[i][3], chunks[i][4], hs[i], chunks[i][5]),
                "ff_composition": lambda i: chunks[i][5].unsqueeze(1) * ff(mod(n2[i], chunks[i][3], chunks[i][4])) + hs[i],
            }
            equal = {name: bool(torch.equal(arms[p + "fused"](0), arms[p + "composition"](0)))
                     for name, p in (("block", ""), ("attn", "attn_"), ("ff", "ff_"))}
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
        rec = dict(kind="result", case=cname, images=B, tokens=T, dim=C, heads=heads, top_k=top_k, text_tokens=S,
                   dtype=str(dt).replace("torch.", ""), bfloat=32, flush=True, approximate="tanh", inputs=args.inputs,
                   steps=args.steps, rounds=args.rounds, ms_per_call=best, ms_per_call_median=med,
                   ms_per_call_all=times, fused_over_composition=best["fused"] / best["composition"],
                   attn_fused_over_composition=best["attn_fused"] / best["attn_composition"],
                   ff_fused_over_composition=best["ff_fused"] / best["ff_composition"],
                   bytes_adaln_by_algorithm=traffic(B * T, C, 4 if dt == torch.float32 else 2),
                   outputs_equal=all(equal.values()), outputs_equal_by_arm=equal, kernel_us=kus)
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del blk, hs, ts, encs, chunks, n1, n2, arms
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
