#!/usr/bin/env python
"""Fused MX MLP (ops.mx_mlp: fc1's epilogue applies the GELU and writes fc2's MXINT8 operand) against the composition
mx_linear -> torch GELU -> mx_linear it replaces, and against each of the composition's three passes alone.

Arms per case, run alternating in one process (round-robin over --rounds, each round timing --steps steps of every arm
after --warmup warm-up steps; best and median round reported):
  fused        ops.mx_mlp on prepared weight operands
  composition  ops.mx_linear(fc1) -> F.gelu -> ops.mx_linear(fc2)   (what QuantizedMlp ran before)
  fc1          ops.mx_linear(fc1) alone (writes the hidden activation in x's dtype)
  gelu         F.gelu on that hidden activation alone
  fc2          ops.mx_linear(fc2) alone on the GELU output (includes fc2's quantizer pass)
  module_fused / module_composition   the whole QuantizedMlp with nn.GELU (fused path) and with a GELU subclass (which
                                       keeps the composition), same weights
Cases:
  deit_base_fp32   DeiT-base MLP, 256 x 197 tokens, 768 -> 3072 -> 768, fp32 x, GELU (erf), bfloat 32
  deit_base_bf16   the same with bf16 x
  dit_xl2_tanh     DiT-XL/2 MLP, 256 x 256 tokens, 1152 -> 4608 -> 1152, fp32 x, tanh GELU, bfloat 16
Every step runs on --inputs distinct x tensors in turn (at least 155 MB each in fp32 / 78 MB in bf16; with the hidden
activation every arm's working set exceeds the 126 MB L2).  Device time from CUDA events around whole steps, per call.
outputs_equal says whether fused and composition outputs are bit-identical (they must be).  After the timing, one
torch.profiler pass per case gives the device time of each kernel of the fused call and of the composition (kernel_us).
bytes_* are the DRAM bytes each arm needs by the algorithm, computed from shapes (not measured).
Writes a JSONL file (default profiles/mlp_b200.jsonl) whose first line records the GPU's name and power limit from a
read-only nvidia-smi query.
    python tools/bench_mlp.py [--steps 10] [--rounds 5] [--out profiles/mlp_b200.jsonl]"""
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
from mx_quantization_b200 import ops  # noqa: E402
from mx_quantization_b200.modules import QuantizedMlp  # noqa: E402
from tools.bench_half_module import gpu_info, kernel_us  # noqa: E402

ARMS = ("fused", "composition", "fc1", "gelu", "fc2", "module_fused", "module_composition")
CASES = {  # tokens, C, hidden, dtype, approximate, bfloat
    "deit_base_fp32": (256 * 197, 768, 3072, torch.float32, "none", 32),
    "deit_base_bf16": (256 * 197, 768, 3072, torch.bfloat16, "none", 32),
    "dit_xl2_tanh": (256 * 256, 1152, 4608, torch.float32, "tanh", 16),
}


class _GeluComposition(nn.GELU):
    """nn.GELU under another type: QuantizedMlp runs the layer-by-layer composition for it."""


class _Mlp(nn.Module):
    def __init__(self, dim, hidden, act):
        super().__init__()
        self.fc1, self.act, self.fc2, self.drop = nn.Linear(dim, hidden), act, nn.Linear(hidden, dim), nn.Dropout(0.0)


def traffic(M, C, H, es):
    """DRAM bytes by the algorithm (weights and biases excluded: small and L2-resident).  es = bytes per x element."""
    hid, op, xin, out = M * H * es, M * H * 2, M * C * es, M * C * es
    x_op = M * C * 2
    q_x = xin + x_op                         # x -> x's bf16 operand
    fc1 = x_op + hid                         # read x's operand, write the hidden activation
    gelu = 2 * hid
    fc2 = (hid + op) + (op + out)            # fc2's quantizer, then its GEMM
    fused = q_x + x_op + op + op + out       # quantizer, fc1 writes fc2's operand, fc2 reads it
    return dict(fused=fused, composition=q_x + fc1 + gelu + fc2, fc1=q_x + fc1, gelu=gelu, fc2=fc2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--inputs", type=int, default=2)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mlp_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mlp needs a CUDA device: there is no CPU measurement")
    dev = torch.device("cuda:0")
    lines = [dict(kind="device", **gpu_info())]
    print(json.dumps(lines[0]), flush=True)
    for cname in args.cases.split(","):
        M, C, H, dt, approx, bfloat = CASES[cname]
        sp = mx_specs(bfloat, False)
        act = "gelu_tanh" if approx == "tanh" else "gelu"
        torch.manual_seed(0)
        base = _Mlp(C, H, nn.GELU(approx))
        mod_f = QuantizedMlp(base, mx_specs=sp).to(dev).eval()
        mod_c = QuantizedMlp(_Mlp(C, H, _GeluComposition(approx)), mx_specs=sp).to(dev).eval()
        mod_c.fc1, mod_c.fc2 = mod_f.fc1, mod_f.fc2                  # same weights and cached operands
        g = torch.Generator(device=dev).manual_seed(1)
        xs = [torch.randn(M, C, device=dev, generator=g).to(dt) for _ in range(args.inputs)]
        with torch.no_grad():
            w1, w2 = mod_f.fc1._operand(), mod_f.fc2._operand()
            b1, b2 = mod_f.fc1.bias.detach(), mod_f.fc2.bias.detach()
            hs = [ops.mx_linear(x, w1, b1, sp, out_features=H) for x in xs]
            gs = [F.gelu(h, approximate=approx) for h in hs]
            arms = {
                "fused": lambda i: ops.mx_mlp(xs[i], w1, b1, w2, b2, sp, act=act, hidden_features=H, out_features=C),
                "composition": lambda i: ops.mx_linear(F.gelu(ops.mx_linear(xs[i], w1, b1, sp, out_features=H),
                                                              approximate=approx), w2, b2, sp, out_features=C),
                "fc1": lambda i: ops.mx_linear(xs[i], w1, b1, sp, out_features=H),
                "gelu": lambda i: F.gelu(hs[i], approximate=approx),
                "fc2": lambda i: ops.mx_linear(gs[i], w2, b2, sp, out_features=C),
                "module_fused": lambda i: mod_f(xs[i]),
                "module_composition": lambda i: mod_c(xs[i]),
            }
            outs = {a: arms[a](0) for a in ("fused", "composition", "module_fused", "module_composition")}
            equal = bool(torch.equal(outs["fused"], outs["composition"]))
            equal_mod = bool(torch.equal(outs["module_fused"], outs["module_composition"]))
            del outs
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
            kus = {"fused": kernel_us(lambda: arms["fused"](0), 10),
                   "composition": kernel_us(lambda: arms["composition"](0), 10)}
        best = {a: min(times[a]) for a in ARMS}
        med = {a: sorted(times[a])[len(times[a]) // 2] for a in ARMS}
        by = traffic(M, C, H, 4 if dt == torch.float32 else 2)
        rec = dict(kind="result", case=cname, tokens=M, dims=[C, H, C], dtype=str(dt).replace("torch.", ""),
                   approximate=approx, bfloat=bfloat, inputs=args.inputs, steps=args.steps, rounds=args.rounds,
                   ms_per_call=best, ms_per_call_median=med, ms_per_call_all=times,
                   fused_over_composition=best["fused"] / best["composition"],
                   module_fused_over_composition=best["module_fused"] / best["module_composition"],
                   passes_sum_ms=best["fc1"] + best["gelu"] + best["fc2"],
                   bytes_by_algorithm=by, gb_per_s_by_algorithm={a: by[a] / (best[a] * 1e-3) / 1e9 for a in by},
                   outputs_equal=equal, module_outputs_equal=equal_mod, kernel_us=kus)
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del mod_f, mod_c, xs, hs, gs, arms
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
