#!/usr/bin/env python
"""bench.py - pruned-attention throughput of the MXINT8 exponent-sign hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (q,k,v -> out) over the workload's layers, each layer with
its own synthetic q/k/v already resident in HBM (independent tensors per layer, far larger than
L2, so no L2 flush is needed between iterations).  Prints ONE JSON line (rank 0).

Default workload = BASELINE.json configs[1]: DeiT-base attention, batch 256 x 197 tokens,
12 heads, head_dim 64, all 12 layers, k = 30 (workloads/deit/scripts/run_deit.sh:51).
Multi-GPU (one process per GPU, torchrun): independent (batch, head) units, no data-path collective.
  --scaling weak (default)  every rank runs its own full batch (seed per rank); value = all ranks' heads / max time
  --scaling strong          ONE global batch (same seed everywhere) cut into contiguous batch slices
                            (mx_quantization_b200.sharding); after the timed region the ranks all_gather per-entry
                            digests of masks and outputs and rank 0 compares them with its own single-GPU run of
                            the whole batch ("verification" in the JSON line)
NCCL is used for the barrier, the max-over-ranks time and that verification gather only.
roofline: the dominant kernel of the default call (the fused launch where it applies: algorithmic bytes 16 N hd
per head, SURVEY 8(d)) + full_path_frac of the whole step + the per-kernel view of the three-kernel path.
--dump-outputs DIR: after the timed steps, DIR/out.npy holds what the last timed step returned (rank 0), so that two
builds run with the same arguments can be compared output for output (see dump_outputs).  For that, the last timed
step writes every layer into an output buffer of its own: one extra (B,N,H,hd) fp32 tensor per layer on rank 0.
--steps sets the step count of every GPU timing (main loop, per-kernel view, e2e, other workloads); cpu_baseline runs
on a time budget (cpu_port_heads_per_s).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: B, H, N, hd, top_k, layers, bfloat, flush     (SURVEY.md section 8 config shapes)
    "deit_base_c2": dict(B=256, H=12, N=197, hd=64, top_k=30, layers=12, bfloat=32, flush=False),
    "dit_xl2_c3": dict(B=256, H=16, N=256, hd=72, top_k=154, layers=28, bfloat=16, flush=False),
    "pixart_c4": dict(B=256, H=16, N=256, hd=72, top_k=77, layers=28, bfloat=32, flush=True),
    "deit_tiny_c1": dict(B=8, H=3, N=197, hd=64, top_k=80, layers=1, bfloat=32, flush=False),
}
# device-timed only, as an `other_workloads` entry of the default line (the long-sequence kernels; tools/sweep_c5.py has the sweep)
LONG_WORKLOADS = {
    "dit_long_c5": dict(B=16, H=16, N=4096, hd=72, top_k=1024, layers=1, bfloat=32, flush=False),   # BASELINE.json configs[4], N = 4096
}
CPU_SAMPLE_B = 8          # cpu_baseline / reference arm: a B=8 slice of one layer (BASELINE.md 4)
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs writes at most this many bytes


def mx_specs(bfloat, flush):
    return {
        'w_elem_format': 'int8', 'a_elem_format': 'int8', 'scale_bits': 8, 'shared_exp_method': 'max',
        'block_size': 32, 'bfloat': bfloat, 'fp': 0, 'bfloat_subnorms': True, 'round': 'nearest',
        'round_mx_output': 'nearest', 'round_output': 'nearest', 'round_weight': 'nearest',
        'mx_flush_fp32_subnorms': flush, 'custom_cuda': False, 'quantize_backprop': False,
    }


def bytes_per_head(N, hd):
    """ALGORITHMIC bytes per (batch, head) unit (SURVEY.md 8d, DESIGN.md 'Measurement')."""
    nb, nw = (hd + 31) // 32, (N + 31) // 32
    hdp = (hd + 15) // 16 * 16
    pred = 2 * N * hd * 4 + N * nw * 4                       # Q,K fp32 in ; bitmask out
    prep = N * hd * 4 + N * hdp * 2                          # V fp32 in ; bf16 V^T operand out
    attn = 3 * N * hdp * 2 + N * nw * 4 + N * hd * 4         # bf16 Q,K,V operands + mask in ; O fp32 out
    full = 16 * N * hd                                       # Q,K,V in ; O out
    return {"predict_topk": pred, "prep_v": prep, "exact_attention": attn, "full": full}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(path, outs):
    """Write the fp32 (B,H,N,hd) outputs ``outs`` of one step (one per layer) to path/out.npy, float32
    (layers, rows, hd), a row being one (batch, head, query) entry in that order.  When every row of every layer would
    exceed DUMP_BYTES, each layer contributes the same rows: the first `keep` of torch.randperm(B*H*N) under a CPU
    generator seeded with 0, ascending - fixed for a workload, so the files of two builds line up.  Returns the bytes."""
    import numpy as np
    import torch
    B, H, N, hd = outs[0].shape
    rows = B * H * N
    keep = min(rows, (DUMP_BYTES - 4096) // (4 * hd * len(outs)))      # 4096: room for the .npy header
    sel = None
    if keep < rows:
        sel = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    arr = np.empty((len(outs), keep, hd), dtype=np.float32)
    for i, o in enumerate(outs):
        flat = o.reshape(rows, hd)
        arr[i] = (flat if sel is None else flat[sel.to(flat.device)]).cpu().numpy()
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "out.npy"), arr)
    return arr.nbytes


def cpu_port_heads_per_s(w, budget_s=12.0, threads=None):
    """The oracle port of the reference's CPU path (torch.topk left in place, as the reference
    does), all host threads, on a B=CPU_SAMPLE_B slice of one layer."""
    import torch
    from oracle import mxint8_oracle as O
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    B = min(CPU_SAMPLE_B, w["B"])
    g = torch.Generator().manual_seed(0)
    q, k, v = (torch.randn(B, w["H"], w["N"], w["hd"], generator=g) for _ in range(3))

    def run():
        O.pruned_attention(q, k, v, w["top_k"], bfloat=w["bfloat"], flush=w["flush"], use_torch_topk=True)

    run()                                           # warm-up
    times, t_end = [], time.perf_counter() + budget_s
    while len(times) < 3 or (time.perf_counter() < t_end and len(times) < 50):
        t0 = time.perf_counter(); run(); times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return B * w["H"] / med, threads, f"B={B} slice of one layer ({B * w['H']} heads), median of {len(times)} reps"


def config_dict(name, w, gpus, scaling="weak"):
    if scaling == "strong":
        par = (f"one global batch of {w['B']} split into contiguous batch slices over {gpus} GPU(s) "
               "(mx_quantization_b200.sharding.take_shard), no data-path collective; digests all_gathered for verification")
    else:
        par = (f"{gpus} GPU(s), each running its own full batch of {w['B']} (weak scaling: independent (batch, head) "
               "units, no data-path collective)")
    return {"workload": name, "batch": w["B"], "heads": w["H"], "tokens": w["N"], "head_dim": w["hd"],
            "top_k": w["top_k"], "layers": w["layers"], "mx_specs": f"int8/block32/bfloat{w['bfloat']}"
            + ("/flush" if w["flush"] else ""), "parallelism": par,
            "l2": "inputs (one q/k/v set per layer) exceed L2; no flush needed"}


def run_reference(args, name, w):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the
    Python reference itself cannot travel to the GPU box), host cores only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import mxint8_oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    B = min(CPU_SAMPLE_B, w["B"])
    g = torch.Generator().manual_seed(0)
    q, k, v = (torch.randn(B, w["H"], w["N"], w["hd"], generator=g) for _ in range(3))

    def step():
        return O.pruned_attention(q, k, v, w["top_k"], bfloat=w["bfloat"], flush=w["flush"], use_torch_topk=True)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [res["out"]])
    heads = B * w["H"]
    val = heads / dt
    sample = f"each step = B={B} slice of one layer ({heads} heads) of {name}"
    print(json.dumps({
        "impl": "reference", "metric": "pruned-attention heads/s", "value": val, "unit": "heads/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
        "config": config_dict(name, w, args.gpus), "tokens_per_s": B * w["N"] / dt,
        "cpu_baseline": {"value": val, "unit": "heads/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "heads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def make_layers(torch, w, dev, seed, batch_slice=None):
    """One fused qkv buffer per layer; q/k/v are the permuted views the attention modules produce
    (workloads/deit/scripts/main.py:87-88).  batch_slice = (lo, hi): keep only that slice of the (seeded) global batch."""
    B, H, N, hd, L = w["B"], w["H"], w["N"], w["hd"], w["layers"]
    g = torch.Generator(device=dev).manual_seed(seed)
    layers = []
    for _ in range(L):
        buf = torch.randn(B, N, 3, H, hd, device=dev, generator=g)
        if batch_slice is not None:
            buf = buf[batch_slice[0]:batch_slice[1]].clone()
        qkv = buf.permute(2, 0, 3, 1, 4)
        layers.append((qkv[0], qkv[1], qkv[2]))
    return layers


def time_steps(torch, step, steps, barrier, last_outs=None):
    """Mean ms per step over `steps` steps.  last_outs: output buffers the last step writes in place of the step's own
    (the same work; what --dump-outputs saves)."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(steps):
        if last_outs is not None and i == steps - 1:
            step(last_outs)
        else:
            step()
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1) / steps


def kernel_breakdown(torch, mxq, layers, specs, top_k, out_view, reps):
    """Per-kernel CUDA-event times of one call (mxp_pruned_attention_profile), averaged over layers x reps.
    Default policy first (one fused launch where it applies), then the three-kernel path for the per-stage view."""
    res = {}
    for label, mode in (("default", 1), ("three_kernels", 0)):
        acc, n = [0.0, 0.0, 0.0], 0
        mxq.set_fused_path(mode)
        try:
            for it in range(1 + reps):                          # first pass untimed
                for (q, k, v) in layers:
                    ms3 = []
                    mxq.pruned_attention(q, k, v, specs, top_k, out=out_view, _kernel_ms=ms3)
                    if it:
                        acc = [a + m for a, m in zip(acc, ms3)]
                        n += 1
            res[label] = ([a / n for a in acc], mxq.last_launch_count())
        finally:
            mxq.set_fused_path(1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of every GPU timing (cpu_baseline runs on a time budget of its own)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="deit_base_c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank runs the full batch; strong: one global batch partitioned over the ranks, verified")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the device-timed lines of the other workload shapes")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/out.npy (float32; a fixed sample when over 64 MB); "
                         "holds one extra output buffer per layer on the GPU for the whole run (deit_base_c2: 1.9 GB, "
                         "dit_xl2_c3 / pixart_c4: 8.5 GB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    name, w = args.workload, WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, name, w)
        return

    import torch
    import torch.distributed as dist
    import mx_quantization_b200 as mxq
    from mx_quantization_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    specs = mx_specs(w["bfloat"], w["flush"])
    B, H, N, hd, L, top_k = w["B"], w["H"], w["N"], w["hd"], w["layers"], w["top_k"]
    strong = args.scaling == "strong"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs.  weak: every rank its own full batch (seed per rank).  strong: ONE global batch (same seed on every
    # rank), each rank keeps its contiguous batch slice (sharding.shard_batch_heads / take_shard)
    if strong:
        kind, lo, hi = sharding.shard_batch_heads(B, H, world, rank)
        if kind != "batch":
            raise SystemExit("bench.py --scaling strong: batch < ranks is not a bench configuration")
        layers = make_layers(torch, w, dev, 1234, (lo, hi))
        Bl = hi - lo
    else:
        layers = make_layers(torch, w, dev, 1000 * rank)
        Bl = B
    heads_per_step_total = (B if strong else world * B) * H * L
    out = torch.empty(Bl, N, H, hd, device=dev)     # (B,N,H,hd): the module's transpose(1,2) is free
    out_view = out.permute(0, 2, 1, 3)
    # --dump-outputs: the last timed step writes each layer's output into a buffer of its own, laid out like `out`
    dump = None
    if args.dump_outputs and rank == 0:
        dump = [torch.empty(Bl, N, H, hd, device=dev).permute(0, 2, 1, 3) for _ in range(L)]

    def step(outs=None):
        for li, (q, k, v) in enumerate(layers):
            mxq.pruned_attention(q, k, v, specs, top_k, out=out_view if outs is None else outs[li])

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    W = max(args.warmup, 3)
    for _ in range(W):
        step()
    launches_per_call = mxq.last_launch_count()
    ms_per_step = time_steps(torch, step, args.steps, barrier, dump)
    kb = kernel_breakdown(torch, mxq, layers, specs, top_k, out_view, args.steps) if rank == 0 or world > 1 else None
    if rank == 0:
        # the timed region (a few tens of ms) can be shorter than one nvidia-smi period: keep the SAME
        # step loop running, untimed, until a few samples have been taken under that load
        t_end = time.perf_counter() + 3.0
        while len(sampler.lines) < 4 and time.perf_counter() < t_end:
            step()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["note"] = ("sampled from warm-up to the end of an untimed continuation of the same step loop "
                          "(nvidia-smi period 50 ms; the timed region alone can be shorter than one period)")
    if world > 1:
        t = torch.tensor([ms_per_step], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step = float(t.item())
    value = heads_per_step_total / (ms_per_step * 1e-3)
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
        del dump

    # ---- strong scaling: cross-rank verification, outside every timed region.  Each rank digests the masks and the
    # outputs of its slice of layer 0; the digests are all_gathered (NCCL over NVLink) and rank 0 compares them with
    # its own single-GPU run of the WHOLE global batch
    verification = None
    if strong:
        q, k, v = layers[0]
        o_s, m_s = mxq.pruned_attention(q, k, v, specs, top_k, return_mask=True)
        dig = torch.stack([m_s.to(torch.int64).reshape(Bl, -1).sum(1).double(),
                           o_s.double().reshape(Bl, -1).sum(1), o_s.double().abs().reshape(Bl, -1).sum(1)], 1)
        parts = sharding.gather_for_verification(dig, world)
        if rank == 0:
            full = make_layers(torch, dict(w, layers=1), dev, 1234)[0]
            o_f, m_f = mxq.pruned_attention(full[0], full[1], full[2], specs, top_k, return_mask=True)
            ref = torch.stack([m_f.to(torch.int64).reshape(B, -1).sum(1).double(),
                               o_f.double().reshape(B, -1).sum(1), o_f.double().abs().reshape(B, -1).sum(1)], 1)
            got = torch.cat(parts, 0)
            verification = {"what": "per-batch-entry digests (mask word sums, output sums) of layer 0: all_gather of the "
                                    f"{world} shards vs rank 0's single-GPU run of the whole batch",
                            "batch_entries": int(got.shape[0]), "masks_equal": bool(torch.equal(got[:, 0], ref[:, 0])),
                            "outputs_equal": bool(torch.equal(got[:, 1:], ref[:, 1:]))}
            del full, o_f, m_f
        del o_s, m_s

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timing
    e2e = None
    if not args.no_e2e:
        e2e_layers = L
        try:
            host_in = [torch.empty(Bl, N, 3, H, hd).pin_memory() for _ in range(e2e_layers)]
            host_out = [torch.empty(Bl, N, H, hd).pin_memory() for _ in range(e2e_layers)]
        except RuntimeError:                        # pinned-memory limit of the box: fall back to a third of the layers
            e2e_layers = max(1, L // 3)
            host_in = [torch.empty(Bl, N, 3, H, hd).pin_memory() for _ in range(e2e_layers)]
            host_out = [torch.empty(Bl, N, H, hd).pin_memory() for _ in range(e2e_layers)]
        for hbuf in host_in:
            hbuf.normal_()
        NBUF = 3                                    # device staging buffers: keeps the H2D engine busy back to back
        dev_in = [torch.empty(Bl, N, 3, H, hd, device=dev) for _ in range(NBUF)]
        dev_out = [torch.empty(Bl, N, H, hd, device=dev) for _ in range(NBUF)]
        s_in, s_out, s_cmp = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()
        ev_in = [torch.cuda.Event() for _ in range(NBUF)]
        ev_cmp = [torch.cuda.Event() for _ in range(NBUF)]
        ev_free = [torch.cuda.Event() for _ in range(NBUF)]
        ev_out = [torch.cuda.Event() for _ in range(NBUF)]

        def e2e_step():
            for li in range(e2e_layers):
                s = li % NBUF
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_free[s])                       # compute finished with dev_in[s]
                    dev_in[s].copy_(host_in[li], non_blocking=True)
                    ev_in[s].record(s_in)
                s_cmp.wait_event(ev_in[s])
                s_cmp.wait_event(ev_out[s])                           # previous D2H of dev_out[s] done
                qkv = dev_in[s].permute(2, 0, 3, 1, 4)
                mxq.pruned_attention(qkv[0], qkv[1], qkv[2], specs, top_k, out=dev_out[s].permute(0, 2, 1, 3))
                ev_cmp[s].record(s_cmp)
                ev_free[s].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[s])
                    host_out[li].copy_(dev_out[s], non_blocking=True)
                    ev_out[s].record(s_out)
            s_cmp.wait_stream(s_out)

        e2e_step()
        ems = time_steps(torch, e2e_step, args.steps, barrier)
        if world > 1:
            t = torch.tensor([ems], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        scale_l = L / e2e_layers                    # bytes/heads reported for the full L-layer step
        h2d, d2h = host_in[0].numel() * 4 * e2e_layers, host_out[0].numel() * 4 * e2e_layers
        e2e = {"value": (B if strong else world * B) * H * e2e_layers / (ems * 1e-3), "unit": "heads/s",
               "h2d_bytes_per_step": int(h2d * scale_l), "d2h_bytes_per_step": int(d2h * scale_l),
               "ms_per_step": ems * scale_l, "h2d_gbs_per_rank": h2d / (ems * 1e-3) / 1e9,
               "note": f"timed on {e2e_layers} of {L} layers per step, every layer from its own pinned host buffer "
                       "(H2D / compute / D2H triple-buffered on 3 streams); bytes are per rank"}
        del host_in, host_out, dev_in, dev_out

    # ---- the other workload shapes, device-timed only (their own lines: --workload NAME)
    others = None
    if rank == 0 and world == 1 and not args.no_others and name == "deit_base_c2":
        others = {}
        del layers
        torch.cuda.empty_cache()
        for oname in ("dit_xl2_c3", "pixart_c4", "dit_long_c5"):
            ow = WORKLOADS.get(oname) or LONG_WORKLOADS[oname]
            ol = make_layers(torch, ow, dev, 7)
            oo = torch.empty(ow["B"], ow["N"], ow["H"], ow["hd"], device=dev).permute(0, 2, 1, 3)
            osp = mx_specs(ow["bfloat"], ow["flush"])

            def ostep():
                for (q, k, v) in ol:
                    mxq.pruned_attention(q, k, v, osp, ow["top_k"], out=oo)

            for _ in range(3):
                ostep()
            oms = time_steps(torch, ostep, args.steps, barrier)
            oh = ow["B"] * ow["H"] * ow["layers"]
            ob = bytes_per_head(ow["N"], ow["hd"])
            peak, _ = hbm_peak()
            others[oname] = {"value": oh / (oms * 1e-3), "unit": "heads/s", "ms_per_step": oms,
                             "full_path_gbs": ob["full"] * oh / (oms * 1e-3) / 1e9,
                             "full_path_frac": ob["full"] * oh / (oms * 1e-3) / 1e9 / peak,
                             "config": {k: ow[k] for k in ("B", "H", "N", "hd", "top_k", "layers", "bfloat", "flush")}}
            del ol, oo
            torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = hbm_peak()
        bph = bytes_per_head(N, hd)
        heads_call = Bl * H                                     # heads one launch processes on this rank
        (dms, dlaunch), (tms, tlaunch) = kb["default"], kb["three_kernels"]
        full_gbs = bph["full"] * (heads_per_step_total / world) / (ms_per_step * 1e-3) / 1e9     # per GPU
        kernels = {}
        for kname, avg_ms in zip(("predict_topk", "prep_v", "exact_attention"), tms):
            ach = bph[kname] * heads_call / (avg_ms * 1e-3) / 1e9
            kernels[kname] = {"avg_ms": avg_ms, "achieved_gbs": ach, "frac": ach / peak, "bytes_per_launch": bph[kname] * heads_call}
        fused = dlaunch == 1
        tj = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(name, {})
        if fused:
            # the dominant (only) kernel of the default path: k_fused_pruned_attention, q,k,v -> out in one launch;
            # algorithmic bytes = SURVEY 8(d)'s full-path figure 16 N hd per head
            ach = bph["full"] * heads_call / (dms[0] * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": "k_fused_pruned_attention", "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": ach / peak, "traffic": tj.get("fused"), "bytes_per_launch": bph["full"] * heads_call,
                        "avg_ms": dms[0]}
        else:
            # three launches per call: SURVEY 8(d)'s metric kernel is the fused predictor + top-k (8 N hd + 4 N ceil(N/32))
            roofline = {"bound": "hbm", "kernel": "predict_topk", "achieved": kernels["predict_topk"]["achieved_gbs"],
                        "peak": peak, "unit": "GB/s", "frac": kernels["predict_topk"]["frac"], "traffic": tj.get("predict_topk"),
                        "bytes_per_launch": kernels["predict_topk"]["bytes_per_launch"], "avg_ms": tms[0]}
        # SURVEY 8(d): both denominators - the measured copy bandwidth (peak, above) and the north star's nominal ~8 TB/s
        NOMINAL_GBS = 8000.0
        for kv in kernels.values():
            kv["frac_of_nominal_8tbs"] = kv["achieved_gbs"] / NOMINAL_GBS
        roofline.update({"frac_of_nominal_8tbs": roofline["achieved"] / NOMINAL_GBS,
                         "full_path_frac_of_nominal_8tbs": full_gbs / NOMINAL_GBS})
        roofline.update({"peak_source": peak_src, "full_path_gbs": full_gbs, "full_path_frac": full_gbs / peak,
                         "three_kernel_path": {"note": "the same call with mxp_set_fused_path(0): per-kernel CUDA-event times "
                                                       "against each kernel's bytes (predict_topk: SURVEY 8(d)'s 8 N hd + 4 N ceil(N/32); "
                                                       "prep_v / exact_attention: the bytes those kernels move, operands included)",
                                               "kernels": kernels, "ms_per_layer": sum(tms)},
                         "launches_per_call": dlaunch})
        line = {
            "metric": "pruned-attention heads/s", "value": value, "unit": "heads/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int8",
            "data": "synthetic", "config": config_dict(name, w, world, args.scaling),
            "tokens_per_s": value / H * N,
            "roofline": roofline, "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches_per_call * L * args.steps,
        }
        if verification is not None:
            line["verification"] = verification
        if others:
            line["other_workloads"] = others
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_port_heads_per_s(w)
            line["cpu_baseline"] = {"value": v, "unit": "heads/s", "cores": cores, "kind": "port", "sample": sample}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
