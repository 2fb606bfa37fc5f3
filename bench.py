#!/usr/bin/env python
"""bench.py — clips/sec of the InternVideo2 stage-1 masked-video pre-training step (BASELINE.json cfg-2).

  python bench.py --gpus N --steps K --warmup W            # ivb200 arm (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's PyTorch path on the host cores

A step = student forward + backward + gradient all-reduce + AdamW on one batch of synthetic
(B,3,8,224,224) clips with synthetic (seeded, L2-normalised) teacher targets, InternVideo2-1B dims
(D=1408, 16x88 heads, hidden 6144, depth 40, 6 CLIP taps + 4 MAE taps), attention-style 80 % masking
(n = 417 visible tokens / clip), bf16, B = 32 clips per GPU (scripts/pretraining/1B_pt.sh:50).
One JSON line on stdout (rank 0).  See DESIGN.md §Measurement for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "clips/sec (device-timed) InternVideo2-1B VideoMAE 8x224^2 at 1/2/4/8 B200"

CFGS = {
    # name: (embed_dim, depth, heads, mlp_ratio, frames, clip taps, mae taps, default batch/GPU)
    "1B": dict(embed_dim=1408, depth=40, num_heads=16, mlp_ratio=48 / 11, num_frames=8, clip_return_layer=6,
               mae_return_layer=4, batch=32),
    # cfg-4: InternVideo2-6B stage-1, 16 frames, B=8/GPU (scripts/pretraining/6B_pt.sh:50), n = 1+16*52 = 833
    "6B": dict(embed_dim=3200, depth=48, num_heads=25, mlp_ratio=4, num_frames=16, clip_return_layer=6,
               mae_return_layer=4, batch=8),
    "S": dict(embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, num_frames=4, clip_return_layer=1,
              mae_return_layer=1, batch=8),
    # cfg-3: InternVideo2-L CLIP tower (scripts/pretraining/clip/L14/config.py: D=1024, 24 blocks, 16 heads, init 0.1,
    # frozen tower with open clip_projector), 4 frames, B = 128/GPU -> global batch 1024 on 8 GPUs
    "L": dict(embed_dim=1024, depth=24, num_heads=16, mlp_ratio=4, num_frames=4, batch=128),
}


CFG_TAG = {"1B": "cfg2", "6B": "cfg4", "S": "cfg1-like (small)", "L": "cfg3"}   # BASELINE.json configs[] indices


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json; dram__bytes_read.sum + dram__bytes_write.sum), or null."""
    f = ROOT / "profiles" / "ncu_traffic.json"
    if not f.exists():
        return {"traffic": None}
    t = json.loads(f.read_text())
    return {"traffic": t["dram_bytes_per_launch"], "traffic_unit": "bytes/launch",
            "traffic_algorithmic": t["algorithmic_bytes_per_launch"], "traffic_launch": t["launch"],
            "traffic_source": t["source"]}


def measured_peak_tflops():
    """(sustained bf16 TFLOP/s of this pool, where the number comes from)."""
    pk_file = ROOT / "MEASURED_PEAKS.json"
    if pk_file.exists():
        return (json.loads(pk_file.read_text()).get("bf16_tflops_sustained", 1400.0),
                "measured (MEASURED_PEAKS.json bf16_tflops_sustained)")
    return 1400.0, "fallback 1.4 PF/s sustained (B200_PROFILING.md)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ivb200", choices=["ivb200", "reference"])
    ap.add_argument("--model", default="1B", choices=list(CFGS))
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (default: recipe value)")
    ap.add_argument("--drop-path", type=float, default=0.25)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager steps instead of one CUDA graph per step")
    ap.add_argument("--one-cta", action="store_true", help="use the single-CTA GEMM kernel everywhere")
    ap.add_argument("--cpu-clips", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--seq", type=int, default=12544, help="--task attn: tokens per sequence (cfg-5: 1568 / 3136 / 6272 / 12544)")
    ap.add_argument("--head-dim", type=int, default=88, help="--task attn: head dimension (64 / 88 / 128), 16 heads")
    ap.add_argument("--task", default="mae", choices=["mae", "vtc", "attn"],
                    help="mae: stage-1 masked-video pretrain step (cfg-2/4); vtc: video-text contrastive step (cfg-3, use --model L)")
    ap.add_argument("--with-teachers", action="store_true",
                    help="mae: run the FULL recipe step — frozen InternVL-6B + VideoMAEv2-g teachers (random init) and the "
                         "attention-guided mask in front of the student step (SURVEY §8f-1); reported, not the headline config")
    ap.add_argument("--unfrozen", action="store_true",
                    help="vtc: train the whole vision tower (activation checkpointing on every block) instead of the "
                         "recipe's frozen tower + open clip_projector")
    ap.add_argument("--bucket-mb", type=float, default=256, help="gradient all-reduce bucket size (MB of bf16)")
    ap.add_argument("--first-bucket-mb", type=float, default=32,
                    help="size of the bucket that is reduced LAST (first layers), doubling per bucket up to --bucket-mb; 0 = uniform")
    ap.add_argument("--nccl-max-ctas", type=int, default=int(os.environ.get("IVB_NCCL_MAX_CTAS", "0")),
                    help="cap NCCL's CTAs per collective (NCCL_MAX_CTAS): the gradient all-reduce shares the SMs with the "
                         "persistent one-CTA-per-SM tcgen05 GEMMs of backward; 0 = NCCL's default")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "nvls", "nccl"],
                    help="gradient all-reduce: libivb200's in-switch NVLS kernel, ncclAllReduce, or nvls-if-available")
    ap.add_argument("--nvls-blocks", type=int, default=0, help="CTAs of the NVLS all-reduce kernel (default 8)")
    ap.add_argument("--zero1", action="store_true", help="shard the fp32 optimizer state over the ranks (ZeRO-1)")
    ap.add_argument("--lean", action="store_true",
                    help="profiling aid (ncu launch lists): skip the e2e and roofline passes; the line is NOT a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32; "
                         "large arrays as a fixed, seeded sample) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ivb200":
        ap.error("--dump-outputs writes the outputs of the ivb200 arm")
    return args


def host_cores():
    """Usable host cores: min(affinity mask, cgroup CPU quota); os.cpu_count() alone over-subscribes in containers."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(float(q[0]) / float(q[1]))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except Exception:
            pass
    return max(1, min(n, 64))


_THREADS = [None]


def pick_threads():
    """Thread count for the CPU arm: the fastest of {8,16,32,host_cores} on a 1.5 s matmul probe.
    (On the GPU boxes os.cpu_count() is 128 but the container gets far fewer real cores; 128 torch threads
    ran the same step 30x slower than 8 threads do here.)"""
    if _THREADS[0] is not None:
        return _THREADS[0]
    import torch
    hc = host_cores()
    cands = sorted({c for c in (8, 16, 32, hc) if c <= hc} or {hc})
    a = torch.randn(1536, 1536); b = torch.randn(1536, 1536)
    best, best_t = cands[0], 1e30
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.perf_counter()
        for _ in range(4):
            a @ b
        dt = time.perf_counter() - t0
        if dt < best_t * 0.9:
            best, best_t = c, dt
    torch.set_num_threads(best)
    _THREADS[0] = best
    return best


def flops_per_clip(cfg, n, fwd_only=False):
    D = cfg["embed_dim"]; Hd = int(D * cfg["mlp_ratio"]); L = cfg["depth"]
    blk = 2 * n * (4 * D * D + 2 * D * Hd) + 4 * n * n * D
    dec = cfg["clip_return_layer"] * 2 * n * D * 3200 + cfg["mae_return_layer"] * 2 * (n - 1) * (D * D + D * 1408)
    f = L * blk + dec
    return f if fwd_only else 3 * f


class ClockSampler:
    """nvidia-smi clocks / throttle reasons polled DURING the timed region (B200_PROFILING.md).
    One short nvidia-smi query every ~150 ms from a host thread (a `-lms` child block-buffers its pipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.index, self._stop, self.thread = [], index, False, None

    def _poll(self):
        while not self._stop:
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                    "-i", str(self.index)], capture_output=True, text=True, timeout=5)
                for line in r.stdout.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                return
            time.sleep(0.15)

    def start(self):
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self):
        self._stop = True
        if self.thread is not None:
            self.thread.join(timeout=6)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        sm.sort()
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_MAX_ELEMS = 1 << 22          # per array: 16 MB of float32; at most 3 arrays per task stay under 64 MB in all
PARAM_SAMPLE = 4096               # elements sampled from every parameter


def write_outputs(out_dir, arrays):
    """--dump-outputs: each tensor as out_dir/<name>.npy in float32.  A tensor of more than DUMP_MAX_ELEMS elements is
    replaced by the elements at DUMP_MAX_ELEMS fixed, seeded positions (the same positions in every run)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for i, (name, t) in enumerate(arrays.items()):
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(i)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def param_sample(model):
    """PARAM_SAMPLE elements at fixed, seeded positions of every parameter (in named_parameters() order), concatenated."""
    import torch
    g = torch.Generator().manual_seed(0)
    parts = []
    for _, p in model.named_parameters():
        idx = torch.randint(p.numel(), (min(p.numel(), PARAM_SAMPLE),), generator=g).sort().values
        parts.append(p.detach().reshape(-1)[idx.to(p.device)].float())
    return torch.cat(parts)


def make_mask(B, T, L, keep, seed):
    """Attention-style mask of the recipe with uniform importance: per frame keep 52 of 256 patches
    (engine_for_pretraining.py:105-116), cls always visible.  bool [B, 1+T*L], True = masked."""
    import torch
    g = torch.Generator().manual_seed(seed)
    m = torch.ones(B, T, L, dtype=torch.bool)
    for b in range(B):
        for t in range(T):
            m[b, t, torch.randperm(L, generator=g)[:keep]] = False
    return torch.cat([torch.zeros(B, 1, dtype=torch.bool), m.reshape(B, T * L)], dim=1)


def _finish(world):
    """Multi-rank exit: barrier, then leave without tearing NCCL down — destroy_process_group() after a CUDA
    graph that holds NCCL nodes was observed to hang the 2-GPU run at exit (the JSON line was already out)."""
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


# ============================================================================================ cfg-5: attention only
def run_attn(args):
    """BASELINE cfg-5: attention forward + backward alone at one sequence length (single GPU by definition; with N > 1 every
    rank runs a replica — "replicas only", no collective).  A step = one forward + one backward over B sequences of `--seq`
    tokens, 16 heads of `--head-dim`, read in place from a packed [B*n, 3D] projection buffer (flash_attention_class.py:47-50
    is the seam).  value = sequences/s; roofline = algorithmic 14 n^2 D flop per sequence / device time against the sustained
    bf16 peak.  L2 is flushed between steps."""
    import torch
    import torch.distributed as dist
    from internvideo_b200 import lowlevel as ll

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ll.device_check()
    n, H, d = args.seq, 16, args.head_dim
    D = H * d
    B = args.batch or max(1, 12544 // n)
    bf = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(7 + rank)
    qkv = (torch.randn(B * n, 3 * D, device="cuda", generator=g) * 0.5).to(bf)
    dout = torch.randn(B * n, D, device="cuda", generator=g).to(bf)
    host_qkv = qkv.cpu().pin_memory()
    dqkv = torch.empty_like(qkv)
    q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
    out, lse = ll.attn_fwd(q, k, v, B, n, H, d, d ** -0.5)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def step():
        ll.attn_fwd(q, k, v, B, n, H, d, d ** -0.5, out=out)
        ll.attn_bwd(q, k, v, out, dout, lse, B, n, H, d, d ** -0.5, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:])

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sync()
    clocks = ClockSampler(local); clocks.start()
    ll.reset_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for e0, e1 in ev:
        flush.zero_()
        e0.record(); step(); e1.record()
    sync()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"out": out, "lse": lse, "dqkv": dqkv})
    ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = ll.launch_count()
    # end to end: the projection buffer comes from pinned host memory, one gradient element is read back
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        qkv.copy_(host_qkv, non_blocking=True)
        step()
        lv = float(dqkv[0, 0].item())
    e3.record(); sync()
    ms_e2e = e2.elapsed_time(e3)
    clk = clocks.stop()
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    if rank == 0:
        peak_tf, peak_src = measured_peak_tflops()
        flops = 14.0 * B * H * n * n * d                                   # 4 n^2 D forward + 10 n^2 D backward
        achieved = flops * args.steps / ms / 1e9
        out_line = {
            "metric": "attention fwd+bwd sequences/sec (device-timed) and fraction of the attention-GEMM roofline", "value": round(B * world * args.steps / (ms / 1e3), 3), "unit": "sequences/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"cfg5: attention forward + backward only, {n} tokens x 16 heads x {d}, batch {B} "
                                   f"(replicas only at N > 1)", "seq_len": n, "head_dim": d, "batch_per_gpu": B,
                       "l2": "256 MB written between steps"},
            "clocks": clk,
            "e2e": {"value": round(B * world * args.steps / (ms_e2e / 1e3), 3), "unit": "sequences/s",
                    "h2d_bytes_per_step": host_qkv.numel() * 2, "d2h_bytes_per_step": 2, "last": lv},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "attn_fwd2_kernel + attn_bwd_kernel (tcgen05)", "achieved": round(achieved, 1),
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4), "peak_source": peak_src,
                         "traffic": None},
            "cpu_baseline": None}
        print(json.dumps(out_line), flush=True)
    _finish(world)


# ============================================================================================ ivb200 arm
def attention_roofline(attn, nprof, ms_step, peak=None):
    """BASELINE's metric asks for the achieved fraction of the attention-GEMM roofline: algorithmic attention FLOPs
    (fwd 4 n^2 D, bwd 10 n^2 D per clip per block) / CUDA-event time of the attention launches, against the same
    measured sustained bf16 peak as the GEMM record."""
    pk_file = ROOT / "MEASURED_PEAKS.json"
    if peak is None:
        peak = json.loads(pk_file.read_text()).get("bf16_tflops_sustained", 1400.0) if pk_file.exists() else 1400.0
    out = {"peak": peak, "unit": "TFLOP/s"}
    tot_f = tot_ms = 0.0
    for k, (fl, ms_) in attn.items():
        if ms_ > 0:
            out[k] = {"achieved": round(fl / (ms_ * 1e-3) / 1e12, 1), "frac": round(fl / (ms_ * 1e-3) / 1e12 / peak, 4),
                      "ms_per_step": round(ms_ / nprof, 3)}
            tot_f += fl; tot_ms += ms_
    if tot_ms > 0:
        out["achieved"] = round(tot_f / (tot_ms * 1e-3) / 1e12, 1)
        out["frac"] = round(out["achieved"] / peak, 4)
        out["ms_per_step"] = round(tot_ms / nprof, 3)
        out["share_of_step"] = round((tot_ms / nprof) / ms_step, 4)
    return out


def measure(args, world, local, step, dev_inputs, host_inputs, engine):
    """Warm up, capture the step into one CUDA graph, then time: (1) K steps on device-resident inputs, (2) K steps
    fed from pinned HOST buffers with the loss read back every step (e2e), (3) a few eager steps with CUDA events
    around every GEMM launch (roofline).  Barrier + synchronize on both sides, max over ranks.  With --dump-outputs,
    the loss of the last step of (1) and a sample of the parameters it left are written before (2) changes them."""
    import torch
    import torch.distributed as dist
    from internvideo_b200 import lowlevel as ll

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # -------- warm-up (eager), then optionally capture the whole step into one CUDA graph
    for _ in range(args.warmup):
        step(*dev_inputs)
    sync()
    graphed = None
    launches_per_step = None
    # Whole-step CUDA graph (NCCL all-reduce nodes included when N > 1; verified at N=2).
    if not args.no_graph:
        from internvideo_b200.engine import GraphedStep
        ll.reset_launch_count()
        try:
            graphed = GraphedStep(step, list(dev_inputs), warmup=1)
            launches_per_step = ll.launch_count() // 2          # 1 warm-up + 1 captured pass
        except Exception as e:                                  # noqa: BLE001 — report and fall back to eager
            print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); timing eager steps", file=sys.stderr)
            graphed = None
            torch.cuda.synchronize()
    run = (lambda *a: graphed(*a)) if graphed is not None else step
    for _ in range(2):
        run(*dev_inputs)
    sync()
    # -------- device-resident timing (value)
    clocks = ClockSampler(local); clocks.start()
    ll.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if args.lean:
        torch.cuda.profiler.start()     # `ncu --profile-from-start off`: the launch list covers the timed steps only
    e0.record()
    for _ in range(args.steps):
        loss = run(*dev_inputs)
    e1.record(); sync()
    if args.lean:
        torch.cuda.profiler.stop()
    if args.dump_outputs and int(os.environ.get("RANK", 0)) == 0:
        write_outputs(args.dump_outputs, {"loss": loss, "params_sample": param_sample(engine.model)})
    ms = e0.elapsed_time(e1)
    launches = ll.launch_count() if graphed is None else launches_per_step * args.steps
    # -------- end-to-end timing through the public API with HOST buffers (e2e)
    if graphed is not None:
        feed = lambda: host_inputs                              # GraphedStep copies them into its static buffers
    else:
        feed = lambda: tuple(t.cuda(non_blocking=True) for t in host_inputs)
    for _ in range(0 if args.lean else 2):
        float(run(*feed()).item())
    sync()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    lv = float("nan")
    for _ in range(0 if args.lean else args.steps):
        lv = float(run(*feed()).item())          # H2D of video+mask and D2H read of the loss every step
    e3.record(); sync()
    ms_e2e = e2.elapsed_time(e3) if not args.lean else ms
    clk = clocks.stop()
    # -------- roofline pass: the same step, eager, with CUDA events around every GEMM launch.  The graph's private pool
    # (every activation of a step) is released first: with it alive the eager steps run at the edge of the 180 GB and
    # the caching allocator's retries dominate them (6B: out of memory).
    was_graphed = graphed is not None
    if was_graphed and world == 1:      # (multi-rank graphs hold an NCCL node: they are left alone, as measured at N = 2 / 8)
        import gc
        loss = None; run = None; feed = None
        graphed.graph.reset(); graphed = None
        gc.collect(); torch.cuda.empty_cache()
    prof = ll.GemmProfiler(); prof.enable()
    nprof = 1 if args.lean else min(args.steps, 3)
    engine.comm_profile = world > 1
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record()
    for _ in range(nprof):
        step(*dev_inputs)
    e5.record(); sync()
    prof.disable()
    comm = engine.comm_report(nprof) if world > 1 else None
    engine.comm_profile = False
    if comm is not None and engine.allreduce_note:
        comm["note"] = engine.allreduce_note
    ms_prof = e4.elapsed_time(e5)
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    gflops, gms = prof.totals()
    attn = {k: prof.totals(k) for k in ("attn_fwd", "attn_bwd")}
    # data-parallel sanity: after identical updates every rank must hold bit-identical parameters.
    # max |param - rank 0's param| over all parameters and ranks; anything but 0.0 fails the run.
    spread = None
    if world > 1:
        spread = float(engine.replica_divergence().item())
        if spread != 0.0:
            print(f"[bench] FATAL: data-parallel replicas diverged (max |param - rank0 param| = {spread:.3e})",
                  file=sys.stderr, flush=True)
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(3)
    return dict(ms=ms, ms_e2e=ms_e2e, clk=clk, gflops=gflops, gms=gms, prof_count=prof.count, nprof=nprof, ms_prof=ms_prof,
                graphed=(True if was_graphed else None), launches=launches, lv=lv, spread=spread, attn=attn, comm=comm)


def run_ivb200(args):
    import torch
    import torch.distributed as dist
    from internvideo_b200 import lowlevel as ll
    from internvideo_b200.engine import PretrainEngine
    from internvideo_b200.modules import PretrainInternVideo2

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        if args.nccl_max_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(args.nccl_max_ctas)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ll.device_check()
    ll.set_default_2cta(not args.one_cta)
    cfg = dict(CFGS[args.model])
    B = args.batch or cfg.pop("batch"); cfg.pop("batch", None)
    T, L, keep = cfg["num_frames"], 256, 52
    n = 1 + T * keep
    torch.manual_seed(0)           # identical init on every rank (the engine broadcasts rank 0's parameters anyway)
    with torch.device("cuda"):     # random init of the named architecture directly in HBM (no checkpoints offline)
        model = PretrainInternVideo2(drop_path_rate=args.drop_path, clip_teacher_embed_dim=3200,
                                     clip_teacher_final_dim=768, mae_teacher_embed_dim=1408, init_values=1e-5,
                                     attn_pool_num_heads=16, clip_embed_dim=768, use_flash_attn=True,
                                     use_fused_rmsnorm=True, use_fused_mlp=True, **cfg)
    model = model.bfloat16().cuda().train()
    engine = PretrainEngine(model, lr=1.5e-4, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.05, clip_grad=3.0,
                            bucket_mb=args.bucket_mb, first_bucket_mb=args.first_bucket_mb, zero1=args.zero1, check_finite=True,
                            allreduce=args.allreduce)
    if args.nvls_blocks > 0 and engine.nvls is not None:
        engine.nvls.nblocks = args.nvls_blocks
    torch.manual_seed(args.seed + rank)    # run_pretraining.py:  seed = args.seed + get_rank() — per-rank DropPath draws
    nparams = sum(p.numel() for p in model.parameters())
    g = torch.Generator().manual_seed(1234 + rank)
    K, Km = cfg["clip_return_layer"], cfg["mae_return_layer"]
    host_video = torch.randn(B, 3, T, 224, 224, generator=g).to(torch.bfloat16).pin_memory()
    host_mask = make_mask(B, T, L, keep, 1234 + rank).pin_memory()
    dev_video = host_video.cuda(); dev_mask = host_mask.cuda()
    gd = torch.Generator(device="cuda").manual_seed(99 + rank)
    nrm = torch.nn.functional.normalize
    tgt_clip = nrm(torch.randn(K, B * n, 3200, device="cuda", generator=gd), dim=-1).to(torch.bfloat16)
    tgt_final = nrm(torch.randn(B, 768, device="cuda", generator=gd), dim=-1).to(torch.bfloat16)
    tgt_mae = nrm(torch.randn(Km, B * (n - 1), 1408, device="cuda", generator=gd), dim=-1).to(torch.bfloat16)

    def step(video, mask):
        engine.zero_grad()
        lc, lf, lm = model.forward_loss(video, mask, tgt_clip, tgt_final, tgt_mae, n_visible=n)
        loss = lc + lf + lm
        loss.backward()
        engine.step()
        return loss

    teacher_note = ""
    if args.with_teachers:
        # the real recipe (scripts/pretraining/1B_pt.sh): InternVL-6B CLIP teacher on the 8 student frames (per-frame,
        # 257 tokens, 6 taps) + VideoMAEv2-g on 16 frames (tubelet 2 -> 2048 tokens, 4 taps), attention-guided 80 % mask
        from functools import partial
        from internvideo_b200.teachers import DistillationStep, InternVL_CLIP, VisionTransformer
        del tgt_clip, tgt_final, tgt_mae
        with torch.device("cuda"):
            clip_t = InternVL_CLIP(img_size=224, layerscale_no_force_fp32=False, clip_return_layer=K, clip_return_interval=1)
            mae_t = VisionTransformer(img_size=224, patch_size=14, embed_dim=1408, depth=40, num_heads=16, mlp_ratio=48 / 11,
                                      qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), all_frames=2 * T,
                                      tubelet_size=2, mae_return_layer=Km, mae_return_interval=1)
        clip_t = clip_t.bfloat16().cuda().eval(); mae_t = mae_t.bfloat16().cuda().eval()
        dstep = DistillationStep(model, engine, clip_t, mae_t, mask_ratio=0.8, td_ratio=2)
        host_video = torch.randn(B, 3, 2 * T, 224, 224, generator=g).to(torch.bfloat16).pin_memory()
        dev_video = host_video.cuda()
        tp = sum(p.numel() for p in clip_t.parameters()) + sum(p.numel() for p in mae_t.parameters())
        teacher_note = f" + frozen teachers (InternVL-6B per-frame + VideoMAEv2-g, {tp / 1e9:.2f} B params, random init) + attention-guided mask"

        def step(video, _mask):          # noqa: F811 — same signature as the student-only step
            return dstep(video)

    m = measure(args, world, local, step, (dev_video, dev_mask), (host_video, host_mask), engine)
    ms, ms_e2e, clk, gflops, gms, prof_count, nprof, ms_prof = (m[k] for k in ("ms", "ms_e2e", "clk", "gflops", "gms", "prof_count", "nprof", "ms_prof"))
    graphed, launches, lv, spread = m["graphed"], m["launches"], m["lv"], m["spread"]
    attn_roof = attention_roofline(m["attn"], nprof, ms / args.steps)
    if rank != 0:
        _finish(world)
        return
    peaks = {}
    pk_file = ROOT / "MEASURED_PEAKS.json"
    if pk_file.exists():
        peaks = json.loads(pk_file.read_text())
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PF/s sustained (B200_PROFILING.md)"
    achieved = gflops / (gms * 1e-3) / 1e12 if gms > 0 else 0.0
    total_clips = B * world * args.steps
    value = total_clips / (ms * 1e-3)
    e2e_value = total_clips / (ms_e2e * 1e-3)
    fpc = flops_per_clip(CFGS[args.model], n)
    metric = METRIC if args.model == "1B" else METRIC.replace("InternVideo2-1B VideoMAE 8x224^2", f"InternVideo2-{args.model} VideoMAE {T}x224^2")
    out = {
        "metric": metric, "value": round(value, 3), "unit": "clips/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{CFG_TAG.get(args.model, 'cfg')}: InternVideo2-{args.model} stage-1 masked-video pretrain step "
                               f"(student fwd+bwd + grad all-reduce + AdamW, clip 3.0), {T}f 224^2, "
                               f"n={n} visible tokens, {K} CLIP + {Km} MAE taps, drop_path {args.drop_path}" + teacher_note,
                   "batch_per_gpu": B, "global_batch": B * world, "params": nparams, "parallelism": f"dp{world}", "cuda_graph": graphed is not None,
                   "l2": "per-step working set (2 GB weights + >30 GB activations) >> 126 MB L2; no flush needed",
                   "model_tflops_per_clip": round(fpc / 1e12, 4),
                   "model_tflops_per_s": round(value * fpc / 1e12, 1),
                   "replica_param_max_abs_diff": spread, "zero1": bool(args.zero1),
                   "bucket_mb": args.bucket_mb, "nccl_max_ctas": args.nccl_max_ctas or None,
                   "allreduce": engine.allreduce, "comm": m["comm"]},
        "clocks": clk,
        "e2e": {"value": round(e2e_value, 3), "unit": "clips/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": host_video.numel() * 2 + host_mask.numel(), "d2h_bytes_per_step": 4,
                "last_loss": lv},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05)", "achieved": round(achieved, 1),
                     "peak": peak_tf, "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4),
                     "peak_source": peak_src, **ncu_traffic(),
                     # device time of the GEMM launches per step / the timed (graph-replayed) step: the eager
                     # profiling pass itself is host-issue bound, so its wall time is not the denominator
                     "gemm_share_of_step": round((gms / nprof) / (ms / args.steps), 4),
                     "gemm_ms_per_step": round(gms / nprof, 3), "gemm_launches": prof_count,
                     "timed": f"CUDA events around every GEMM launch in {nprof} eager step(s) of the same workload "
                              f"run right after the timed region ({round(ms_prof / nprof, 2)} ms/step eager)",
                     "attention": attn_roof},
    }
    if args.lean:
        out["lean"] = "profiling run: no e2e / single roofline pass — not a bench value"
    if not args.no_cpu_baseline and world == 1 and not args.lean:
        out["cpu_baseline"] = cpu_baseline(args, clips=args.cpu_clips, reps=1)
    print(json.dumps(out), flush=True)
    _finish(world)


# ============================================================================================ cfg-3: contrastive step
def run_vtc(args):
    """BASELINE cfg-3: InternVideo2-L video-text contrastive step — unmasked tower over 1 + 4*256 tokens, attention-pool
    projector, vision_align, packed cross-rank all-gather of (vision | text | idx), soft-target two-way CE with the
    learnable temperature, backward, gradient all-reduce, AdamW.  Text embeddings are synthetic [B, 512] (the
    MobileCLIP text tower is outside the hot path and frozen in the recipe).  Default = the recipe's frozen tower with
    the clip_projector open (scripts/pretraining/clip/L14/config.py); --unfrozen trains every block with activation
    checkpointing (the recipe's gradient_checkpointing=True)."""
    import torch
    import torch.distributed as dist
    from internvideo_b200 import lowlevel as ll
    from internvideo_b200.clip_modules import InternVideo2_CLIP_small
    from internvideo_b200.engine import PretrainEngine

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        if args.nccl_max_ctas > 0:
            os.environ["NCCL_MAX_CTAS"] = str(args.nccl_max_ctas)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ll.device_check()
    ll.set_default_2cta(not args.one_cta)
    if args.model not in ("L", "S"):
        raise SystemExit("--task vtc is defined for --model L (cfg-3) or S (smoke)")
    cfg = dict(CFGS[args.model])
    B = args.batch or cfg.pop("batch"); cfg.pop("batch", None)
    for k in ("clip_return_layer", "mae_return_layer"):
        cfg.pop(k, None)
    T = cfg["num_frames"]
    n = 1 + T * 256
    ve = dict(in_chans=3, patch_size=14, img_size=224, qkv_bias=False, drop_path_rate=0.0, head_drop_path_rate=0.0,
              init_values=0.1, qk_normalization=True, use_flash_attn=True, use_fused_rmsnorm=True, use_fused_mlp=True,
              fused_mlp_heuristic=1, attn_pool_num_heads=16, clip_embed_dim=768, layerscale_no_force_fp32=True,
              tubelet_size=1, sep_pos_embed=False, use_checkpoint=bool(args.unfrozen),
              checkpoint_num=cfg["depth"] if args.unfrozen else 0, align_dim=512, **cfg)
    conf = dict(model=dict(vision_encoder=ve, temp=1 / 100.0, temp_min=1 / 100.0, freeze_vision=not args.unfrozen,
                           open_vision_clip_projector=True, freeze_text=True))
    torch.manual_seed(0)
    with torch.device("cuda"):
        model = InternVideo2_CLIP_small(conf)
    model = model.bfloat16().cuda().train()
    engine = PretrainEngine(model, lr=4e-4, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.2, clip_grad=0.0,
                            bucket_mb=args.bucket_mb, first_bucket_mb=args.first_bucket_mb, zero1=args.zero1, check_finite=True,
                            allreduce=args.allreduce)
    if args.nvls_blocks > 0 and engine.nvls is not None:
        engine.nvls.nblocks = args.nvls_blocks
    torch.manual_seed(args.seed + rank)
    nparams = sum(p.numel() for p in model.parameters())
    ntrain = sum(p.numel() for p in model.parameters() if p.requires_grad)
    g = torch.Generator().manual_seed(1234 + rank)
    host_image = torch.randn(B, T, 3, 224, 224, generator=g).to(torch.bfloat16).pin_memory()     # [B,T,C,H,W]
    host_text = torch.randn(B, 512, generator=g).pin_memory()
    idx = (torch.arange(B) + rank * B).cuda()                      # all captions distinct (SURVEY §8d)
    dev_image, dev_text = host_image.cuda(), host_text.cuda()

    def step(image, text):
        engine.zero_grad()
        loss = model(image, text, idx)["loss_vtc"]
        loss.backward()
        engine.step()
        return loss

    m = measure(args, world, local, step, (dev_image, dev_text), (host_image, host_text), engine)
    ms, ms_e2e, clk, gflops, gms, nprof = (m[k] for k in ("ms", "ms_e2e", "clk", "gflops", "gms", "nprof"))
    if rank != 0:
        _finish(world)
        return
    pk_file = ROOT / "MEASURED_PEAKS.json"
    peaks = json.loads(pk_file.read_text()) if pk_file.exists() else {}
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    D, Hd, depth = cfg["embed_dim"], int(cfg["embed_dim"] * cfg["mlp_ratio"]), cfg["depth"]
    fwd = depth * (2 * n * (4 * D * D + 2 * D * Hd) + 4 * n * n * D)
    fpc = fwd * (4 if args.unfrozen else 1)           # unfrozen: fwd + recompute + 2x bwd; frozen: tower forward only
    total = B * world * args.steps
    value, e2e_value = total / (ms * 1e-3), total / (ms_e2e * 1e-3)
    achieved = gflops / (gms * 1e-3) / 1e12 if gms > 0 else 0.0
    out = {
        "metric": f"clips/sec (device-timed) InternVideo2-{args.model} video-text contrastive {T}x224^2 at 1/2/4/8 B200",
        "value": round(value, 3), "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{CFG_TAG.get(args.model)}: InternVideo2-{args.model} multi_modality video-text contrastive step "
                               f"({'whole tower trained, every block checkpointed' if args.unfrozen else 'frozen tower, open clip_projector (recipe)'}; "
                               f"fwd over n={n} unmasked tokens + vision_align + packed all-gather + VTC loss + bwd + grad all-reduce + AdamW), "
                               f"{T}f 224^2, synthetic text embeddings [B,512]",
                   "batch_per_gpu": B, "global_batch": B * world, "params": nparams, "trainable_params": ntrain,
                   "parallelism": f"dp{world}", "cuda_graph": m["graphed"] is not None,
                   "l2": "per-step working set (activations of 131k tokens) >> 126 MB L2; no flush needed",
                   "model_tflops_per_clip": round(fpc / 1e12, 4), "model_tflops_per_s": round(value * fpc / 1e12, 1),
                   "replica_param_max_abs_diff": m["spread"], "zero1": bool(args.zero1),
                   "allreduce": engine.allreduce, "comm": m["comm"]},
        "clocks": clk,
        "e2e": {"value": round(e2e_value, 3), "unit": "clips/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": host_image.numel() * 2 + host_text.numel() * 4, "d2h_bytes_per_step": 4,
                "last_loss": m["lv"]},
        "gpu_launches": int(m["launches"]),
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05)", "achieved": round(achieved, 1), "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4), "traffic": None,
                     "gemm_share_of_step": round((gms / nprof) / (ms / args.steps), 4),
                     "gemm_ms_per_step": round(gms / nprof, 3), "gemm_launches": m["prof_count"],
                     "attention": attention_roofline(m["attn"], nprof, ms / args.steps, peak_tf)},
    }
    print(json.dumps(out), flush=True)
    _finish(world)


# ============================================================================================ CPU arms
def cpu_step_fn(args, clips):
    """The reference's path on the host cores: the UNMODIFIED reference modules when /root/reference is
    mounted (kind 'reference'), else the oracle port (oracle/restate.py, kind 'port')."""
    import torch
    from oracle import ref_shim, restate
    cfg = dict(CFGS[args.model]); cfg.pop("batch")
    T, L, keep = cfg["num_frames"], 256, 52
    n = 1 + T * keep
    pick_threads()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(clips, 3, T, 224, 224, generator=g)
    mask = make_mask(clips, T, L, keep, 1234)
    K, Km = cfg["clip_return_layer"], cfg["mae_return_layer"]
    nrm = torch.nn.functional.normalize
    tg = [nrm(torch.randn(K, clips, n, 3200, generator=g), dim=-1), nrm(torch.randn(clips, 768, generator=g), dim=-1),
          nrm(torch.randn(Km, clips, n - 1, 1408, generator=g), dim=-1)]
    if ref_shim.available():
        kind = "reference"
        model = ref_shim.build_reference_model(drop_path_rate=0.0, init_values=1e-5, **cfg).train()
        params = list(model.parameters())

        def fwd():
            return model(x, mask)
    else:
        kind = "port"
        from internvideo_b200.modules import PretrainInternVideo2
        with torch.device("meta"):            # key/shape layout only; values drawn below (cheap, no 1B-param init pass)
            shell = PretrainInternVideo2(drop_path_rate=0.0, init_values=1e-5, use_flash_attn=False,
                                         use_fused_rmsnorm=False, use_fused_mlp=False, **cfg)
        p = {}
        for k, v in shell.state_dict().items():
            t = torch.empty(v.shape, dtype=torch.float32)
            if k.endswith("gamma"):
                t.fill_(1e-5)
            elif "norm" in k and k.endswith("weight"):
                t.fill_(1.0)
            elif k.endswith("bias"):
                t.zero_()
            else:
                t.normal_(0.0, 0.02, generator=g)
            p[k] = t.requires_grad_(True)
        del shell
        params = [v for v in p.values() if v.requires_grad]
        depth = cfg["depth"]
        rc = dict(depth=depth, num_heads=cfg["num_heads"], attn_pool_num_heads=16, patch_size=14, tubelet_size=1,
                  clip_return_index=[depth - 1 - i for i in range(K)], mae_return_index=[depth - 1 - i for i in range(Km)])

        def fwd():
            return restate.forward_pretrain(p, rc, x, mask)

    def step():
        for q in params:
            q.grad = None
        out = fwd()
        loss = sum((2 - 2 * (o * t).sum(-1)).mean() for o, t in zip(out, tg))
        loss.backward()
        return float(loss)
    return step, kind, clips


def cpu_baseline(args, clips=1, reps=1):
    step, kind, clips = cpu_step_fn(args, clips)
    step()  # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    return {"value": round(clips / dt, 5), "unit": "clips/s", "cores": pick_threads(), "kind": kind,
            "sample": f"{clips} clip(s) fwd+bwd of the same cfg (fp32, torch CPU, {pick_threads()} threads), "
                      f"{reps} timed rep(s) after 1 warm-up; no optimizer step"}


def cpu_vtc_step_fn(args, clips):
    """cfg-3 on the host cores: the reference's unmasked InternVideo2 tower (unmodified module when the reference
    sources are present, else the oracle port) -> vision_align -> vtc_loss, frozen tower (forward only) + backward
    through the projector, fp32."""
    import torch
    from oracle import ref_shim, restate
    cfg = dict(CFGS[args.model]); cfg.pop("batch")
    for k in ("clip_return_layer", "mae_return_layer"):
        cfg.pop(k, None)
    T = cfg["num_frames"]
    pick_threads()
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(1234)
    image = torch.randn(clips, T, 3, 224, 224, generator=g)
    text = torch.randn(clips, 512, generator=g)
    idx = torch.arange(clips)
    D = cfg["embed_dim"]
    if ref_shim.available():
        kind = "reference"
        mod = ref_shim.import_clip_vision()
        crit, _ = ref_shim.import_criterions()
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            tower = mod.InternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, drop_path_rate=0.0,
                                     init_values=0.1, clip_embed_dim=768, attn_pool_num_heads=16, **cfg).train()
        align = torch.nn.Sequential(torch.nn.LayerNorm(768), torch.nn.Linear(768, 512))
        for n_, p_ in tower.named_parameters():
            p_.requires_grad = n_.startswith("clip_projector")
        temp = torch.nn.Parameter(torch.ones([]) * 0.01)
        loss_fn = crit.VTC_VTM_Loss(False)

        def step():
            for q in list(tower.parameters()) + list(align.parameters()) + [temp]:
                q.grad = None
            v = align(tower(image.permute(0, 2, 1, 3, 4)))
            loss = loss_fn.vtc_loss(v, text, idx, temp, all_gather=False)
            loss.backward()
            return float(loss.detach())
    else:
        kind = "port"
        from internvideo_b200.clip_modules import InternVideo2
        with torch.device("meta"):
            shell = InternVideo2(use_flash_attn=False, use_fused_rmsnorm=False, use_fused_mlp=False, init_values=0.1,
                                 clip_embed_dim=768, attn_pool_num_heads=16, **cfg)
        p = {}
        for k, v in shell.state_dict().items():
            t = torch.empty(v.shape, dtype=torch.float32)
            if k.endswith("gamma"):
                t.fill_(0.1)
            elif "norm" in k and k.endswith("weight"):
                t.fill_(1.0)
            elif k.endswith("bias"):
                t.zero_()
            else:
                t.normal_(0.0, 0.02, generator=g)
            p["vision_encoder." + k] = t.requires_grad_(k.startswith("clip_projector"))
        p["vision_align.0.weight"] = torch.ones(768, requires_grad=True); p["vision_align.0.bias"] = torch.zeros(768, requires_grad=True)
        p["vision_align.1.weight"] = (torch.randn(512, 768, generator=g) * 0.02).requires_grad_(True)
        p["vision_align.1.bias"] = torch.zeros(512, requires_grad=True)
        temp = torch.tensor(0.01, requires_grad=True)
        rc = dict(depth=cfg["depth"], num_heads=cfg["num_heads"], attn_pool_num_heads=16, patch_size=14, tubelet_size=1,
                  num_frames=T)

        def step():
            for q in p.values():
                q.grad = None
            v = restate.clip_small_embed(p, rc, image)
            loss = restate.vtc_loss(v, text, idx, temp)
            loss.backward()
            return float(loss.detach())
    return step, kind, clips


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    if args.task == "vtc":
        clips = max(args.cpu_clips, 2)
        step, kind, clips = cpu_vtc_step_fn(args, clips)
        for _ in range(min(args.warmup, 1)):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = time.perf_counter() - t0
        value = clips * args.steps / dt
        T = CFGS[args.model]["num_frames"]
        out = {"impl": "reference",
               "metric": f"clips/sec (device-timed) InternVideo2-{args.model} video-text contrastive {T}x224^2 at 1/2/4/8 B200",
               "value": round(value, 5), "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps,
               "warmup": min(args.warmup, 1), "ms_per_step": round(dt / args.steps * 1e3, 1), "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": f"{CFG_TAG.get(args.model)}: InternVideo2-{args.model} video-text contrastive step on the host cores "
                                      f"(frozen tower fwd + projector/vision_align/temp bwd, naive PyTorch path), {T}f 224^2, n={1 + T * 256}",
                          "batch_per_step": clips},
               "cpu_baseline": {"value": round(value, 5), "unit": "clips/s", "cores": pick_threads(), "kind": kind,
                                "sample": f"each step = {clips} clip(s), fp32, {pick_threads()} threads"},
               "e2e": {"value": round(value, 5), "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "gpu_launches": 0}
        print(json.dumps(out), flush=True)
        return
    clips = args.cpu_clips
    step, kind, clips = cpu_step_fn(args, clips)
    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = clips * args.steps / dt
    cfg = CFGS[args.model]
    n = 1 + cfg["num_frames"] * 52
    out = {"impl": "reference", "metric": METRIC, "value": round(value, 5), "unit": "clips/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1),
           "ms_per_step": round(dt / args.steps * 1e3, 1), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{CFG_TAG.get(args.model, 'cfg')}: InternVideo2-{args.model} stage-1 masked-video pretrain step on the host "
                                  f"cores (student fwd+bwd, naive PyTorch path), {cfg['num_frames']}f 224^2, n={n}",
                      "batch_per_step": clips},
           "cpu_baseline": {"value": round(value, 5), "unit": "clips/s", "cores": pick_threads(), "kind": kind,
                            "sample": f"each step = {clips} clip(s) fwd+bwd, fp32, {pick_threads()} threads"},
           "e2e": {"value": round(value, 5), "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.task == "vtc":
        run_vtc(a)
    elif a.task == "attn":
        run_attn(a)
    else:
        run_ivb200(a)
