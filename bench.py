#!/usr/bin/env python
"""bench.py -- throughput of the ABC-Net hot path (batched U-Net forward + heat-map decode) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 256] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): v2 ABC-Net U-Net, 256 synthetic binary 1x512x512 images per GPU per step,
bf16 activations / fp32 accumulation, followed by the fused peak-decode kernel. One "step" = one batch.
  value  : images/s, inputs already resident in HBM, timed with CUDA events, max over ranks
  e2e    : same metric through the public API with pinned HOST images (H2D inside the timed region) and a D2H read
           of the decoded peak records every step
  roofline: the dominant launch (the fused 8-head conv1 implicit GEMM) timed live with CUDA events inside the timed
           steps; peak from MEASURED_PEAKS.json (sustained bf16, kernel timed inside a long step)
  cpu_baseline: the CPU oracle port of the same path (fp32 torch on the host cores) on a bounded sample
--impl reference times that CPU path alone (the reference ships no native code; /root/reference is absent on the
GPU box, so the oracle port -- same ATen ops on a state_dict -- stands in; kind "port").
Multi-GPU: one process per GPU (torchrun), images sharded, no data-path collective, weak scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HEADS = [1, 14, 3, 2, 1, 360, 60, 60]
HEAD_NAMES = ("atom_target", "atom_type", "atom_charge", "atom_hs", "bond_target", "bond_type", "bond_rho", "bond_omega_type")
# (image, y, x) positions whose logits --dump-outputs writes: 8192 x 501 channels x 4 B = 16 MB; with the records at the default
# batch and capacities filled to the brim (256 x (1024 + 4096) x 24 B = 31 MB) the dump stays under 64 MB
DUMP_PIXELS = 8192
METRIC = "images_per_sec_unet_fwd_decode"
UNIT = "images/s"
FLOPS_PER_IMAGE = 93.98e9          # SURVEY.md section 6 (forward, v2 heads, 512x512)
HEADS_CONV1_FLOPS_PER_IMAGE = 2.0 * 128 * 128 * 1024 * 1152      # fused 8-head 3x3 conv: M=16384, N=1024, K=1152
# dram__bytes_read.sum + dram__bytes_write.sum of that launch at batch 256 are READ from the newest committed `ncu --set full`
# summary of the kernel under profiles/ (see ncu_traffic); algorithmic: 1.07 GB trunk in + 8.59 GB hidden out
HEADS_CONV1_SUMMARY_GLOB = "r*_heads_conv1_b256*.summary.txt"
HEADS_CONV2_FLOPS_PER_IMAGE = 2.0 * 128 * 128 * 128 * 501        # the eight 1x1 convs, algorithmic (unpadded) channels
HEADS_FUSED_DRAM_BYTES_B256 = None                                # filled from the ncu capture of heads_fused_kernel


def _conv_flops(cin, cout, hw, taps=9):
    return 2.0 * cin * cout * taps * hw * hw


# Per-image algorithmic work of every launch group of the forward pass (SURVEY.md App. A.1 / section 8d): FLOPs for the
# tensor-class layers, bytes (input read once + output written once, bf16 activations, fp32 logits) for the HBM class.
LAYER_CLASSES = {
    "first conv 1->16 @512 (HBM)": ("hbm", {"inc1.0": 512 * 512 * (4 + 32)}),
    "16/32-channel convs @512/@256 (HBM)": ("hbm", {"inc1.3": 512 * 512 * 64, "inc2.0": 512 * 512 * 64, "inc2.3": 512 * 512 * 32 + 256 * 256 * 32,
                                                    "down1.0": 256 * 256 * (32 + 64), "down1.3": 256 * 256 * 64 + 128 * 128 * 64}),
    "32/64-channel convs @128 (tensor)": ("tensor", {"down2.0": _conv_flops(32, 64, 128), "down2.3": _conv_flops(64, 64, 128),
                                                     "inc3.0": _conv_flops(64, 64, 128), "inc3.3": _conv_flops(64, 64, 128)}),
    "deep encoder / decoder convs @64..@16 (tensor)": ("tensor", {
        "down3.0": _conv_flops(64, 128, 64), "down3.3": _conv_flops(128, 128, 64), "down4.0": _conv_flops(128, 256, 32),
        "down4.3": _conv_flops(256, 256, 32), "down5.0": _conv_flops(256, 512, 16), "down5.3": _conv_flops(512, 512, 16),
        "up1.conv.0": _conv_flops(512, 256, 32), "up1.conv.3": _conv_flops(256, 256, 32), "up2.conv.0": _conv_flops(256, 128, 64),
        "up2.conv.3": _conv_flops(128, 128, 64)}),
    "up-sampling convs (tensor)": ("tensor", {"up1.up": _conv_flops(512, 256, 16), "up2.up": _conv_flops(256, 128, 32),
                                              "up3.up": _conv_flops(128, 64, 64)}),
    "mid U-Net 128->128 @128 (tensor)": ("tensor", {k: _conv_flops(128, 128, 128) for k in
                                                    ("up3.conv.0", "up3.conv.3", "dconv1.0", "dconv1.3", "dconv2.0", "dconv2.3")}),
    "8-head conv1 128->1024 @128 (tensor)": ("tensor", {"heads.conv1": _conv_flops(128, 1024, 128)}),
    "8-head conv2 1x1 (HBM)": ("hbm", {"heads.conv2": 128 * 128 * (1024 * 2 + (1 + 16 + 8 + 8 + 1 + 360 + 64 + 64) * 4)}),
}


def decode_bytes_per_image(n_atoms, n_bpeaks, n_brecs, hw=128 * 128):
    """Algorithmic bytes of the peak decoder per image (SURVEY.md section 8d): the two centre maps are read densely
    (2 x HW x 4 B); every other map is touched at peaks only, counted as the 32-byte sectors of the planar-8 fp32 layout:
    per atom peak type (14 ch = 2 sectors) + charge + H-count = 4 sectors and an 8-byte record; per bond-centre peak the 60
    omega logits = 8 sectors; per emitted bond record 6 bond-type sectors + 1 rho sector and a 12-byte record; 16 B of counts."""
    return 2 * hw * 4 + n_atoms * (4 * 32 + 8) + n_bpeaks * 8 * 32 + n_brecs * (7 * 32 + 12) + 16


def layer_class_report(layers_ms, B, pk, decode_bytes=None):
    """Fraction of the relevant measured roofline per layer class (north_star), from the live per-launch CUDA-event times."""
    out = {}
    classes = dict(LAYER_CLASSES)
    if decode_bytes is not None:
        classes["peak decode (HBM; latency-bound at this size)"] = ("hbm", {"decode": decode_bytes})
    for name, (kind, members) in classes.items():
        if not all(k in layers_ms for k in members):
            continue
        ms = sum(layers_ms[k] for k in members)
        work = sum(members.values()) * B
        if kind == "tensor":
            ach, peak, unit = work / (ms * 1e-3) / 1e12, pk["bf16_tflops_sustained"], "TFLOP/s"
        else:
            ach, peak, unit = work / (ms * 1e-3) / 1e9, pk["hbm_gbs"], "GB/s"
        out[name] = {"ms": ms, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak}
    return out


def ncu_traffic(pattern):
    """(bytes, file) = dram__bytes_read.sum + dram__bytes_write.sum of the FIRST kernel in the newest profiles/ summary matching
    ``pattern`` (written by tools/ncu_summary.py from an `ncu --set full` capture); (None, None) when there is none."""
    import glob
    import re
    files = glob.glob(os.path.join(ROOT, "profiles", pattern))
    if not files:
        return None, None

    def version(f):                                      # r02_..._v12 sorts after r01_..._v25 and after r02_..._v3
        m = re.search(r"r(\d+)_.*?(?:_v(\d+))?\.summary\.txt$", os.path.basename(f))
        return (int(m.group(1)), int(m.group(2) or 0)) if m else (0, 0)
    f = max(files, key=version)
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total, seen = 0.0, set()
    for line in open(f):
        parts = line.split()
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and parts[0] not in seen:
            seen.add(parts[0])
            total += float(parts[1]) * unit.get(parts[2], 1.0)
    return (total, os.path.relpath(f, ROOT)) if len(seen) == 2 else (None, None)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Summary of the samples received between host times t0 and t1 (the timed region). nvidia-smi needs a second or
        so to start, so the sampler is started before the warm-up; when the region is too short to contain a sample the
        samples taken under load right before it (the warm-up steps) are used and the summary says so."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for _, r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        window = "timed region"
        if t0 is not None:
            inside = [r for ts, r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit() and t0 <= ts <= t1 + 0.15]
            if inside:
                rows = inside
            else:
                rows = rows[-5:]
                window = "last samples before the end of the timed region (region shorter than the sampling period)"
        sm = [float(r[0]) for r in rows]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window": window}


def make_weights(seed=0):
    import synthdata                       # deterministic synthetic weights / inputs: not the oracle
    return synthdata.make_state_dict(seed=seed, variant="W1")


def make_images(seed, n, H=512, W=512):
    import synthdata
    return torch.from_numpy(synthdata.binary_images(seed, n, H, W, 0.05))


# ----------------------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_path(sd, imgs, calib):
    """The reference's path on the host: fp32 U-Net forward (oracle port of src/unet.py) + decode (img2smiles.py:62-193)."""
    from oracle import decode_ref, unet_ref
    with torch.no_grad():
        outs = unet_ref.forward(imgs, sd)
    outs = [o.numpy() for o in outs]
    for k, v in calib.items():
        outs[k] = outs[k] + np.float32(v)
    recs = []
    for j in range(imgs.shape[0]):
        a, b = decode_ref.decode_records([o[j] for o in outs], -1.0, "nms")
        recs.append(decode_ref.records_to_lists(a, b))
    return recs


def time_cpu(sd, calib, n_images, iters, warmup=1):
    torch.set_num_threads(os.cpu_count() or 1)
    imgs = make_images(100, n_images)
    for _ in range(warmup):
        cpu_path(sd, imgs, calib)
    t0 = time.perf_counter()
    for _ in range(iters):
        cpu_path(sd, imgs, calib)
    dt = time.perf_counter() - t0
    return n_images * iters / dt, dt / iters


def calibrate_offsets_cpu(sd):
    """Constant logit offsets for the centre / omega heads so that a random-init network yields a realistic number of
    peaks (~0.3 % of pixels above the -1 threshold); see DESIGN.md 'synthetic inputs'. CPU version for --impl reference."""
    from oracle import unet_ref
    with torch.no_grad():
        outs = unet_ref.forward(make_images(99, 1), sd)
    return {k: float(-1.0 - torch.quantile(outs[k].flatten(), 0.997)) for k in (0, 4, 7)}


def run_reference(args, rank, world):
    if rank != 0:
        return
    sd = make_weights()
    calib = calibrate_offsets_cpu(sd)
    n = 8                                        # BASELINE.json configs[0]: batch of 8 images = one bounded sample of the 256-image step
    torch.set_num_threads(os.cpu_count() or 1)
    imgs = make_images(100, n)
    # --steps / --warmup are honoured as given (about 1 s per 8-image step on 16 cores)
    warm = max(args.warmup, 0)
    for _ in range(warm):
        cpu_path(sd, imgs, calib)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_path(sd, imgs, calib)
    dt = time.perf_counter() - t0
    v = n * steps / dt
    cores = torch.get_num_threads()
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
           "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "ABC-Net v2 U-Net fwd + heat-map decode, 1x512x512 binary images, CPU fp32",
                      "sample": f"{n} images per step (bounded sample of the GPU arm's 256-image batch: the rate is per image, "
                                "the CPU path has no batch-size dependence beyond thread occupancy)", "images_per_step": n,
                      "steps_requested": args.steps, "warmup_requested": args.warmup},
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"{steps} x {n} images, oracle port of src/unet.py + img2smiles.py:62-193"},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(out)


# ----------------------------------------------------------------------------------------- GPU arm: training step
TRAIN_FLOPS_PER_IMAGE = 281.9e9    # SURVEY.md section 8d: fprop + dgrad + wgrad


def run_train(args, rank, world, dev):
    """BASELINE.json configs[3] / [4]: one training iteration = forward (batch-statistics BN, dropout 0.2) + the 8 fused
    losses + full backward + bucketed NCCL gradient all-reduce (world > 1, overlapped with backward) + Adam, at the
    reference's batch size (train.py:44: 64 per GPU), replayed as one CUDA graph. Inputs resident in HBM."""
    import torch.distributed as dist

    import abcnet_b200
    from abcnet_b200.ddp import GradBuckets
    import synthdata as synth
    B = args.train_batch
    torch.cuda.reset_peak_memory_stats()                 # `mem_gb` = the training leg's own peak, not the inference legs before it
    model = abcnet_b200.UNet(1, HEADS).to(dev)
    model.load_state_dict(make_weights())
    model.train()
    buckets = GradBuckets(list(model.parameters())) if world > 1 else None
    opt = abcnet_b200.make_optimizer(model, capturable=True)
    step = abcnet_b200.TrainStep(model, opt, class_weights=True, buckets=buckets, use_graph=True)
    x = make_images(2000 + rank, 8).repeat((B + 7) // 8, 1, 1, 1)[:B].contiguous().to(dev)
    tg = [torch.from_numpy(t).repeat(*([(B + 7) // 8] + [1] * (t.ndim - 1)))[:B].contiguous().to(dev)
          for t in synth.dense_targets(rank, 8, 128, 128)]
    from abcnet_b200 import _lib
    for _ in range(max(args.warmup, 3)):
        loss = step(x, tg)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(x, tg)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    if os.environ.get("ABCNET_BENCH_WATCHDOG"):
        print(f"[rank {rank}] run_train: timed {args.steps} steps, {ms / args.steps:.2f} ms each", file=sys.stderr, flush=True)
    v = world * B * args.steps / (ms * 1e-3)
    ddp = ddp_evidence(args, world, dev, model, opt, buckets, x, tg, ms / args.steps) if world > 1 else None
    return {"metric": "images_per_sec_train_step", "value": v, "unit": UNIT, "ms_per_step": ms / args.steps, "ddp": ddp,
            "batch_per_gpu": B, "scaling": "weak", "dtype": "bf16 activations / fp32 master weights, accumulators and gradients",
            "workload": "forward (train-mode BN, dropout) + 8 losses + backward + gradient all-reduce + Adam, 1x512x512 images, "
                        "dense targets resident in HBM (BASELINE configs[3]/[4])",
            "whole_step_tflops": TRAIN_FLOPS_PER_IMAGE * v / 1e12, "loss": float(loss.item()),
            "replay": "one CUDA graph per iteration (kernels counted at capture: %d)" % step.launches_per_step,
            "mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}


def ddp_evidence(args, world, dev, model, opt, buckets, x, tg, ms_on):
    """Evidence for the data-parallel exchange (multi_gpu_train2.py:89), measured inside the SCALE run itself:
      * known_gradients_mean_exact: every rank fills ALL its gradient buckets with rank-dependent known values through the same
        grad_ready() path the backward uses; the result must be the exact mean over ranks for every parameter element
        (DistributedDataParallel's averaging) -- exact because the values are small integers;
      * real step: bucketed + overlapped all-reduce vs ONE plain NCCL all-reduce of the locally computed gradients
        (relative error), and all replicas bit-identical afterwards;
      * ms_per_step with the exchange disabled (same graph otherwise) vs enabled = exposed communication time;
      * the all-reduce alone: time and bus bandwidth 2 (N - 1) / N * bytes / t for the 42.8 MB of gradients in their buckets."""
    import torch.distributed as dist

    import abcnet_b200
    rank = dist.get_rank()
    out = {}

    def mark(msg):
        if os.environ.get("ABCNET_BENCH_WATCHDOG"):
            print(f"[rank {rank}] ddp_evidence: {msg}", file=sys.stderr, flush=True)
    mark("start")
    # ---- known gradients
    params = buckets.params
    buckets.zero()
    torch.cuda.synchronize()
    for i, p in enumerate(params):
        p.grad.copy_(((torch.arange(p.numel(), device=dev) % 7) + 1).view_as(p).float() * (rank + 1) * ((i % 3) + 1))
        buckets.grad_ready(p)
    buckets.finish()
    torch.cuda.synchronize()
    mean_factor = (world + 1) / 2.0
    ok = True
    for i, p in enumerate(params):
        want = ((torch.arange(p.numel(), device=dev) % 7) + 1).view_as(p).float() * mean_factor * ((i % 3) + 1)
        ok = ok and bool(torch.equal(p.grad, want))
    t = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    out["known_gradients_mean_exact"] = bool(t.item() == 1.0)
    mark("known gradients done")
    # ---- real gradients: bucketed / overlapped vs one plain all-reduce of the local gradients
    step_noopt = abcnet_b200.TrainStep(model, None, class_weights=True, buckets=buckets, use_graph=False)
    p_drop, model.dropout_p = model.dropout_p, 0.0      # the two evaluations below must see the same function (new masks every step)
    buckets.comm_enabled = False
    step_noopt(x, tg)
    torch.cuda.synchronize()
    local = torch.cat([b.clone() for b in buckets.buckets])
    dist.all_reduce(local)
    local /= world
    buckets.comm_enabled = True
    step_noopt(x, tg)
    torch.cuda.synchronize()
    model.dropout_p = p_drop
    got = torch.cat(buckets.buckets)
    # weight gradients use fp32 atomics: two evaluations of the same step differ in the last bits, hence a tolerance
    rel = ((got - local).norm() / (local.norm() + 1e-30)).item()
    chk = torch.stack([got.double().sum(), got.double().abs().sum()])
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    out["bucketed_vs_plain_allreduce_rel_err"] = rel
    out["replicas_bit_identical"] = bool(torch.equal(lo, hi))
    out["correct"] = bool(out["known_gradients_mean_exact"] and rel < 1e-3 and out["replicas_bit_identical"])
    mark("real gradients done")
    # ---- the exchange alone
    nbytes = sum(b.numel() for b in buckets.buckets) * 4
    for _ in range(3):
        for b in buckets.buckets:
            dist.all_reduce(b)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        for b in buckets.buckets:
            dist.all_reduce(b)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ar_ms = t.item()
    out.update(allreduce_alone_ms=ar_ms, allreduce_bytes=nbytes, n_buckets=len(buckets.buckets),
               allreduce_bus_gbs=2.0 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9)
    mark("exchange alone done")
    # ---- the same step with the exchange switched off (new capture)
    buckets.comm_enabled = False
    step_off = abcnet_b200.TrainStep(model, opt, class_weights=True, buckets=buckets, use_graph=True)
    for _ in range(3):
        step_off(x, tg)
    torch.cuda.synchronize()
    dist.barrier()
    e0.record()
    for _ in range(args.steps):
        step_off(x, tg)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    buckets.comm_enabled = True
    out.update(ms_per_step_comm_off=t.item(), ms_per_step_comm_on=ms_on, exposed_comm_ms=ms_on - t.item(),
               nccl={k: os.environ[k] for k in os.environ if k.startswith("NCCL_")})
    return out


def run_small_batches(model, pool, dev, args):
    """The reference's own inference batch sizes (img2smiles.py:39: 32 images; BASELINE configs[0]: 8): per-batch latency and
    throughput of forward + decode, (a) eager = ~47 launches enqueued one by one through the C-ABI, (b) the same work replayed
    as ONE CUDA graph (abcnet_b200.InferGraph), (c) end to end with a pinned uint8 host batch: H2D + graph + D2H of the records
    + stream sync, i.e. what a caller waits for."""
    import abcnet_b200
    res = {}
    for b in (8, 32):
        hx = (pool[:b] > 0).to(torch.uint8).contiguous().pin_memory()
        dx = hx.to(dev)
        g = abcnet_b200.InferGraph(model, b, hx.shape[2], hx.shape[3], atom_cap=args.atom_cap, bond_cap=args.bond_cap, dtype=torch.uint8)
        g(dx)                                            # capture
        outs = None
        dec = g.decoder
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 50

        def timed(fn):
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / iters

        def eager():
            nonlocal outs
            outs = model.infer(dx, outs, layout="p8f")
            dec.launch(outs)
        ms_eager = timed(eager)
        ms_graph = timed(lambda: g.launch(dx))
        t0 = time.perf_counter()
        for _ in range(iters):
            g(hx)                                        # H2D (pinned, async) + replay + D2H + sync: one caller-visible latency
        ms_e2e = (time.perf_counter() - t0) / iters * 1e3
        res[str(b)] = {"eager_ms": ms_eager, "graph_ms": ms_graph, "e2e_latency_ms": ms_e2e, "graph_images_per_s": b / (ms_graph * 1e-3),
                       "e2e_images_per_s": b / (ms_e2e * 1e-3), "launches_per_replay": g.launches_per_replay}
        del g
    return res


def run_comparator(args, dev, pool, B):
    """SURVEY.md section 8d config 2 / 4 comparator: the reference's graph through torch / cuDNN on this same GPU (tools/gpu_comparator.py)
    -- forward + the dense decode tensor ops at batch B, forward + losses + backward at the training batch size."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gpu_comparator

    import abcnet_b200
    import synthdata as synth
    m = abcnet_b200.UNet(1, HEADS).to(dev)
    m.load_state_dict(make_weights())
    xi = pool.repeat((B + 63) // 64, 1, 1, 1)[:B].contiguous().to(dev)
    Bt = args.train_batch
    xt = xi[:Bt].contiguous()
    tg = [torch.from_numpy(t).repeat(*([(Bt + 7) // 8] + [1] * (t.ndim - 1)))[:Bt].contiguous().to(dev)
          for t in synth.dense_targets(0, 8, 128, 128)]
    res = gpu_comparator.run(m, xi, xt, tg, iters=3, warmup=2)
    res["what"] = ("src/unet.py's graph executed by stock torch ops (cuDNN convolutions, ATen BatchNorm / pooling / losses, autograd) on "
                   "the same B200: infer = forward + dense decode tensor ops (img2smiles.py:62-80,115-124) at batch %d; train = forward + "
                   "8 losses + backward (no optimizer step) at batch %d; CUDA events, cudnn.benchmark on" % (B, Bt))
    return res


# ----------------------------------------------------------------------------------------- GPU arm
def dump_outputs(out_dir, outs, recs):
    """Write what one inference step hands its caller, as float32 .npy files (exact for every field below), so that two builds
    can be compared output for output on the same inputs:
      atoms.npy   [n, 6]  image, x, y, type, charge, hs of every decoded atom peak, in decoder order
      bonds.npy   [n, 6]  image, x, y, omega, type, rho of every decoded bond record, in decoder order
      counts.npy  [B, 3]  atom peaks, bond records and bond-centre peaks per image
      logit_positions.npy [DUMP_PIXELS, 3]  (image, y, x), drawn with a fixed seed (the dense maps are 8.4 GB at batch 256)
      logits_<head>.npy [DUMP_PIXELS, channels]  logits of every channel of the head at those positions"""
    os.makedirs(out_dir, exist_ok=True)

    def save(name, arr):
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    img_a = np.concatenate([np.full(len(ra), i) for i, (ra, _, _) in enumerate(recs)])
    img_b = np.concatenate([np.full(len(rb), i) for i, (_, rb, _) in enumerate(recs)])
    a = np.concatenate([ra for ra, _, _ in recs])
    b = np.concatenate([rb for _, rb, _ in recs])
    save("atoms", np.stack([img_a, a["x"], a["y"], a["type"], a["charge"], a["hs"]], -1).astype(np.float32))
    save("bonds", np.stack([img_b, b["x"], b["y"], b["omega"], b["type"], b["rho"]], -1).astype(np.float32))
    save("counts", np.array([(len(ra), len(rb), nbp) for ra, rb, nbp in recs], np.float32).reshape(-1, 3))
    B, H, W = outs[0].shape[0], outs[0].shape[2], outs[0].shape[3]
    rng = np.random.default_rng(0)
    pos = np.stack([rng.integers(0, n, DUMP_PIXELS) for n in (B, H, W)], -1)
    save("logit_positions", pos.astype(np.float32))
    n, y, x = (torch.from_numpy(pos[:, k:k + 1]).to(outs[0].device) for k in range(3))
    for name, t, h in zip(HEAD_NAMES, outs, HEADS):
        c = torch.arange(h, device=t.device)[None]
        v = t[n, c // 8, y, x, c % 8] if t.dim() == 5 else t[n, c, y, x]           # planar-8 [B, ceil(h/8), H, W, 8] or NCHW
        save("logits_" + name, v.float().cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist

    import abcnet_b200
    from abcnet_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.require_device()
    B = args.batch
    sd = make_weights()
    model = abcnet_b200.UNet(1, HEADS).to(dev).eval()
    model.load_state_dict(sd)
    # synthetic images: a pool of 64 distinct images tiled to the batch (generation of 256 x 512^2 takes a while on the host)
    pool = make_images(1000 + rank, 64)
    host_f32 = pool.repeat((B + 63) // 64, 1, 1, 1)[:B].contiguous()
    x = host_f32.to(dev)                                 # `value`: fp32 {0,1} images resident in HBM (the reference DataLoader's format)
    # e2e transport: the same binary images as uint8 in pinned host memory (utils.py:80-81 binarises before the float cast;
    # UNet.forward accepts uint8 / bool / fp32 and produces identical bits) -- 4x fewer PCIe bytes than fp32
    host = (host_f32 > 0).to(torch.uint8).pin_memory()
    del host_f32
    # calibrate constant offsets of the centre / omega heads for a realistic peak density, folded into the conv2 biases
    outs = model(x[:8].contiguous())
    torch.cuda.synchronize()
    calib = {}
    with torch.no_grad():
        for k in (0, 4, 7):
            off = -1.0 - torch.quantile(outs[k].flatten()[:4_000_000].float(), 0.997)
            model.out_modules[k].conv2.bias += off
            calib[k] = float(off)
    dec = abcnet_b200.PeakDecoder(B, atom_cap=args.atom_cap, bond_cap=args.bond_cap, device=dev)
    out_bufs = None

    def step_device():
        nonlocal out_bufs
        out_bufs = model.infer(x, out_bufs, layout="p8f")
        if model.timing is not None:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dec.launch(out_bufs)
            b.record()
            model.timing.append(("decode", a, b))
        else:
            dec.launch(out_bufs)

    sampler = ClockSampler(local_rank)
    sampler.start()                                      # before the warm-up: nvidia-smi takes a moment to deliver its first row
    for _ in range(max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    counts = dec.fetch(B)
    n_atoms = float(np.mean([len(a) for a, _, _ in counts]))
    n_bonds = float(np.mean([len(b) for _, b, _ in counts]))
    n_bpeaks = float(np.mean([c for _, _, c in counts]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed: device-resident inputs
    model.timing = []                                    # (name, start_event, end_event) per launch, filled by the model
    barrier()
    t_host0 = time.time()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    barrier()
    launches = _lib.launch_count() - l0
    clocks = sampler.stop(t_host0, time.time())
    ms = e0.elapsed_time(e1)
    timing, model.timing = model.timing, None
    if args.dump_outputs and rank == 0:                  # the last timed step's logits and records, before other legs reuse the buffers
        dump_outputs(args.dump_outputs, out_bufs, dec.fetch(B))
    # ---- timed: end to end through the public API with HOST buffers. Every step copies its own images host -> device
    # (pinned memory, side stream, double-buffered so that the copy of step i+1 overlaps the kernels of step i) and reads
    # the decoded records back (one D2H + stream sync per step).
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    xbuf = [torch.empty(host.shape, dtype=torch.uint8, device=dev), torch.empty(host.shape, dtype=torch.uint8, device=dev)]
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def enqueue_copy(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            xbuf[i % 2].copy_(host, non_blocking=True)
            copied[i % 2].record(copy_stream)

    dec2 = [dec, abcnet_b200.PeakDecoder(B, atom_cap=args.atom_cap, bond_cap=args.bond_cap, device=dev)]
    obufs = [out_bufs, None]

    mol_threads = max(1, (os.cpu_count() or 1) // world)          # host assembler threads per rank (the ranks share the host cores)

    def run_e2e(steps, mol=False, pipes=None):
        """Every step: H2D of its own images (side stream, double-buffered), forward, decode, D2H of the records; the host
        collects the records of step i - 1 (waiting on that step's event only) after it has enqueued step i.
        mol=True: the host additionally assembles every image's records into MOL-block text (native assembler).
        pipes: two SparseHeadsPipeline objects -> the opt-in sparse-heads path instead of dense heads + PeakDecoder."""
        sink = pipes if pipes is not None else dec2
        for ev in consumed:
            ev.record(main_stream)
        enqueue_copy(0)
        recs = None
        for i in range(steps):
            if i + 1 < steps:
                enqueue_copy(i + 1)
            main_stream.wait_event(copied[i % 2])
            if pipes is not None:
                n = pipes[i % 2].launch(xbuf[i % 2])
                consumed[i % 2].record(main_stream)
            else:
                obufs[i % 2] = model.infer(xbuf[i % 2], obufs[i % 2], layout="p8f")
                consumed[i % 2].record(main_stream)
                n = dec2[i % 2].launch(obufs[i % 2])
            sink[i % 2].fetch_async(n)
            if i > 0:
                if mol:                                  # records stay in the pinned buffers; the assembler reads them there
                    sink[(i - 1) % 2].wait(n)
                    sink[(i - 1) % 2].molblocks(n, mol_threads)
                else:
                    recs = sink[(i - 1) % 2].collect(n)
        if mol:
            sink[(steps - 1) % 2].wait(B)
            return sink[(steps - 1) % 2].molblocks(B, mol_threads)
        return sink[(steps - 1) % 2].collect(B)

    run_e2e(2)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    recs = run_e2e(args.steps)
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    d2h = int(sum(a.nbytes + b.nbytes for a, b, _ in recs) + 16 * B)
    # same loop + native host assembly of the records into MOL-block text (SURVEY section 8f N1), and the assembler alone
    barrier()
    t0.record()
    texts = run_e2e(args.steps, mol=True)
    t1.record()
    barrier()
    ms_mol = t0.elapsed_time(t1)
    th0 = time.perf_counter()
    for _ in range(3):
        dec2[(args.steps - 1) % 2].molblocks(B, n_threads=1)
    asm_rate = 3 * B / (time.perf_counter() - th0)
    # opt-in sparse-heads path (SURVEY section 8f N4): class / offset heads evaluated at the peaks only, identical records
    pipe = abcnet_b200.SparseHeadsPipeline(model, B, peak_cap=128, bond_cap=args.bond_cap, device=dev)
    for _ in range(3):
        pipe.launch(x)
    barrier()
    l_sp = _lib.launch_count()
    t0.record()
    for _ in range(args.steps):
        pipe.launch(x)
    t1.record()
    barrier()
    ms_sp = t0.elapsed_time(t1)
    l_sp = (_lib.launch_count() - l_sp) // args.steps
    sp_error, ms_sp_e2e = None, None
    try:
        got_sp = pipe.fetch(B)                           # raises if an image has more than peak_cap peaks
        step_device()
        want_sp = dec.fetch(B)
        sp_equal = all(wn == gn and np.array_equal(wa, ga) and np.array_equal(wb, gb)
                       for (wa, wb, wn), (ga, gb, gn) in zip(want_sp, got_sp))
        # the same path end to end with host buffers (H2D of the images, D2H of the records, MOL-block text on the host)
        pipes = [pipe, abcnet_b200.SparseHeadsPipeline(model, B, peak_cap=128, bond_cap=args.bond_cap, device=dev)]
        run_e2e(2, mol=True, pipes=pipes)
        barrier()
        t0.record()
        run_e2e(args.steps, mol=True, pipes=pipes)
        t1.record()
        barrier()
        ms_sp_e2e = t0.elapsed_time(t1)
        del pipes
    except RuntimeError as e:                            # reported, never fatal for the headline numbers
        sp_equal, sp_error = False, str(e)[:200]
    del pipe
    if world > 1:
        t = torch.tensor([ms, ms_e2e, ms_mol, ms_sp, ms_sp_e2e if ms_sp_e2e is not None else 1e30], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_mol, ms_sp, ms_sp_e2e = t.tolist()
        ms_sp_e2e = None if ms_sp_e2e >= 1e29 else ms_sp_e2e
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    # the decision-stable inference mode: the same step with IEEE fp16 activations / weights (UNet(act_dtype="fp16")): same kernels,
    # same tensor-core rate, 8 x smaller rounding error per stored value (DESIGN.md section 2); NOT the headline, which stays bf16
    fp16_leg = None
    if not args.no_small:
        try:
            m16 = abcnet_b200.UNet(1, HEADS, act_dtype="fp16").to(dev).eval()
            m16.load_state_dict(model.state_dict())
            dec16 = abcnet_b200.PeakDecoder(B, atom_cap=args.atom_cap, bond_cap=args.bond_cap, device=dev)
            o16 = None
            for _ in range(3):
                o16 = m16.infer(x, o16, layout="p8f")
                dec16.launch(o16)
            torch.cuda.synchronize()
            t0.record()
            for _ in range(args.steps):
                o16 = m16.infer(x, o16, layout="p8f")
                dec16.launch(o16)
            t1.record()
            torch.cuda.synchronize()
            ms16 = t0.elapsed_time(t1) / args.steps
            ref_l = [o.float() for o in model.infer(x[:8].contiguous(), layout="nchw")]
            got_l = [o.float() for o in m16.infer(x[:8].contiguous(), layout="nchw")]
            fp16_leg = {"value_per_gpu": B / (ms16 * 1e-3), "unit": UNIT, "ms_per_step": ms16,
                        "rel_l2_vs_bf16_path": [float(((a - b).norm() / (b.norm() + 1e-30)).item()) for a, b in zip(got_l, ref_l)],
                        "what": "UNet(act_dtype='fp16') on this rank, device-resident inputs, dense heads + decode (opt-in precision mode)"}
            del m16, dec16, o16, ref_l, got_l
            torch.cuda.empty_cache()
        except Exception as e:                           # noqa: BLE001
            fp16_leg = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    small = None
    if not args.no_small:
        try:                                             # auxiliary legs never cost the headline line
            small = run_small_batches(model, pool, dev, args)
        except Exception as e:                           # noqa: BLE001
            small = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    # the same 256-image step replayed as ONE CUDA graph (SURVEY.md section 8d config 2: "graph-captured and eager both reported")
    graph_ms = None
    if not args.no_small and world == 1:                 # single-GPU configuration (configs[1]); no collective-style barriers inside the try
        try:
            g = abcnet_b200.InferGraph(model, B, x.shape[2], x.shape[3], atom_cap=args.atom_cap, bond_cap=args.bond_cap, dtype=x.dtype)
            for _ in range(3):
                g.launch(x)
            barrier()
            t0.record()
            for _ in range(args.steps):
                g.launch(x)
            t1.record()
            barrier()
            graph_ms = t0.elapsed_time(t1) / args.steps
            del g
        except Exception:                                # noqa: BLE001
            graph_ms = None
        torch.cuda.empty_cache()
    comparator = None
    train = None
    if not args.no_train:
        model._bufs.clear()
        model._packed = None
        out_bufs = xbuf = x = obufs = dec2 = dec = None      # the inference legs' buffers (2 x 8.4 GB of logits among them)
        torch.cuda.empty_cache()
        train = run_train(args, rank, world, dev)
    if world == 1 and not args.no_comparator:
        model._bufs.clear()
        model._packed = None
        out_bufs = xbuf = x = obufs = dec2 = None
        torch.cuda.empty_cache()
        try:
            comparator = run_comparator(args, dev, pool, B)
        except Exception as e:                           # noqa: BLE001
            comparator = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    if rank != 0:
        return
    pk, pk_src = peaks()
    # per-layer breakdown (CUDA events recorded around every launch inside the timed steps)
    agg = {}
    for name, a, b in timing:
        agg.setdefault(name, []).append(a.elapsed_time(b))
    layers = {k: float(np.mean(v)) for k, v in agg.items()}
    fused = "heads.fused" in layers
    dom = "heads.fused" if fused else "heads.conv1"
    dom_ms = layers.get(dom)
    roof = None
    if dom_ms:
        flops = (HEADS_CONV1_FLOPS_PER_IMAGE + (HEADS_CONV2_FLOPS_PER_IMAGE if fused else 0.0)) * B
        ach = flops / (dom_ms * 1e-3) / 1e12
        peak = pk["bf16_tflops_sustained"]
        traffic, traffic_src = (None, None) if (fused or B != 256) else ncu_traffic(HEADS_CONV1_SUMMARY_GLOB)
        roof = {"bound": "tensor",
                "kernel": "heads_fused_kernel[8 x (128->128 3x3 + LeakyReLU + 128->h 1x1) @128x128]" if fused
                else "conv_igemm_kernel[heads.conv1 128->1024 3x3 @128x128]", "achieved": ach,
                "peak": peak, "peak_source": pk_src + " (sustained bf16)", "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic,
                "traffic_unit": "bytes per launch (ncu dram read + write of the committed --set full capture under profiles/)",
                "traffic_source": traffic_src,
                "ms_per_launch": dom_ms, "flops_per_launch": flops}
    total_tflops = FLOPS_PER_IMAGE * B * args.steps / (ms * 1e-3) / 1e12
    cpu = None
    if not args.no_cpu:
        v, per = time_cpu(sd, calib, 8, 2)
        cpu = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
               "sample": "2 x 8 images (bounded sample of the 256-image batch), oracle port: fp32 U-Net + decode"}
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic",
           "config": {"workload": f"ABC-Net v2 U-Net fwd + fused peak decode, batch {B} x 1x512x512 per GPU (BASELINE configs[1])",
                      "batch_per_gpu": B, "weights": "random-init (deterministic), BN folded, centre/omega biases calibrated",
                      "l2": "inputs (268 MB / batch) and activations exceed the 126 MB L2; no explicit flush",
                      "avg_atom_peaks": n_atoms, "avg_bond_records": n_bonds, "avg_bond_centre_peaks": n_bpeaks,
                      "whole_forward_tflops": total_tflops, "layers_ms": layers,
                      "layer_classes": layer_class_report(layers, B, pk, decode_bytes_per_image(n_atoms, n_bpeaks, n_bonds))},
           "roofline": roof, "cpu_baseline": cpu,
           "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(host.numel() * host.element_size()), "d2h_bytes_per_step": d2h,
                   "ms_per_step": ms_e2e / args.steps, "input_format": "uint8 {0,1} [B,1,512,512] in pinned host memory"},
           "e2e_molblock": {"value": world * B * args.steps / (ms_mol * 1e-3), "unit": UNIT, "ms_per_step": ms_mol / args.steps,
                            "what": "e2e loop + native multi-threaded host assembly of every image's records into V2000 MOL-block "
                                    "text (abc_assemble_molblocks: img2smiles.py:183-318 + generate_smiles.py:18-105)",
                            "molecules_per_step": int(sum(t is not None for t in texts)),
                            "assembler_alone_images_per_s_1_thread": asm_rate},
           "sparse_heads": {"value": world * B * args.steps / (ms_sp * 1e-3), "unit": UNIT, "ms_per_step": ms_sp / args.steps,
                            "launches_per_step": int(l_sp), "records_identical_to_dense_path": bool(sp_equal), "peak_cap": 128, "error": sp_error,
                            "e2e_molblock_value": (world * B * args.steps / (ms_sp_e2e * 1e-3)) if ms_sp_e2e else None,
                            "what": "opt-in SparseHeadsPipeline, device-resident inputs: trunk + dense centre heads + peak search + "
                                    "class / offset heads at the peaks only (same kernels, same packed weights, same MMA order); "
                                    "NOT the headline `value`, which evaluates all eight heads densely"},
           "small_batch": small, "gpu_comparator": comparator, "fp16_activation_mode": fp16_leg,
           "graph_replay": None if graph_ms is None else {"ms_per_step": graph_ms, "value": world * B / (graph_ms * 1e-3), "unit": UNIT,
                                                           "what": "the device-resident step (`value` = eager launches) as one CUDA-graph replay"},
           "gpu_launches": int(launches), "clocks": clocks, "train": train}
    _emit(out)


_REAL_STDOUT = None


def _emit(obj):
    """The ONE JSON line, on the process's original stdout."""
    f = _REAL_STDOUT or sys.stdout
    f.write(json.dumps(obj) + "\n")
    f.flush()


def _reserve_stdout():
    """Keep a private handle on the original stdout and point file descriptor 1 at stderr: libraries that write to stdout from C
    (NCCL prints 'NCCL version ...' there at NCCL_DEBUG=VERSION / WARN) can then not put a second line next to the JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every headline leg (device-resident, e2e, MOL-block, sparse heads, fp16, graph replay, "
                         "training step, reference arm); the side measurements cpu_baseline (2 x 8 images), small_batch (50 "
                         "iterations per size), gpu_comparator (3 iterations) and, with several GPUs, the all-reduce alone "
                         "(20 repetitions) keep fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--atom-cap", type=int, default=1024)
    ap.add_argument("--bond-cap", type=int, default=4096)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg (the 'train' object)")
    ap.add_argument("--no-small", action="store_true", help="skip the batch-8 / batch-32 latency leg ('small_batch')")
    ap.add_argument("--no-comparator", action="store_true", help="skip the torch / cuDNN comparator leg ('gpu_comparator')")
    ap.add_argument("--train-batch", type=int, default=64, help="images per GPU per training step (train.py:44; multi_gpu_train2.py:20 uses 60)")
    ap.add_argument("--train-only", action="store_true", help="only the training-step leg: prints its object as the JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's decoded records and a fixed "
                    "sample of its logits to DIR/<name>.npy (rank 0's images). Inference path only: the reference arm decodes a "
                    "different 8-image sample with its own calibration, so its records are not comparable with these")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.train_only):
        ap.error("--dump-outputs writes the outputs of the inference path (--impl ours without --train-only)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("ABCNET_BENCH_WATCHDOG"):          # debugging aid: dump every thread's stack and exit if the run takes too long
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["ABCNET_BENCH_WATCHDOG"]), exit=True)
    if world > 1 or args.gpus == 1:
        _reserve_stdout()                                # (not in the convenience re-launch below: the children inherit fd 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line (NCCL prints its version there)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.train_only:
            torch.cuda.set_device(local_rank)
            out = run_train(args, rank, world, torch.device("cuda", local_rank))
            if rank == 0:
                out.update(n_gpus=world, steps=args.steps, higher_is_better=True)
                _emit(out)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
