"""Per-CTA timeline of the fused output-heads kernel on the benchmark's shape.

    python tools/heads_trace.py OUT.json [--batch 256] [--launches 5] [--warmup 5] [--fp16]

Weights and images are those of bench.py (make_weights(), 256 images of 512 x 512, p8f logits). After a warm-up of the
whole inference step, the trunk is run once and abc_heads_fused is launched `launches` times with a trace buffer: each CTA
records its head pair, its tile count, %globaltimer at start and end, and the clock64 cycles its issuing warps and one
epilogue warp spent in each barrier wait (the HfTraceWord record of csrc/heads_fused_sm100.cu). The kernel time with the
trace off (CUDA events over the same number of launches) is measured as well, so the cost of tracing shows.

Per pair it prints and writes: CTAs, tiles per CTA, the mean and max end time (from the earliest CTA start of the launch),
and the mean cycles per CTA of every wait site, also as a share of the CTA's cycles. The card's name, power limit and SM
clocks are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import abcnet_b200  # noqa: E402
import synthdata  # noqa: E402
from abcnet_b200 import _lib  # noqa: E402

HEADS = [1, 14, 3, 2, 1, 360, 60, 60]
WORDS = ["pair", "tiles", "start_ns", "end_ns", "cycles",
         "c1_b_full", "c1_a_full", "c1_acc_empty",
         "c2_hid_full", "c2_c2_empty", "c2_w_full", "c2_w_empty",
         "ep_acc_full", "ep_phase1", "ep_c2_full", "ep_phase2"]
WAITS = WORDS[5:]


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr[:200]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("out")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--fp16", action="store_true", help="UNet(act_dtype='fp16') instead of bf16")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    model = abcnet_b200.UNet(1, HEADS, act_dtype="fp16" if args.fp16 else "bf16").to(dev).eval()
    model.load_state_dict(synthdata.make_state_dict(seed=0, variant="W1"))
    pool = torch.from_numpy(synthdata.binary_images(1000, 64, 512, 512, 0.05))
    x = pool.repeat((B + 63) // 64, 1, 1, 1)[:B].contiguous().to(dev)
    outs = None
    for _ in range(args.warmup):
        outs = model.infer(x, outs, layout="p8f", fused=True)
    with torch.no_grad():
        k2 = model.trunk(x)
    torch.cuda.synchronize()
    st = _lib.current_stream_ptr()
    d = model._heads_fused_desc(k2, outs)

    def launch():
        _lib.check(_lib.lib.abc_heads_fused(C.byref(d), st), "abc_heads_fused")

    # kernel time, trace off
    launch()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(args.launches):
        launch()
    ev[1].record()
    torch.cuda.synchronize()
    ms_plain = ev[0].elapsed_time(ev[1]) / args.launches

    max_ctas = max(_lib.lib.abc_sm_count(), 16)
    buf = torch.zeros((args.launches, max_ctas, len(WORDS)), dtype=torch.int64, device=dev)
    ev[0].record()
    for i in range(args.launches):
        d.trace = buf[i].data_ptr()
        launch()
    ev[1].record()
    torch.cuda.synchronize()
    ms_trace = ev[0].elapsed_time(ev[1]) / args.launches
    d.trace = None
    rec = buf.cpu().numpy()

    per_launch_end = []
    pairs = {}
    for li in range(args.launches):
        r = rec[li][rec[li][:, WORDS.index("end_ns")] != 0]
        t0 = r[:, WORDS.index("start_ns")].min()
        per_launch_end.append((r[:, WORDS.index("end_ns")].max() - t0) / 1e3)
        for row in r:
            pairs.setdefault(int(row[0]), []).append((row, (row[WORDS.index("end_ns")] - t0) / 1e3))
    report = {"device": smi(), "batch": B, "act_dtype": "fp16" if args.fp16 else "bf16", "launches": args.launches,
              "kernel_ms_trace_off": ms_plain, "kernel_ms_trace_on": ms_trace,
              "kernel_span_us_mean": float(np.mean(per_launch_end)), "pairs": {}}
    for pr in sorted(pairs):
        rows = np.stack([r for r, _ in pairs[pr]])
        ends = np.array([e for _, e in pairs[pr]])
        cyc = rows[:, WORDS.index("cycles")].astype(np.float64)
        ns = (rows[:, WORDS.index("end_ns")] - rows[:, WORDS.index("start_ns")]).astype(np.float64)
        waits = {w: float(rows[:, WORDS.index(w)].mean()) for w in WAITS}
        report["pairs"][str(pr)] = {
            "heads": HEADS[2 * pr:2 * pr + 2],
            "ctas": int(len(rows) // args.launches),
            "tiles_per_cta": [int(rows[:, 1].min()), int(rows[:, 1].max())],
            "end_us_mean": float(ends.mean()), "end_us_max": float(ends.max()),
            "cta_cycles_mean": float(cyc.mean()),
            "sm_mhz_mean": float((cyc / ns).mean() * 1e3),
            "wait_cycles_mean": waits,
            "wait_share_of_cta_cycles": {w: v / float(cyc.mean()) for w, v in waits.items()},
        }
    text = json.dumps(report, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
