#!/usr/bin/env python
"""Cost of the deterministic training step (torch.use_deterministic_algorithms(True)) against the default one.

    python tools/det_train_ab.py [--batch 64] [--size 512] [--rounds 3] [--steps 10] [--out DIR]

Alternates the two arms (one TrainStep each, CUDA-graph replays, fixed-order reductions vs atomics) for `rounds` rounds of
`steps` timed replays (CUDA events), then profiles one step of each arm with torch.profiler in a run of its own and reports
the kernels whose time changed, the workspace the deterministic arm allocated, and the card name and power limit read in
the same call. Writes det_train_ab.json to --out (default: the current directory)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import abcnet_b200  # noqa: E402
import synthdata as synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


def make_arm(B, S, det):
    torch.use_deterministic_algorithms(det)
    m = abcnet_b200.UNet(1, list(synth.V2_HEADS)).cuda()
    m.load_state_dict(synth.make_state_dict(0))
    m.train()
    x = torch.from_numpy(synth.binary_images(0, 8, S, S, 0.05)).repeat(B // 8, 1, 1, 1).cuda()
    tg = [torch.from_numpy(t).repeat(*([B // 8] + [1] * (t.ndim - 1))).cuda().contiguous() for t in synth.dense_targets(0, 8, S // 4, S // 4)]
    step = abcnet_b200.TrainStep(m, abcnet_b200.make_optimizer(m), class_weights=True)
    step(x, tg)                                            # capture (+ its two warm-up steps)
    torch.cuda.synchronize()
    return dict(model=m, step=step, x=x, tg=tg, det=det)


def run(arm, steps):
    torch.use_deterministic_algorithms(arm["det"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        arm["step"](arm["x"], arm["tg"])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_times(arm):
    from torch.profiler import ProfilerActivity, profile
    torch.use_deterministic_algorithms(arm["det"])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            arm["step"](arm["x"], arm["tg"])
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" or getattr(e, "self_device_time_total", 0) > 0:
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = e.self_cuda_time_total
            out[e.key] = (out.get(e.key, (0.0, 0))[0] + t / 3.0 / 1000.0, e.count // 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=".", help="directory for det_train_ab.json (default: the current directory)")
    a = ap.parse_args()
    arms = {"default": make_arm(a.batch, a.size, False), "deterministic": make_arm(a.batch, a.size, True)}
    ms = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, arm in arms.items():
            ms[k].append(run(arm, a.steps))
    kt = {k: kernel_times(arm) for k, arm in arms.items()}
    changed = {}
    for name in set(kt["default"]) | set(kt["deterministic"]):
        d0, d1 = kt["default"].get(name, (0.0, 0)), kt["deterministic"].get(name, (0.0, 0))
        if any(s in name for s in ("wgrad", "bn_stats", "bn_act_bwd_reduce", "nchw_to_p8_ex", "conv_c1", "loss_kernel", "det_reduce",
                                   "conv_igemm_kernel<1, true, false, false, true", "Memset")) or abs(d1[0] - d0[0]) > 0.05:
            changed[name] = {"default_ms": round(d0[0], 4), "default_calls": d0[1], "det_ms": round(d1[0], 4), "det_calls": d1[1]}
    ws = arms["deterministic"]["model"]._train_engine().bufs.get("det:ws")
    res = {
        "card": card(), "batch": a.batch, "size": a.size, "rounds": a.rounds, "steps_per_round": a.steps,
        "ms_per_step": {k: [round(v, 3) for v in vs] for k, vs in ms.items()},
        "ms_per_step_median": {k: sorted(vs)[len(vs) // 2] for k, vs in ms.items()},
        "det_overhead_pct": round(100.0 * (sorted(ms["deterministic"])[a.rounds // 2] / sorted(ms["default"])[a.rounds // 2] - 1.0), 2),
        "det_workspace_bytes": int(ws.numel()) if ws is not None else 0,
        "kernels_per_step_ms": dict(sorted(changed.items(), key=lambda kv: -max(kv[1]["default_ms"], kv[1]["det_ms"]))),
    }
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "det_train_ab.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "kernels_per_step_ms"}))


if __name__ == "__main__":
    main()
