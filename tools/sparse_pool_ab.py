"""A/B of the two slot layouts of SparseHeadsPipeline on the benchmark's workload, plus one crowded batch.

    python tools/sparse_pool_ab.py OUT_DIR [--steps 50] [--rounds 3]

Weights, images and the centre / omega calibration are those of bench.py (256 images of 512 x 512, seeded synthetic
weights, offsets at the 0.997 quantile). The fixed layout (peak_cap=128) and the pooled layout with the same number of slots
(peak_pool = 2 * 256 * 128) alternate `rounds` times; each arm's time is CUDA events around `steps` launches after a
warm-up. Their records must be identical to each other and to the dense path. Then image 2 of the batch gets an amplified
input, enough for more than 1024 bond-centre peaks if the scales reach that: the fixed layout must reject that batch and the
pooled one must decode it exactly as UNet.infer + PeakDecoder do. Writes OUT_DIR/sparse_pool_ab.json with the card's name,
power limit and SM clocks read in the same run.
"""
from __future__ import annotations

import argparse
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

HEADS = [1, 14, 3, 2, 1, 360, 60, 60]
CROWDED = 2


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr[:200]}


def same(want, got):
    return len(want) == len(got) and all(wn == gn and np.array_equal(wa, ga) and np.array_equal(wb, gb)
                                         for (wa, wb, wn), (ga, gb, gn) in zip(want, got))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    model = abcnet_b200.UNet(1, HEADS).to(dev).eval()
    model.load_state_dict(synthdata.make_state_dict(seed=0, variant="W1"))
    pool = torch.from_numpy(synthdata.binary_images(1000, 64, 512, 512, 0.05))
    x = pool.repeat((B + 63) // 64, 1, 1, 1)[:B].contiguous().to(dev)
    outs = model(x[:8].contiguous())
    with torch.no_grad():
        for k in (0, 4, 7):
            model.out_modules[k].conv2.bias += -1.0 - torch.quantile(outs[k].flatten()[:4_000_000].float(), 0.997)
    del outs

    dense = abcnet_b200.PeakDecoder(B, atom_cap=1024, bond_cap=4096, device=dev)
    want = dense(model.infer(x, layout="p8f"))
    counts = dense.h_counts[:B].numpy().copy()
    cap = 128
    arms = {"fixed": abcnet_b200.SparseHeadsPipeline(model, B, peak_cap=cap, bond_cap=4096, device=dev),
            "pooled": abcnet_b200.SparseHeadsPipeline(model, B, bond_cap=4096, device=dev, peak_pool=2 * B * cap)}
    recs, ms = {}, {k: [] for k in arms}
    for name, pipe in arms.items():
        recs[name] = pipe.fetch(pipe.launch(x))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for name, pipe in arms.items():
            for _ in range(3):
                pipe.launch(x)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                pipe.launch(x)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / args.steps)
    last = {name: pipe.fetch(B) for name, pipe in arms.items()}
    identical = same(recs["fixed"], recs["pooled"]) and same(last["fixed"], last["pooled"])
    equal_dense = same(want, recs["fixed"]) and same(want, recs["pooled"])
    del arms

    # crowded batch: one image with an amplified input
    big = abcnet_b200.PeakDecoder(B, atom_cap=128 * 128, bond_cap=1 << 16, device=dev)
    for scale in (1.5, 2, 3, 4, 6, 8, 12, 16, 24, 32):
        xc = x.clone()
        xc[CROWDED] *= scale
        want_c = big(model.infer(xc, layout="p8f"))
        cc = big.h_counts[:B].numpy().copy()
        if cc[CROWDED, 2] > 1024:
            break
    total = int(cc[:, 0].sum() + cc[:, 2].sum())
    fixed = abcnet_b200.SparseHeadsPipeline(model, B, peak_cap=cap, bond_cap=1 << 16, device=dev)
    try:
        fixed.fetch(fixed.launch(xc))
        fixed_error = None
    except RuntimeError as e:
        fixed_error = str(e)[:200]
    del fixed
    pooled = abcnet_b200.SparseHeadsPipeline(model, B, bond_cap=1 << 16, device=dev, peak_pool=2 * B * cap, atom_cap=128 * 128)
    crowd_err, crowd_equal = None, False
    try:
        crowd_equal = same(want_c, pooled.fetch(pooled.launch(xc)))
    except RuntimeError as e:
        crowd_err = str(e)[:200]

    res = {
        "gpu": smi(),
        "workload": {"batch": B, "image": [512, 512], "weights": "bench.py: synthdata seed 0, centre / omega offsets at the 0.997 quantile",
                     "steps_per_arm_round": args.steps, "rounds": args.rounds},
        "mean_peaks_per_image": {"atoms": float(counts[:, 0].mean()), "bond_centres": float(counts[:, 2].mean()),
                                 "max_atoms": int(counts[:, 0].max()), "max_bond_centres": int(counts[:, 2].max())},
        "ms_per_step": {"fixed_peak_cap_128": ms["fixed"], "pooled_peak_pool_%d" % (2 * B * cap): ms["pooled"]},
        "median_ms": {k: float(np.median(v)) for k, v in ms.items()},
        "records_identical_fixed_vs_pooled": bool(identical),
        "records_identical_to_dense_path": bool(equal_dense),
        "crowded_batch": {"scale": scale, "crowded_image_atoms": int(cc[CROWDED, 0]), "crowded_image_bond_centres": int(cc[CROWDED, 2]),
                          "batch_total_peaks": total, "pool_slots": 2 * B * cap, "average_share_per_image": 2 * cap,
                          "fixed_layout_error": fixed_error, "pooled_error": crowd_err,
                          "pooled_records_identical_to_dense_path": bool(crowd_equal)},
    }
    res["gpu_after"] = smi()
    with open(os.path.join(args.out_dir, "sparse_pool_ab.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    ok = identical and equal_dense and fixed_error is not None and crowd_equal
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
