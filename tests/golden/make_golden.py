#!/usr/bin/env python
"""Mint golden vectors FROM THE REFERENCE ITSELF (run in the build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz / *.json

The reference (/root/reference, read-only, absent on the GPU box) ships no tests, weights or
fixtures (SURVEY.md section 4), so the oracle is pinned against outputs of the reference's own code
executed here:

  * U-Net: ``src/unet.py`` is imported by path and run with deterministic weights
    (``oracle.unet_ref.make_state_dict``) on deterministic binary images.
  * decode + assembly + MOL text: the statements of ``src/img2smiles.py`` (lines 62-80 and
    105-320) -- and the ``img2smiles2.py`` variant -- are read from the reference file and
    exec'd in place on planted logit maps; ``generate_smiles.sdf2smiles`` is imported with stub
    ``rdkit`` / ``indigo`` modules whose MolFromMolBlock/MolToSmiles return the MOL-block text.
  * losses: ``src/train.py`` lines 95-137 (and ``multi_gpu_train2.py`` 140-192) are exec'd on
    deterministic logits / dense targets; gradients come from autograd on those statements.
  * dense training targets: ``src/utils.py`` lines 83-228 are exec'd on deterministic label strings.

No reference source is copied into the repository: slices are read at run time.
"""
from __future__ import annotations

import json
import os
import sys
import textwrap
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/src"
sys.path.insert(0, ROOT)

from oracle import detrand, synth, unet_ref  # noqa: E402


def ref_lines(fname, a, b):
    with open(os.path.join(REF, fname)) as f:
        lines = f.readlines()
    return textwrap.dedent("".join(lines[a - 1:b]))


def import_ref_unet():
    sys.path.insert(0, REF)
    from unet import UNet  # noqa
    sys.path.pop(0)
    return UNet


def sample_positions(seed, n, H, W):
    r = detrand.integers(detrand.key("samplepos", seed), (n, 2), 0, 1 << 30)
    return r[:, 0] % H, r[:, 1] % W


UNET_SAMPLE_PIXELS = 32             # pixels per output set kept in unet_small.npz / unet_rgb.npz: the files stay far below 1 MB


def pixel_sample(seed, B, H, W, n=UNET_SAMPLE_PIXELS):
    """n distinct (image, y, x) positions of a [B, *, H, W] output, sorted, as int64 [n, 3]."""
    r = np.sort(np.random.default_rng(seed).choice(B * H * W, n, replace=False))
    return np.stack(np.unravel_index(r, (B, H, W)), -1).astype(np.int64)


def reduce_logits(key, ys, pos):
    """What the golden keeps of the 8 head outputs ys [B, C, H, W]: every channel at the pixels pos ({key}{i}, [n, C]) and
    the float64 sum and absolute sum of the whole map ({key}_sum{i}, {key}_abssum{i})."""
    out = {}
    for i, y in enumerate(ys):
        y = np.asarray(y)
        y64 = y.astype(np.float64)
        out[f"{key}{i}"] = y[pos[:, 0], :, pos[:, 1], pos[:, 2]]
        out[f"{key}_sum{i}"] = np.array(y64.sum())
        out[f"{key}_abssum{i}"] = np.array(np.abs(y64).sum())
    return out


# ----------------------------------------------------------------------------- U-Net
def golden_unet():
    UNet = import_ref_unet()
    torch.manual_seed(0)
    out = {}
    for tag, (B, H, W, seed) in {"small": (2, 64, 96, 3), "tiny": (2, 32, 32, 4)}.items():
        sd = unet_ref.make_state_dict(seed=seed, variant="W1")
        m = UNet(in_channels=1, heads=list(unet_ref.V2_HEADS))
        m.load_state_dict(sd)
        m.eval()
        x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08))
        pos = out[f"{tag}_pos"] = pixel_sample(seed, B, H // 4, W // 4)
        with torch.no_grad():
            ys = m(x)
        out.update(reduce_logits(f"{tag}_out", ys, pos))
        # train-mode forward (BN batch statistics; dropout disabled by p=0 so it is deterministic)
        m.train()
        for om in m.out_modules:
            om.drop.p = 0.0
        with torch.no_grad():
            ys = m(x)
        out.update(reduce_logits(f"{tag}_train_out", ys, pos))
    np.savez_compressed(os.path.join(HERE, "unet_small.npz"), **out)

    # full resolution: samples + checksums only (dense output is 32.8 MB / image)
    sd = unet_ref.make_state_dict(seed=1, variant="W1")
    m = UNet(in_channels=1, heads=list(unet_ref.V2_HEADS))
    m.load_state_dict(sd)
    m.eval()
    x = torch.from_numpy(synth.binary_images(1, 1, 512, 512, 0.05))
    with torch.no_grad():
        ys = m(x)
    px, py = sample_positions(1, 256, 128, 128)
    full = {}
    for i, y in enumerate(ys):
        full[f"samples{i}"] = y[0][:, px, py].numpy()
        full[f"sum{i}"] = np.array(y.double().sum().item())
        full[f"abssum{i}"] = np.array(y.double().abs().sum().item())
    full["atom_map"] = ys[0][0, 0].numpy()
    full["bond_map"] = ys[4][0, 0].numpy()
    np.savez_compressed(os.path.join(HERE, "unet_full_samples.npz"), **full)
    print("unet goldens written")


def golden_unet_rgb():
    """UNet(in_channels=3) on real-valued input -- the configuration of the reference's own self-check (src/unet.py:122-134),
    at a size that keeps the fixture small. Eval and train-mode (dropout p = 0) logits."""
    UNet = import_ref_unet()
    B, H, W, seed = 1, 96, 64, 9
    sd = unet_ref.make_state_dict(seed=seed, in_channels=3, variant="W1")
    m = UNet(in_channels=3, heads=list(unet_ref.V2_HEADS))
    m.load_state_dict(sd)
    x = torch.from_numpy(detrand.uniform(77, (B, 3, H, W), 0.0, 1.0).astype(np.float32))       # torch.rand-like
    out = {}
    pos = out["pos"] = pixel_sample(seed, B, H // 4, W // 4)
    m.eval()
    with torch.no_grad():
        out.update(reduce_logits("out", m(x), pos))
    m.train()
    for om in m.out_modules:
        om.drop.p = 0.0
    with torch.no_grad():
        out.update(reduce_logits("train_out", m(x), pos))
    np.savez_compressed(os.path.join(HERE, "unet_rgb.npz"), **out)
    print("3-channel unet golden written")


# ----------------------------------------------------------------------------- decode
class _FakeChem:
    @staticmethod
    def MolFromSmiles(s):
        return s

    @staticmethod
    def MolToSmiles(mol, **kw):
        return mol

    @staticmethod
    def MolFromMolBlock(text):
        return text


def _stub_modules():
    rd = types.ModuleType("rdkit")
    rd.Chem = _FakeChem
    chem = types.ModuleType("rdkit.Chem")
    for k in ("MolFromSmiles", "MolToSmiles", "MolFromMolBlock"):
        setattr(chem, k, getattr(_FakeChem, k))
    ind = types.ModuleType("indigo")
    ind.Indigo = lambda: object()
    ind.IndigoObject = object
    inchi = types.ModuleType("indigo.inchi")
    inchi.IndigoInchi = lambda x: object()
    sys.modules.update({"rdkit": rd, "rdkit.Chem": chem, "indigo": ind, "indigo.inchi": inchi})


class _FakeDF:
    class _Loc:
        def __getitem__(self, k):
            return "C"
    loc = _Loc()


def run_reference_decode(outs, script="img2smiles.py"):
    """Execute the reference's decode + assembly statements on the logits of ONE image."""
    _stub_modules()
    sys.path.insert(0, REF)
    import generate_smiles  # noqa  (reference module, stubbed rdkit/indigo)
    sys.path.pop(0)
    from copy import deepcopy
    ns = dict(torch=torch, np=np, deepcopy=deepcopy, sdf2smiles=generate_smiles.sdf2smiles, Chem=_FakeChem,
              df=_FakeDF(), total_nums=0, results=[], device=torch.device("cpu"))
    exec(ref_lines("utils.py", 12, 16), ns)                     # vocabularies
    exec(ref_lines(script, 20, 34), ns)                         # devocabs, leaky_relu, max valence
    names = ["atom_targets_pred", "atom_types_pred", "atom_charges_pred", "atom_hs_pred",
             "bond_targets_pred", "bond_types_pred", "bond_rhos_pred", "bond_omega_types_pred"]
    for n, o in zip(names, outs):
        ns[n] = torch.from_numpy(np.asarray(o, np.float32))[None]
    ns["imgs"] = torch.zeros(1, 1, 8, 8)
    if script == "img2smiles.py":
        exec(ref_lines(script, 62, 80), ns)
        exec(ref_lines(script, 105, 320), ns)
    else:                                                        # img2smiles2.py: shifted by -1 / -3 lines
        exec(ref_lines(script, 61, 79), ns)
        exec(ref_lines(script, 104, 317), ns)
    res = ns["results"][0]
    rec = {"molblock": res}
    if res is not None or "bonds_position_list" in ns:
        for k in ("bonds_position_list", "bonds_property_list", "bonds_delta_list", "atoms_position_list",
                  "atoms_type_list", "atoms_charge_list", "atoms_hs_list"):
            v = ns.get(k)
            rec[k] = json.loads(json.dumps(v, default=lambda o: o.item() if hasattr(o, "item") else float(o)))
        for k in ("bond2atom_index_final", "bonds_property_list_final", "atoms_type_list_final",
                  "atoms_charge_list_final", "atom_implicit_hs_list"):
            v = ns.get(k)
            rec[k] = json.loads(json.dumps(v, default=lambda o: o.item() if hasattr(o, "item") else float(o)))
    return rec


def golden_decode():
    cases = {}
    for seed in range(4):
        outs, info = synth.planted_logits(seed)
        cases[f"planted{seed}"] = run_reference_decode(outs, "img2smiles.py")
        cases[f"planted{seed}_raw"] = run_reference_decode(outs, "img2smiles2.py")
    outs, _ = synth.planted_logits(7, n_atoms=0, n_bonds=5, edge_cases=False)
    cases["no_atoms"] = run_reference_decode(outs, "img2smiles.py")
    with open(os.path.join(HERE, "decode_cases.json"), "w") as f:
        json.dump(cases, f)
    print("decode goldens written:", {k: (None if v["molblock"] is None else len(v["molblock"])) for k, v in cases.items()})


# ----------------------------------------------------------------------------- losses
def run_reference_loss(outs, targets, s, script="train.py"):
    class _M:
        pass
    model = _M()
    model.module = _M()
    model.module.s = s
    names_p = ["atom_targets_pred", "atom_types_pred", "atom_charges_pred", "atom_hs_pred",
               "bond_targets_pred", "bond_types_pred", "bond_rhos_pred", "bond_omega_types_pred"]
    names_t = ["atom_targets", "atom_types", "atom_charges", "atom_hs", "bond_targets", "bond_types",
               "bond_rhos", "bond_omega_types"]
    ns = dict(torch=torch, model=model, device=torch.device("cpu"))
    exec(ref_lines("train.py", 16, 16), ns)                      # atom_type_weights
    for n, o in zip(names_p, outs):
        ns[n] = o
    for n, t in zip(names_t, targets):
        ns[n] = t
    if script == "train.py":
        exec(ref_lines("train.py", 95, 137), ns)
    else:
        exec(ref_lines("multi_gpu_train2.py", 140, 192), ns)
    return ns


def golden_loss():
    rec = {}
    B, H, W = 1, 128, 128          # the reference hard-codes view(-1, 6, 60, 128, 128)
    tg = synth.dense_targets(5, B, H, W)
    targets = [torch.from_numpy(t) for t in tg]
    s = torch.from_numpy(detrand.normalish(detrand.key("s", 5), (10,), 0.3)).requires_grad_(True)
    grads = {}
    for script in ("train.py", "multi_gpu_train2.py"):
        outs = [torch.from_numpy(o).requires_grad_(True) for o in synth.random_logits(5, B, H, W)]
        ns = run_reference_loss(outs, targets, s, script)
        loss = ns["loss"]
        s.grad = None
        loss.backward()
        key = "train" if script == "train.py" else "train2"
        rec[key] = {
            "loss": float(loss.item()), "loss_dtype": str(loss.dtype),
            "parts": {n: float(ns[n + "_loss"].item()) for n in
                      ("atom_targets", "bond_targets", "atom_types", "atom_charges", "bond_types", "bond_rhos",
                       "bond_omega_types", "atom_hs")},
            "ds": [float(v) for v in s.grad.tolist()],
            "grad_abssum": [float(o.grad.double().abs().sum().item()) for o in outs],
        }
        px, py = sample_positions(9, 64, H, W)
        # samples: all channels at 64 pixels, plus all channels at the first 64 target pixels
        tx, ty = np.nonzero(tg[0][0, 0] == 1)
        ix = np.concatenate([px, tx[:64]])
        iy = np.concatenate([py, ty[:64]])
        for i, o in enumerate(outs):
            grads[f"{key}_g{i}"] = o.grad[0][:, ix, iy].numpy()
        grads["ix"], grads["iy"] = ix, iy
    with open(os.path.join(HERE, "loss_cases.json"), "w") as f:
        json.dump(rec, f, indent=1)
    np.savez_compressed(os.path.join(HERE, "loss_grads.npz"), **grads)
    print("loss goldens written", rec["train"]["loss"], rec["train2"]["loss"])


# ----------------------------------------------------------------------------- dense training targets
TARGET_NAMES = ("atom_target", "atom_type", "atom_charge", "atom_hs", "bond_target", "bond_type", "bond_rho", "bond_omega_type")
TARGET_CASES = [(seed, sx, sy, ddx, ddy) for seed in range(4) for (sx, sy, ddx, ddy) in ((1, 1, 0, 0), (0.87, 1, 33, 0), (1, 0.93, 0, 17))]


def run_reference_rasteriser(atoms_string, bonds_string, scale_x, scale_y, ddx, ddy):
    """utils.py:83-228 (the body of MolDataset.__getitem__ after the image augmentation) exec'd on the given labels. The only
    shim: ``np.math`` (removed in numpy 2) is mapped to the ``math`` module the reference's ``np.math.atan`` resolved to."""
    import math

    class NPShim:
        def __getattr__(self, k):
            return getattr(np, k)
    shim = NPShim()
    shim.math = math
    ns = {"np": shim, "torch": torch}
    exec(ref_lines("utils.py", 11, 16), ns)                         # device, vocabularies
    ns.update(atoms_string=atoms_string, bonds_string=bonds_string, scale_x=scale_x, scale_y=scale_y, ddx=ddx, ddy=ddy)
    exec(ref_lines("utils.py", 83, 228), ns)
    return [ns[k] for k in TARGET_NAMES]


def golden_targets():
    from oracle import targets_ref
    out = {}
    for i, (seed, sx, sy, ddx, ddy) in enumerate(TARGET_CASES):
        a, b = targets_ref.label_strings(seed)
        for name, arr in zip(TARGET_NAMES, run_reference_rasteriser(a, b, sx, sy, ddx, ddy)):
            nz = np.flatnonzero(arr)                                  # the maps are > 99.9 % zeros: store the support only
            out[f"c{i}_{name}_idx"] = nz.astype(np.int32)
            out[f"c{i}_{name}_val"] = arr.reshape(-1)[nz]
            out[f"c{i}_{name}_shape"] = np.array(arr.shape, np.int32)
    out["cases"] = np.array(TARGET_CASES, np.float64)                 # (label seed, scale_x, scale_y, ddx, ddy) per case
    np.savez_compressed(os.path.join(HERE, "target_cases.npz"), **out)
    print("target goldens written", len(TARGET_CASES), "cases")


if __name__ == "__main__":
    which = sys.argv[1:] or ["unet", "unet_rgb", "decode", "loss", "targets"]
    torch.set_num_threads(os.cpu_count() or 1)
    if "unet" in which:
        golden_unet()
    if "unet_rgb" in which:
        golden_unet_rgb()
    if "decode" in which:
        golden_decode()
    if "loss" in which:
        golden_loss()
    if "targets" in which:
        golden_targets()
