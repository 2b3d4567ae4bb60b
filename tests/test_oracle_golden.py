"""Pin the CPU oracle against golden vectors minted from the reference itself
(tests/golden/make_golden.py, executed in the build container). CPU only."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import assemble_ref, decode_ref, detrand, loss_ref, synth, unet_ref


def test_param_inventory():
    shapes = unet_ref.param_shapes()
    assert len(shapes) == 261                                   # SURVEY.md section 1
    n = sum(int(np.prod(s)) for k, s in shapes.items()
            if not k.endswith(("running_mean", "running_var", "num_batches_tracked")))
    assert n == 10_698_575


def at_pixels(y, pos):
    """Every channel of the maps y [B, C, H, W] (numpy or torch) at the pixels pos [n, 3] = (image, y, x) -> [n, C]."""
    return y[pos[:, 0], :, pos[:, 1], pos[:, 2]]


def assert_matches_unet_golden(y, g, pos, key, i, tol):
    """Head i of y against a U-Net golden (tests/golden/make_golden.py reduce_logits): allclose(rtol = atol = tol) on every
    channel at the stored pixels pos, and on the sum and absolute sum of the whole map the bound that elementwise allclose
    implies."""
    y = y.numpy()
    np.testing.assert_allclose(at_pixels(y, pos), g[f"{key}{i}"], rtol=tol, atol=tol)
    abssum = float(g[f"{key}_abssum{i}"])
    bound = tol * (y.size + abssum)
    y64 = y.astype(np.float64)
    assert abs(y64.sum() - float(g[f"{key}_sum{i}"])) <= bound, (key, i)
    assert abs(np.abs(y64).sum() - abssum) <= bound, (key, i)


@pytest.mark.parametrize("tag,B,H,W,seed", [("small", 2, 64, 96, 3), ("tiny", 2, 32, 32, 4)])
def test_unet_oracle_matches_reference(golden_dir, tag, B, H, W, seed):
    g = np.load(os.path.join(golden_dir, "unet_small.npz"))
    sd = unet_ref.make_state_dict(seed=seed, variant="W1")
    x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08))
    with torch.no_grad():
        ys = unet_ref.forward(x, sd)
        yt = unet_ref.forward(x, sd, training=True)
    for i, (y, t) in enumerate(zip(ys, yt)):
        # same ATen kernels as the reference module -> agreement to fp32 round-off
        assert_matches_unet_golden(y, g, g[f"{tag}_pos"], f"{tag}_out", i, 1e-5)
        assert_matches_unet_golden(t, g, g[f"{tag}_pos"], f"{tag}_train_out", i, 1e-4)


def test_unet_oracle_matches_reference_three_channels(golden_dir):
    """UNet(in_channels=3) on real-valued input (the reference's own self-check configuration, unet.py:122-134): the oracle against
    logits of the reference module itself (tests/golden/make_golden.py unet_rgb)."""
    g = np.load(os.path.join(golden_dir, "unet_rgb.npz"))
    sd = unet_ref.make_state_dict(seed=9, in_channels=3, variant="W1")
    x = torch.from_numpy(synth.detrand.uniform(77, (1, 3, 96, 64), 0.0, 1.0).astype(np.float32))
    with torch.no_grad():
        ys = unet_ref.forward(x, sd)
        yt = unet_ref.forward(x, sd, training=True)
    assert [tuple(y.shape) for y in ys] == [(1, h, 24, 16) for h in unet_ref.V2_HEADS]
    for i, (y, t) in enumerate(zip(ys, yt)):
        assert_matches_unet_golden(y, g, g["pos"], "out", i, 1e-5)
        assert_matches_unet_golden(t, g, g["pos"], "train_out", i, 1e-4)


def test_unet_crop_side_is_first_row_col():
    """unet.py:51-55 under torch 2.x drops the FIRST row/column (SURVEY App. D1)."""
    sd = unet_ref.make_state_dict(seed=4)
    x = torch.from_numpy(synth.binary_images(4, 1, 32, 32, 0.08))
    with torch.no_grad():
        a = unet_ref.forward(x, sd, crop_first=True)[0]
        b = unet_ref.forward(x, sd, crop_first=False)[0]
    assert (a - b).abs().max() > 1e-4


def test_unet_full_resolution_samples(golden_dir):
    g = np.load(os.path.join(golden_dir, "unet_full_samples.npz"))
    sd = unet_ref.make_state_dict(seed=1, variant="W1")
    x = torch.from_numpy(synth.binary_images(1, 1, 512, 512, 0.05))
    with torch.no_grad():
        ys = unet_ref.forward(x, sd)
    r = detrand.integers(detrand.key("samplepos", 1), (256, 2), 0, 1 << 30)
    px, py = r[:, 0] % 128, r[:, 1] % 128
    for i, y in enumerate(ys):
        np.testing.assert_allclose(y[0][:, px, py].numpy(), g[f"samples{i}"], rtol=1e-4, atol=1e-4)
        assert abs(y.double().sum().item() - float(g[f"sum{i}"])) <= 1e-4 * float(g[f"abssum{i}"]) + 1e-3


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("mode,suffix", [("nms", ""), ("raw", "_raw")])
def test_decode_oracle_matches_reference(golden_dir, seed, mode, suffix):
    g = json.load(open(os.path.join(golden_dir, "decode_cases.json")))[f"planted{seed}{suffix}"]
    outs, _ = synth.planted_logits(seed)
    atoms, bonds = decode_ref.decode_records(outs, -1.0, mode)
    L = decode_ref.records_to_lists(atoms, bonds)
    for k in ("bonds_position_list", "bonds_property_list", "bonds_delta_list", "atoms_position_list",
              "atoms_charge_list", "atoms_hs_list"):
        assert L[k] == g[k], k            # bit-exact, including the float64 deltas
    r = assemble_ref.assemble(L)
    assert r[0] == g["atoms_type_list_final"]
    assert [[int(a), int(b)] for a, b in r[1]] == g["bond2atom_index_final"]
    assert r[2] == g["atoms_charge_list_final"]
    assert r[3] == g["bonds_property_list_final"]
    assert r[5] == g["atom_implicit_hs_list"]
    assert assemble_ref.molblock(*r) == g["molblock"]


def test_decode_empty_image(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "decode_cases.json")))["no_atoms"]
    outs, _ = synth.planted_logits(7, n_atoms=0, n_bonds=5, edge_cases=False)
    na, nb = decode_ref.count_peaks(outs)
    assert na == 0 and nb > 0 and g["molblock"] is None         # img2smiles.py:126-129


@pytest.mark.parametrize("key,cw", [("train", True), ("train2", False)])
def test_loss_oracle_matches_reference(golden_dir, key, cw):
    g = json.load(open(os.path.join(golden_dir, "loss_cases.json")))[key]
    gg = np.load(os.path.join(golden_dir, "loss_grads.npz"))
    tg = [torch.from_numpy(t) for t in synth.dense_targets(5, 1, 128, 128)]
    outs = [torch.from_numpy(o).requires_grad_(True) for o in synth.random_logits(5, 1, 128, 128)]
    s = torch.from_numpy(detrand.normalish(detrand.key("s", 5), (10,), 0.3)).requires_grad_(True)
    total, wl, _ = loss_ref.losses(outs, tg, s, class_weights=cw)
    assert str(total.dtype) == g["loss_dtype"] == "torch.float64"     # SURVEY App. C.2
    assert abs(total.item() - g["loss"]) <= 1e-9 * abs(g["loss"])
    for n, v in g["parts"].items():
        assert abs(wl[n].item() - v) <= 1e-6 * abs(v) + 1e-9, n
    total.backward()
    np.testing.assert_allclose(s.grad.numpy(), np.array(g["ds"], np.float32), rtol=1e-5, atol=1e-6)
    ix, iy = gg["ix"], gg["iy"]
    for i, o in enumerate(outs):
        np.testing.assert_allclose(o.grad[0][:, ix, iy].numpy(), gg[f"{key}_g{i}"], rtol=1e-5, atol=1e-9)
        assert abs(o.grad.double().abs().sum().item() - g["grad_abssum"][i]) <= 1e-5 * g["grad_abssum"][i]
    # the fp64 evaluation (truth for the CUDA kernel) agrees with the mixed-precision reference closely
    t64, _, _ = loss_ref.losses([o.detach() for o in outs], tg, s.detach(), class_weights=cw,
                                compute_dtype=torch.float64)
    assert abs(t64.item() - g["loss"]) <= 1e-5 * abs(g["loss"])


TARGET_NAMES = ("atom_target", "atom_type", "atom_charge", "atom_hs", "bond_target", "bond_type", "bond_rho", "bond_omega_type")


def target_cases(golden_dir):
    """(case index, label strings, (scale_x, scale_y, ddx, ddy), {name: dense array}) from tests/golden/target_cases.npz."""
    from oracle import targets_ref
    g = np.load(os.path.join(golden_dir, "target_cases.npz"))
    for i, (seed, sx, sy, ddx, ddy) in enumerate(g["cases"].tolist()):
        sx, sy = (int(sx) if sx == 1 else sx), (int(sy) if sy == 1 else sy)
        dense = {}
        for name in TARGET_NAMES:
            arr = np.zeros(int(np.prod(g[f"c{i}_{name}_shape"])), g[f"c{i}_{name}_val"].dtype)
            arr[g[f"c{i}_{name}_idx"]] = g[f"c{i}_{name}_val"]
            dense[name] = arr.reshape(tuple(g[f"c{i}_{name}_shape"]))
        yield i, targets_ref.label_strings(int(seed)), (sx, sy, int(ddx), int(ddy)), dense


def test_target_rasteriser_oracle_matches_reference(golden_dir):
    """oracle/targets_ref.py vs the maps produced by the reference's own statements (utils.py:83-228), all eight target
    arrays, values and dtypes (float64 rho / omega), bit-exact."""
    from oracle import targets_ref
    n = 0
    for i, (a, b), aug, dense in target_cases(golden_dir):
        for name, arr in zip(TARGET_NAMES, targets_ref.rasterise(a, b, *aug)):
            assert arr.dtype == dense[name].dtype and arr.shape == dense[name].shape, (i, name)
            assert np.array_equal(arr, dense[name]), (i, name)
        n += 1
    assert n == 12
