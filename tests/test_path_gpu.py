"""GPU parity tests of the hot path proper: U-Net forward, heat-map decode, fused losses -- product path
(abcnet_b200, through the C-ABI) against the CPU oracle and the golden vectors minted from the reference."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import assemble_ref, decode_ref, detrand, loss_ref, synth, unet_ref
from test_oracle_golden import at_pixels

pytestmark = pytest.mark.gpu

HEADS = list(unet_ref.V2_HEADS)
# Logit tolerance of the bf16-activation / fp32-accumulate pipeline against the fp32 reference, per output map:
#   max-abs error <= MAX_ABS_FRAC * max|ref| + MAX_ABS_FLOOR   and   relative L2 error <= REL_L2
MAX_ABS_FRAC, MAX_ABS_FLOOR, REL_L2 = 0.04, 0.03, 0.02


def _model(seed, variant="W1"):
    import abcnet_b200
    sd = unet_ref.make_state_dict(seed=seed, variant=variant)
    m = abcnet_b200.UNet(1, HEADS).cuda().eval()
    m.load_state_dict(sd)
    return m, sd


def _check_logits(outs, refs, what):
    report = []
    for i, (o, r) in enumerate(zip(outs, refs)):
        o = o.detach().float().cpu()
        r = torch.as_tensor(r)
        assert o.shape == r.shape and o.is_contiguous()
        err = (o - r).abs().max().item()
        scale = r.abs().max().item()
        rel = ((o - r).norm() / (r.norm() + 1e-12)).item()
        report.append((i, err, scale, rel))
    print(what, " | ".join(f"h{i}: maxabs {e:.4f} (scale {s:.2f}) relL2 {r:.4f}" for i, e, s, r in report))
    for i, err, scale, rel in report:
        assert err <= MAX_ABS_FRAC * scale + MAX_ABS_FLOOR, f"{what} head {i}: max abs err {err} (scale {scale})"
        assert rel <= REL_L2, f"{what} head {i}: rel L2 {rel}"


@pytest.mark.parametrize("tag,B,H,W,seed", [("small", 2, 64, 96, 3), ("tiny", 2, 32, 32, 4)])
def test_unet_forward_vs_golden(golden_dir, tag, B, H, W, seed):
    g = np.load(os.path.join(golden_dir, "unet_small.npz"))
    m, _ = _model(seed)
    x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08)).cuda()
    outs = m(x)
    assert isinstance(outs, list) and len(outs) == 8
    pos = g[f"{tag}_pos"]                   # the golden keeps every channel at these pixels
    _check_logits([at_pixels(o, pos) for o in outs], [g[f"{tag}_out{i}"] for i in range(8)], f"golden[{tag}]")


def test_unet_layer_by_layer_vs_oracle():
    """Every intermediate activation against the oracle (localises a wrong layer)."""
    m, sd = _model(3)
    x = torch.from_numpy(synth.binary_images(3, 2, 64, 96, 0.08))
    acts = {}
    with torch.no_grad():
        unet_ref.forward(x, sd, acts=acts)
    m.infer(x.cuda(), fused=False)          # separate conv1 / conv2 launches: the hidden maps are materialised
    torch.cuda.synchronize()
    pairs = [("k2", "dconv2.double_conv.3"), ("cat3", None), ("h2", "down5.maxpool_conv.1.double_conv.3")]
    got = m.activation("k2").cpu()
    ref = acts["dconv2.double_conv.3"]
    rel = ((got - ref).norm() / ref.norm()).item()
    print("trunk relL2", rel)
    assert rel < 0.02
    got = m.activation("h2").cpu()
    ref = acts["down5.maxpool_conv.1.double_conv.3"]
    assert ((got - ref).norm() / ref.norm()).item() < 0.02
    cat3 = m.activation("cat3").cpu()
    ref = torch.cat([acts["inc3.double_conv.3"], acts["up3.up"]], 1)
    assert ((cat3 - ref).norm() / ref.norm()).item() < 0.02
    hid = m.activation("hid").cpu()
    ref = torch.cat([acts[f"out_modules.{i}.hidden"] for i in range(8)], 1)
    assert ((hid - ref).norm() / ref.norm()).item() < 0.02
    assert pairs


def test_unet_full_resolution_vs_golden_samples(golden_dir):
    g = np.load(os.path.join(golden_dir, "unet_full_samples.npz"))
    m, _ = _model(1)
    x = torch.from_numpy(synth.binary_images(1, 1, 512, 512, 0.05)).cuda()
    outs = m(x)
    r = detrand.integers(detrand.key("samplepos", 1), (256, 2), 0, 1 << 30)
    px, py = r[:, 0] % 128, r[:, 1] % 128
    _check_logits([o[0][:, px, py] for o in outs], [g[f"samples{i}"] for i in range(8)], "golden[full samples]")
    _check_logits([outs[0][0, 0], outs[4][0, 0]], [g["atom_map"], g["bond_map"]], "golden[centre maps]")


def test_unet_batch_invariance_and_module_prefix():
    """Eval-mode results do not depend on batch composition (image sharding is exact), and DataParallel-style
    'module.'-prefixed checkpoints load (train.py:435)."""
    import abcnet_b200
    m, sd = _model(2)
    x = torch.from_numpy(synth.binary_images(2, 3, 64, 64, 0.08)).cuda()
    full = [o.clone() for o in m(x)]
    one = m(x[1:2].contiguous())
    for a, b in zip(full, one):
        assert torch.equal(a[1:2], b)
    m2 = abcnet_b200.UNet(1, HEADS).cuda().eval()
    m2.load_state_dict({"module." + k: v for k, v in sd.items()})
    for a, b in zip(full, m2(x)):
        assert torch.equal(a, b)


def _recs_equal(got, ref_atoms, ref_bonds):
    atoms, bonds, _ = got
    ra, (rb_int, rb_rho) = ref_atoms, ref_bonds
    a = np.stack([atoms["x"], atoms["y"], atoms["type"], atoms["charge"], atoms["hs"]], -1).astype(np.int32).reshape(-1, 5)
    b = np.stack([bonds["x"], bonds["y"], bonds["omega"], bonds["type"]], -1).astype(np.int32).reshape(-1, 4)
    assert np.array_equal(a, ra), "atom records differ"
    assert np.array_equal(b, rb_int), "bond records differ"
    assert np.array_equal(bonds["rho"], rb_rho), "rho differs"        # bit-exact


@pytest.mark.parametrize("mode,suffix", [("nms", ""), ("raw", "_raw")])
def test_decode_planted_batch_bit_exact(golden_dir, mode, suffix):
    import abcnet_b200
    gold = json.load(open(os.path.join(golden_dir, "decode_cases.json")))
    planted = [synth.planted_logits(seed)[0] for seed in range(4)]
    maps = [torch.from_numpy(np.stack([p[i] for p in planted])).cuda() for i in range(8)]
    dec = abcnet_b200.PeakDecoder(4, atom_cap=256, bond_cap=4096)
    res = dec(maps, thr=-1.0, omega_mode=mode)
    for seed in range(4):
        ra, rb = decode_ref.decode_records(planted[seed], -1.0, mode)
        _recs_equal(res[seed], ra, rb)
        # ... and through the product adapter + host assembly down to the reference's own MOL-block text
        atoms, bonds, nbp = res[seed]
        L = abcnet_b200.records_to_lists(atoms, bonds, nbp)
        g = gold[f"planted{seed}{suffix}"]
        for k in ("bonds_position_list", "bonds_property_list", "bonds_delta_list", "atoms_position_list",
                  "atoms_charge_list", "atoms_hs_list"):
            assert L[k] == g[k], k
        assert assemble_ref.records_to_molblock(L) == g["molblock"]
    # the native host assembler on the decoder's own pinned buffers gives the reference's MOL-block text as well
    texts = dec.molblocks(4)
    assert texts == [gold[f"planted{seed}{suffix}"]["molblock"] for seed in range(4)]


def test_decode_probability_mode_matches_training_metric_rule():
    """SURVEY §8 a14: train.py:145-151 finds centre peaks on clamp(sigmoid(z), 1e-5, 1-1e-5) with `> 0.25` instead of on the
    logits with `> -1`. Differences that must show: logits in (-1.0986, -1] become peaks, and saturated neighbours
    (z = 15 next to z = 20: both clamp to 1-1e-5) tie into a plateau of two peaks."""
    import abcnet_b200
    planted = [synth.planted_logits(seed)[0] for seed in range(3)]
    planted = [[np.array(m, np.float32, copy=True) for m in p] for p in planted]
    planted[0][0][0, 60, 60:62] = (15.0, 20.0)          # saturated pair on the atom map
    planted[1][4][0, 90, 17] = -1.05                    # between logit(0.25) and -1 on the bond map
    planted[1][7][:, 90, 17] = -3.0
    planted[1][7][11, 90, 17] = 2.0
    maps = [torch.from_numpy(np.stack([p[i] for p in planted])).cuda() for i in range(8)]
    dec = abcnet_b200.PeakDecoder(3, atom_cap=256, bond_cap=4096)
    res_p = dec(maps, thr=0.25, apply_sigmoid=True, thr_omega=-1.0)
    res_z = dec(maps, thr=-1.0)
    for j in range(3):
        ra, rb = decode_ref.decode_records(planted[j], 0.25, "nms", apply_sigmoid=True, thr_omega=-1.0)
        _recs_equal(res_p[j], ra, rb)
        ra, rb = decode_ref.decode_records(planted[j], -1.0, "nms")
        _recs_equal(res_z[j], ra, rb)

    def has(rec, x, y):
        return bool(((rec["x"] == x) & (rec["y"] == y)).any())
    assert has(res_p[0][0], 60, 60) and has(res_p[0][0], 60, 61)
    assert not has(res_z[0][0], 60, 60) and has(res_z[0][0], 60, 61)
    assert has(res_p[1][1], 90, 17) and not has(res_z[1][1], 90, 17)


def test_decode_empty_and_capacity():
    import abcnet_b200
    outs, _ = synth.planted_logits(7, n_atoms=0, n_bonds=5, edge_cases=False)
    maps = [torch.from_numpy(o[None]).cuda() for o in outs]
    dec = abcnet_b200.PeakDecoder(1, atom_cap=64, bond_cap=64)
    atoms, bonds, nbp = dec(maps)[0]
    assert len(atoms) == 0 and nbp == 5
    assert abcnet_b200.records_to_lists(atoms, bonds, nbp) is None          # img2smiles.py:126-129
    dense = [torch.from_numpy(o[:1]).cuda() for o in synth.random_logits(11, 1)]
    with pytest.raises(RuntimeError, match="capacity"):
        dec(dense)
    with pytest.raises(ValueError):
        dec([m.cpu() for m in maps])                                           # no CPU fallback


def test_decode_dense_random_logits_bit_exact():
    """Worst case: thousands of peaks per map (random logits) -- ordering and compaction at scale."""
    import abcnet_b200
    logits = synth.random_logits(12, 2)
    maps = [torch.from_numpy(o).cuda() for o in logits]
    dec = abcnet_b200.PeakDecoder(2, atom_cap=4096, bond_cap=65536)
    res = dec(maps, thr=-1.0)
    for j in range(2):
        ra, rb = decode_ref.decode_records([o[j] for o in logits], -1.0, "nms")
        assert len(ra) > 500
        _recs_equal(res[j], ra, rb)


def test_decode_of_network_outputs_matches_oracle_decode():
    """decode(CUDA logits) by the kernel == decode(CUDA logits) by the oracle, at the real 128x128 map size."""
    import abcnet_b200
    m, _ = _model(1)
    x = torch.from_numpy(synth.binary_images(1, 2, 512, 512, 0.05)).cuda()
    outs = m(x)
    for k in (0, 4, 7):          # random-init logits sit below the -1 threshold: shift for a realistic peak density
        outs[k] += -1.0 - torch.quantile(outs[k].flatten()[:1_000_000], 0.995)
    dec = abcnet_b200.PeakDecoder(2, atom_cap=16384, bond_cap=262144)
    res = dec(outs)
    assert sum(len(a) for a, _, _ in res) > 10
    host = [o.cpu().numpy() for o in outs]
    for j in range(2):
        ra, rb = decode_ref.decode_records([h[j] for h in host], -1.0, "nms")
        _recs_equal(res[j], ra, rb)


@pytest.mark.parametrize("key,cw,f64", [("train", True, True), ("train2", False, True), ("train", True, False)])
def test_fused_loss_vs_reference(golden_dir, key, cw, f64):
    import abcnet_b200
    g = json.load(open(os.path.join(golden_dir, "loss_cases.json")))[key]
    gg = np.load(os.path.join(golden_dir, "loss_grads.npz"))
    tg = [torch.from_numpy(t) for t in synth.dense_targets(5, 1, 128, 128)]
    if not f64:
        tg = [t.float() for t in tg]
    logits = synth.random_logits(5, 1, 128, 128)
    outs = [torch.from_numpy(o).cuda().requires_grad_(True) for o in logits]
    s = torch.from_numpy(detrand.normalish(detrand.key("s", 5), (10,), 0.3)).cuda().requires_grad_(True)
    lossmod = abcnet_b200.HeatmapLoss(class_weights=cw)
    total = lossmod(outs, [t.cuda().contiguous() for t in tg], s)
    total.backward()
    # tolerance: fp32 per-element math, fp64 accumulation -> 1e-5 relative on the losses, 1e-4 on gradients
    assert total.dtype == torch.float64
    assert abs(total.item() - g["loss"]) <= 2e-5 * abs(g["loss"]), (total.item(), g["loss"])
    np.testing.assert_allclose(s.grad.cpu().numpy(), np.array(g["ds"], np.float32), rtol=1e-4, atol=1e-6)
    ix, iy = gg["ix"], gg["iy"]
    for i, o in enumerate(outs):
        got = o.grad[0][:, ix, iy].cpu().numpy()
        ref = gg[f"{key}_g{i}"]
        np.testing.assert_allclose(got, ref, rtol=2e-3, atol=1e-7 + 1e-4 * np.abs(ref).max())
        asum = o.grad.double().abs().sum().item()
        assert abs(asum - g["grad_abssum"][i]) <= 1e-3 * g["grad_abssum"][i]
    # against the fp64 oracle too
    t64, _, _ = loss_ref.losses([torch.from_numpy(o) for o in logits], tg, s.detach().cpu(), class_weights=cw,
                                compute_dtype=torch.float64)
    assert abs(total.item() - t64.item()) <= 2e-5 * abs(t64.item())


def test_planar_logits_layout_is_equivalent():
    """layout='p8f' (planar-8 fp32 maps, the fused inference+decode format) carries exactly the NCHW values, and the
    decoder returns identical records from either layout."""
    import abcnet_b200
    m, _ = _model(1)
    x = torch.from_numpy(synth.binary_images(5, 2, 512, 512, 0.05)).cuda()
    nchw = [o.clone() for o in m.infer(x, layout="nchw")]
    p8f = m.infer(x, layout="p8f")
    assert p8f[5].dim() == 5 and p8f[0].dim() == 4
    for a, b in zip(nchw, p8f.to_nchw()):
        assert torch.equal(a, b)
    # shift the centre / omega maps so that there are peaks to decode
    for k in (0, 4, 7):
        off = -1.0 - torch.quantile(nchw[k].flatten()[:1_000_000], 0.995)
        nchw[k] += off
        p8f[k] += off
    dec = abcnet_b200.PeakDecoder(2, atom_cap=16384, bond_cap=262144)
    r1 = dec(nchw)
    r2 = dec(p8f)
    assert sum(len(a) for a, _, _ in r1) > 10
    for (a1, b1, n1), (a2, b2, n2) in zip(r1, r2):
        assert n1 == n2 and np.array_equal(a1, a2) and np.array_equal(b1, b2)


@pytest.mark.parametrize("heads,B,H,W", [(HEADS, 3, 64, 96), (HEADS, 2, 32, 32), ([1, 21, 5, 1, 4, 2], 2, 64, 64), ([1, 14, 3], 1, 96, 32),
                                         (HEADS, 2, 512, 512)])
def test_fused_heads_match_separate_launches(heads, B, H, W):
    """abc_heads_fused (conv1 + LeakyReLU + conv2 in one kernel, hidden maps kept on chip) against the separate
    conv_igemm launches: same bf16 hidden values, same fp32 accumulation order over K -> identical logits; both output
    layouts; partial tiles; even / odd head counts (the head list is a constructor argument, unet.py:96-98)."""
    import abcnet_b200
    sd = unet_ref.make_state_dict(seed=9, heads=tuple(heads), variant="W1")
    m = abcnet_b200.UNet(1, list(heads)).cuda().eval()
    m.load_state_dict(sd)
    x = torch.from_numpy(synth.binary_images(9, B, H, W, 0.08)).cuda()
    sep = [o.clone() for o in m.infer(x, fused=False)]
    fus = m.infer(x, fused=True)
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(sep, fus)):
        assert a.shape == b.shape
        d = (a - b).abs().max().item()
        assert d <= 1e-5 * max(1.0, a.abs().max().item()), f"head {i}: fused vs separate differ by {d}"
    p8 = m.infer(x, layout="p8f", fused=True)
    for a, b in zip(sep, p8.to_nchw()):
        assert (a - b).abs().max().item() <= 1e-5 * max(1.0, a.abs().max().item())
    if tuple(heads) == tuple(HEADS) and H <= 96:
        with torch.no_grad():
            ref = unet_ref.forward(x.cpu(), sd)
        _check_logits(fus, ref, "fused heads vs oracle")
