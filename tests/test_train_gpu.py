"""GPU parity of the training-mode U-Net pass (forward with batch statistics + full backward) against the CPU oracle
(torch autograd on oracle/unet_ref.py, fp32). Tolerance: bf16 activations and gradients through ~35 layers ->
relative L2 error per parameter gradient <= 6e-2 (weights) and logits within the eval tolerances."""
import os

import numpy as np
import pytest
import torch

from oracle import synth, unet_ref
from test_oracle_golden import at_pixels

pytestmark = pytest.mark.gpu
HEADS = list(unet_ref.V2_HEADS)


def _setup(seed, B, H, W):
    import abcnet_b200
    sd = unet_ref.make_state_dict(seed=seed, variant="W1")
    m = abcnet_b200.UNet(1, HEADS).cuda()
    m.load_state_dict(sd)
    m.train()
    m.dropout_p = 0.0
    x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08))
    return m, sd, x


def _p8_to_nchw(t, off=0, c=None):
    N, P, H, W, _ = t.shape
    x = t.float().permute(0, 1, 4, 2, 3).reshape(N, P * 8, H, W).cpu()
    return x[:, off * 8: off * 8 + (c if c is not None else P * 8 - off * 8)]


def _rel(got, ref):
    return ((got.double() - ref.double()).norm() / (ref.double().norm() + 1e-30)).item()


def _bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def _ste(t):
    return t + (_bf(t) - t).detach()


def test_train_step_in_situ_layer_parity():
    """Every layer of the real network, forward AND backward, checked in place: the CUDA layer's outputs (activation, pooled
    activation, dz-derived parameter gradients, gradient handed to the previous layer) are compared with an fp64 autograd
    evaluation of the SAME single layer fed with the CUDA path's own inputs (its input activation and the gradient buffers
    produced by the layers after it), with bf16 rounding at the CUDA path's storage points.

    Why not end-to-end against the unrounded oracle: in train mode a randomly initialised net amplifies perturbations ~370x
    from the first layer to the trunk (oracle fp32 vs fp64: 5e-8 -> 2e-5; BatchNorm removes the DC part of the signal, not
    of the noise), so 1-ulp bf16 differences saturate. The first three layers agree bit-exactly with the bf16-emulating
    oracle; the end-to-end figures are printed for the record."""
    import torch.nn.functional as F
    B, H, W, seed = 2, 64, 64, 5
    m, sd, x = _setup(seed, B, H, W)
    m.fuse_bn = False          # this test reads the dA buffers; with the fused reduction they hold dA * act' (checked separately below)
    outs = m(x.cuda())
    R = [torch.from_numpy(synth.detrand.uniform(100 + i, tuple(o.shape), -1, 1)) for i, o in enumerate(outs)]
    sum((o * r.cuda()).sum() for o, r in zip(outs, R)).backward()
    torch.cuda.synchronize()
    eng = m._engine
    bufs = eng.bufs
    grads = {n: p.grad.detach().cpu() for n, p in m.named_parameters() if p.grad is not None}
    names = {id(p): n for n, p in m.named_parameters()}
    report = []

    def get(ref, cin=None, grad=False, off=0):
        kind, key = ref
        t = bufs[("g:" if grad else "") + f"{kind}:{key}"]
        return _p8_to_nchw(t, off, cin)

    # ---- end-to-end vs the bf16-emulating oracle (reported; early layers must be exact)
    acts = {}
    with torch.no_grad():
        ro = unet_ref.forward(x, sd, training=True, acts=acts, emulate_bf16=True)
    e2e = [(k, _rel(_p8_to_nchw(bufs["a:" + k]), acts[rk])) for k, rk in
           (("inc1.0", "inc1.double_conv.0"), ("inc1.3", "inc1.double_conv.3"), ("inc2.0", "inc2.double_conv.0"),
            ("down2.3", "down2.maxpool_conv.1.double_conv.3"), ("dconv2.3", "dconv2.double_conv.3"))]
    print("end-to-end forward rel L2 vs emulated oracle:", [(k, round(v, 5)) for k, v in e2e],
          "logits:", [round(_rel(o.detach().cpu(), r), 4) for o, r in zip(outs, ro)])
    assert e2e[0][1] < 1e-4 and e2e[1][1] < 1e-3 and e2e[2][1] < 2e-3

    # ---- per-unit in-situ checks
    for u in eng.saved["plan"]:
        h, w = u["hw"]
        if "up" in u:
            xin = get(u["src"], u["cin"]).double().requires_grad_(True)
            wt = _bf(u["up"].weight.detach().float().cpu()).double().requires_grad_(True)
            bt = u["up"].bias.detach().cpu().double().requires_grad_(True)
            U = F.conv_transpose2d(xin, wt, bt, stride=2)
            kept = U[:, :, 1:, 1:]
            got_u = get(u["dst"], u["cout"], off=u["dst_off"])
            report.append((u["name"] + ".fwd", _rel(got_u, _bf(kept.detach().float()))))
            du = get(u["dst"], u["cout"], grad=True, off=u["dst_off"]).double()
            (kept * du).sum().backward()
            report.append((u["name"] + ".dx", _rel(get(u["src"], u["cin"], grad=True), xin.grad)))
            report.append((u["name"] + ".dw", _rel(grads[names[id(u["up"].weight)]], wt.grad)))
            report.append((u["name"] + ".db", _rel(grads[names[id(u["up"].bias)]], bt.grad)))
            continue
        cout, cin = u["cout"], u["cin"]
        first = bool(u.get("first"))
        a_in = (x if first else get(u["src"], cin, off=u["src_off"])).double().requires_grad_(not first)
        wt = u["conv"].weight.detach().float().cpu()
        wt = (wt if first else _bf(wt)).double().requires_grad_(True)
        bt = u["conv"].bias.detach().cpu().double()
        gam = u["bn"].weight.detach().cpu().double().requires_grad_(True)
        bet = u["bn"].bias.detach().cpu().double().requires_grad_(True)
        z = _ste(F.conv2d(a_in, wt, bt, padding=1))
        a = _ste(F.relu(F.batch_norm(z, None, None, gam, bet, True, 0.1, 1e-5)))
        loss = 0.0
        has_full = u["keep"] or u["dst"][0] == "cat"
        if has_full:
            report.append((u["name"] + ".fwd", _rel(get(u["dst"], cout, off=u["dst_off"]), a.detach())))
            loss = loss + (a * get(u["dst"], cout, grad=True, off=u["dst_off"]).double()).sum()
        if u["pool"]:
            pooled = F.max_pool2d(a, 2)
            report.append((u["name"] + ".pool", _rel(get(u["pool"]), pooled.detach())))
            loss = loss + (pooled * get(u["pool"], grad=True).double()).sum()
        loss.backward()
        report.append((u["name"] + ".dw", _rel(grads[names[id(u["conv"].weight)]], wt.grad)))
        report.append((u["name"] + ".dgamma", _rel(grads[names[id(u["bn"].weight)]], gam.grad)))
        report.append((u["name"] + ".dbeta", _rel(grads[names[id(u["bn"].bias)]], bet.grad)))
        assert grads[names[id(u["conv"].bias)]].abs().max().item() == 0.0        # bias before a train-mode BN: zero gradient
        if not first:
            report.append((u["name"] + ".dx", _rel(get(u["src"], cin, grad=True, off=u["src_off"]), a_in.grad)))

    # ---- heads (fused conv1 x8 -> BN -> LeakyReLU -> conv2), gradient wrt the trunk and all head parameters
    trunk = get(("a", "dconv2.3")).double().requires_grad_(True)
    loss = 0.0
    hp = []
    for i, om in enumerate(m.out_modules):
        w1 = _bf(om.conv1.weight.detach().float().cpu()).double().requires_grad_(True)
        gam = om.bn.weight.detach().cpu().double().requires_grad_(True)
        bet = om.bn.bias.detach().cpu().double().requires_grad_(True)
        w2 = _bf(om.conv2.weight.detach().float().cpu()).double().requires_grad_(True)
        b2 = om.conv2.bias.detach().cpu().double().requires_grad_(True)
        zh = _ste(F.conv2d(trunk, w1, om.conv1.bias.detach().cpu().double(), padding=1))
        hid = _ste(F.leaky_relu(F.batch_norm(zh, None, None, gam, bet, True, 0.1, 1e-5), 0.01))
        logit = F.conv2d(hid, w2, b2)
        report.append((f"head{i}.logits", _rel(outs[i].detach().cpu(), logit.detach())))
        loss = loss + (logit * R[i].double()).sum()
        hp.append((om, w1, gam, bet, w2, b2))
    loss.backward()
    report.append(("heads.dtrunk", _rel(get(("a", "dconv2.3"), grad=True), trunk.grad)))
    for i, (om, w1, gam, bet, w2, b2) in enumerate(hp):
        for nm, p, g in (("conv1.w", om.conv1.weight, w1.grad), ("bn.g", om.bn.weight, gam.grad), ("bn.b", om.bn.bias, bet.grad),
                         ("conv2.w", om.conv2.weight, w2.grad), ("conv2.b", om.conv2.bias, b2.grad)):
            report.append((f"head{i}.{nm}", _rel(grads[names[id(p)]], g)))

    report.sort(key=lambda kv: -kv[1])
    print("in-situ rel L2 (worst 12):", [(k, round(v, 4)) for k, v in report[:12]])
    for k, v in report:
        # forward tensors: bf16 ulp flips only; gradients: bf16 storage of dA / dz (2^-9 per element, partly coherent)
        tol = 5e-3 if (k.endswith(".fwd") or k.endswith(".pool") or k.endswith(".logits")) else 3e-2
        assert v <= tol, (k, v)


def test_dropout_is_consistent_between_forward_and_backward():
    m, sd, x = _setup(6, 2, 32, 32)
    m.dropout_p = 0.2
    outs = m(x.cuda())
    hid = m._engine.bufs["a:hid"].float()
    keep = (hid != 0).float().mean().item()
    assert 0.70 < keep < 0.90, keep                      # ~80 % kept (LeakyReLU output is never exactly 0 otherwise)
    sum(o.sum() for o in outs).backward()
    assert all(torch.isfinite(p.grad).all() for n, p in m.named_parameters() if n != "s")


def _targets(seed, B, h, w):
    return [torch.from_numpy(t).cuda().contiguous() for t in synth.dense_targets(seed, B, h, w)]


def test_train_step_matches_autograd_path_and_graph_replays(monkeypatch):
    """abcnet_b200.TrainStep (no autograd; eager and CUDA-graph replay) against model(x) + HeatmapLoss + loss.backward():
    same loss, same gradients, and after two optimiser steps the same loss / running statistics. With the fp32 head-gradient maps
    (ABCNET_LOSS_FP32=1) both paths round the same values, so only the fp32 atomics of the wgrad kernels differ (1e-3); the
    default TrainStep path (the loss writes bf16 P8 operands itself) is held to the bf16-storage bound. Dropout off so that all
    runs see the same function."""
    import abcnet_b200
    B, H, W, seed = 2, 64, 64, 11
    tg = None
    results = {}
    for mode in ("autograd", "eager", "graph", "eager-fp32-grad"):
        monkeypatch.delenv("ABCNET_LOSS_FP32", raising=False)
        if mode == "eager-fp32-grad":                      # fp32 gradient maps + conversion pass: the roundings of the autograd path
            monkeypatch.setenv("ABCNET_LOSS_FP32", "1")
        m, sd, x = _setup(seed, B, H, W)
        xg = x.cuda()
        tg = tg or _targets(seed, B, H // 4, W // 4)
        if mode == "autograd":
            opt = torch.optim.Adam(m.parameters(), lr=2.5e-4, weight_decay=1e-8)
            crit = abcnet_b200.HeatmapLoss(class_weights=True)
            losses = []
            for it in range(2):
                opt.zero_grad(set_to_none=True)
                loss = crit(m(xg), tg, m.s)
                loss.backward()
                if it == 0:
                    g0 = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
                opt.step()
                losses.append(loss.item())
        else:
            opt = abcnet_b200.make_optimizer(m, capturable=mode == "graph")
            step = abcnet_b200.TrainStep(m, opt, class_weights=True, use_graph=mode == "graph")
            losses = []
            for it in range(2):
                losses.append(step(xg, tg).item())
                if it == 0:
                    torch.cuda.synchronize()
                    g0 = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
        torch.cuda.synchronize()
        results[mode] = (losses, g0, {n: p.detach().clone() for n, p in m.named_parameters()},
                         {n: b.detach().clone() for n, b in m.named_buffers()})
    la, ga, pa, ba = results["autograd"]
    l, g, p, b = results["eager-fp32-grad"]                # same storage roundings as autograd: fp32 atomics are the only difference
    assert abs(l[0] - la[0]) <= 1e-6 * abs(la[0]) and abs(l[1] - la[1]) <= 2e-3 * abs(la[1]), (l, la)
    for n in ga:
        assert _rel(g[n], ga[n]) <= 1e-3 or ga[n].abs().max().item() == 0.0, (n, _rel(g[n], ga[n]))
    for n in ba:                                                                   # running statistics: exactly two updates
        assert _rel(b[n].float(), ba[n].float()) <= 1e-2, n                    # 2nd update sees a (noise-amplified) step-2 forward
    for mode in ("eager", "graph"):
        l, g, p, b = results[mode]
        assert abs(l[0] - la[0]) <= 1e-6 * abs(la[0]), (mode, l, la)
        # The default TrainStep path rounds the UNSCALED head gradient to bf16 and applies the per-loss factor afterwards
        # (abc_loss_partials_p8 + AbcBnActBwdDesc.gscale; both verified exactly in test_train_ops_gpu.py), the autograd path rounds the
        # scaled one. From the heads down every bf16 storage point then rounds slightly different fp32 values in the two runs, and a
        # randomly initialised train-mode net amplifies such 1-ulp differences by orders of magnitude (see the in-situ test above):
        # measured 1.4e-2 over all gradients (L2), 2.1e-2 on the worst single parameter (the bias of an up-convolution that feeds a
        # BatchNorm: a cancellation-dominated sum), 2.5e-3 on the step-2 loss. The bounds below are sanity bounds against a wrong
        # factor or a mixed-up head (those give O(1) errors); the tight comparison is the fp32-gradient mode above.
        names = [n for n in ga if ga[n].abs().max().item() != 0.0]
        worst = max((_rel(g[n], ga[n]), n) for n in names)
        assert worst[0] <= 1e-1, (mode, worst)
        flat, flat_a = torch.cat([g[n].flatten().double() for n in names]), torch.cat([ga[n].flatten().double() for n in names])
        assert _rel(flat, flat_a) <= 5e-2, (mode, _rel(flat, flat_a))
        assert abs(l[1] - la[1]) <= 1e-2 * abs(la[1]), (mode, l, la)             # after one (sign-like) Adam step
        for n in ba:                                                               # running statistics: exactly two updates
            assert _rel(b[n].float(), ba[n].float()) <= 5e-2, (mode, n, _rel(b[n].float(), ba[n].float()))
        assert int(b["inc1.double_conv.1.num_batches_tracked"]) == 2


def test_pack_arena_equals_torch_repack(monkeypatch):
    """The per-iteration gather (PackArena, one abc_gather_pack per dtype) feeds the convolutions the same packed weights as
    re-packing with torch ops (ABCNET_NO_ARENA=1): logits equal up to the rounding of the fp64-atomic BatchNorm sums, and
    the arena tracks in-place parameter updates (optimiser steps) without being rebuilt."""
    B, H, W, seed = 2, 64, 64, 13
    outs = {}
    for mode in ("arena", "torch"):
        if mode == "torch":
            monkeypatch.setenv("ABCNET_NO_ARENA", "1")
        else:
            monkeypatch.delenv("ABCNET_NO_ARENA", raising=False)
        m, sd, x = _setup(seed, B, H, W)
        res = []
        for it in range(2):
            o = m(x.cuda())
            res.append([t.detach().clone() for t in o])
            sum((t * t).sum() for t in o).backward()
            with torch.no_grad():                                    # in-place update between the two forwards
                for p in m.parameters():
                    p.mul_(1.01)
        eng = m._engine
        assert (eng.arena is not None) == (mode == "arena")
        if mode == "arena":
            assert eng.arena.used["w"] > 15_000_000 and len(eng._packs) > 60
        outs[mode] = (res, {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None})
    for it in range(2):
        for a, b in zip(outs["arena"][0][it], outs["torch"][0][it]):
            assert _rel(a, b) <= 1e-6, (it, _rel(a, b))
    for n, ga in outs["arena"][1].items():
        gb = outs["torch"][1][n]
        assert _rel(ga, gb) <= 1e-3 or gb.abs().max().item() == 0.0, (n, _rel(ga, gb))


@pytest.mark.parametrize("tag,B,H,W,seed", [("small", 2, 64, 96, 3), ("tiny", 2, 32, 32, 4)])
def test_train_forward_against_reference_minted_golden(tag, B, H, W, seed):
    """Train-mode forward (batch-statistics BatchNorm, dropout off) of the CUDA path against the logits minted by the
    reference's own module in train() mode (tests/golden/make_golden.py -> unet_small.npz:*_train_out*; VERDICT r01 weak #3).

    With B = 2 and 64 x 96 / 32 x 32 inputs the deepest BatchNorms normalise over 12 / 2 samples, which amplifies any
    perturbation by orders of magnitude (oracle fp32 vs fp64 already differ by 2e-5 at the trunk), so bf16 storage noise
    cannot vanish end to end. The yardstick is therefore the fp32 oracle with bf16 rounding injected at the CUDA path's
    storage points (unet_ref.forward(emulate_bf16=True)) measured against the SAME golden: the CUDA path may not be further
    from the reference than 3x that emulation + 2 %. The first head (atom centre) error is printed for the record."""
    import numpy as np
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "unet_small.npz"))
    m, sd, x = _setup(seed, B, H, W)
    with torch.no_grad():
        ours = [o.float().cpu() for o in m(x.cuda())]
        emu = unet_ref.forward(x, sd, training=True, emulate_bf16=True)
        exact = unet_ref.forward(x, sd, training=True)
    rows = []
    pos = g[f"{tag}_pos"]                                   # the golden keeps every channel at these pixels
    for i in range(8):
        ref = torch.from_numpy(g[f"{tag}_train_out{i}"])
        assert _rel(at_pixels(exact[i], pos), ref) < 1e-3, "oracle drifted from its golden"
        r_ours, r_emu = _rel(at_pixels(ours[i], pos), ref), _rel(at_pixels(emu[i], pos), ref)
        rows.append((i, round(r_ours, 4), round(r_emu, 4)))
        assert r_ours <= 3.0 * r_emu + 0.02, f"head {i}: CUDA train forward rel L2 {r_ours} vs bf16-emulated oracle {r_emu}"
    print(f"train-mode forward vs reference-minted golden ({tag}): (head, ours, bf16-emulated oracle) = {rows}")


def test_three_channel_stem_forward_and_weight_gradient():
    """UNet(in_channels=3) (the reference's own self-check, unet.py:122-134) on real-valued input: eval logits against the
    oracle, and in train mode the stem's activation / weight gradient / BN gradients in situ against fp64 autograd."""
    import torch.nn.functional as F
    import abcnet_b200
    B, H, W, seed = 2, 64, 64, 9
    sd = unet_ref.make_state_dict(seed=seed, in_channels=3, variant="W1")
    m = abcnet_b200.UNet(3, HEADS).cuda()
    m.load_state_dict(sd)
    x = torch.from_numpy(synth.detrand.uniform(77, (B, 3, H, W), -1.0, 1.0).astype(np.float32))
    m.eval()
    outs = [o.float().cpu() for o in m(x.cuda())]
    with torch.no_grad():
        ref = unet_ref.forward(x, sd)
    for i, (o, r) in enumerate(zip(outs, ref)):
        err, scale = (o - r).abs().max().item(), r.abs().max().item()
        assert err <= 0.04 * scale + 0.03, f"head {i}: max abs err {err} vs scale {scale}"
    m.train()
    m.dropout_p = 0.0
    outs = m(x.cuda())
    R = [torch.from_numpy(synth.detrand.uniform(200 + i, tuple(o.shape), -1, 1)) for i, o in enumerate(outs)]
    sum((o * r.cuda()).sum() for o, r in zip(outs, R)).backward()
    torch.cuda.synchronize()
    bufs = m._engine.bufs
    conv, bn = m.inc1.double_conv[0], m.inc1.double_conv[1]
    wt = conv.weight.detach().cpu().double().requires_grad_(True)
    gam = bn.weight.detach().cpu().double().requires_grad_(True)
    bet = bn.bias.detach().cpu().double().requires_grad_(True)
    z = _ste(F.conv2d(x.double(), wt, conv.bias.detach().cpu().double(), padding=1))
    a = _ste(F.relu(F.batch_norm(z, None, None, gam, bet, True, 0.1, 1e-5)))
    assert _rel(_p8_to_nchw(bufs["a:inc1.0"]), a.detach()) <= 5e-3
    (a * _p8_to_nchw(bufs["g:a:inc1.0"]).double()).sum().backward()
    assert conv.weight.grad.shape == (16, 3, 3, 3)
    assert _rel(conv.weight.grad.cpu(), wt.grad) <= 3e-2
    assert _rel(bn.weight.grad.cpu(), gam.grad) <= 3e-2 and _rel(bn.bias.grad.cpu(), bet.grad) <= 3e-2


@pytest.mark.parametrize("B,H,W", [(2, 64, 64), (3, 96, 160)])
def test_fused_batchnorm_statistics_match_separate_pass(B, H, W):
    """The BatchNorm batch statistics accumulated in the conv epilogues (AbcConvDesc.stat_sum / stat_sq: operand-swap launches
    and the row-folded 16 -> 16 layers) against abc_bn_stats run on the SAME stored conv output: per channel sum and sum of
    squares equal up to fp32 summation order. Partial tiles included (96 x 160 is not a multiple of the 32 / 64 / 128-row swap
    tiles at every level; the deepest maps are narrower than one 8-pixel tile). An end-to-end comparison of the two modes would
    only measure train-mode BatchNorm's amplification of last-bit differences (see test_train_step_in_situ_layer_parity)."""
    import ctypes as C
    from abcnet_b200 import _lib
    m, sd, x = _setup(7, B, H, W)
    assert m.fuse_bn
    m(x.cuda())
    torch.cuda.synchronize()
    eng = m._engine
    st = torch.cuda.current_stream().cuda_stream
    fused, checked = 0, 0
    for u in eng.saved["plan"]:
        if "up" in u or u.get("first"):
            continue
        z = eng.saved["units"][u["name"]]["z"]
        got_s, got_q = [t.clone() for t in eng._stat_bufs("bn:" + u["name"], u["cout"])]
        want_s, want_q = torch.zeros_like(got_s), torch.zeros_like(got_q)
        N, planes, h, w, _ = z.shape
        _lib.check(_lib.lib.abc_bn_stats(z.data_ptr(), N, h, w, planes, 0, u["cout"], want_s.data_ptr(), want_q.data_ptr(), st))
        torch.cuda.synchronize()
        checked += 1
        tol_s = 1e-5 * float(want_q.sqrt().max() * (N * h * w) ** 0.5) + 1e-6
        assert (got_s - want_s).abs().max().item() <= tol_s, (u["name"], (got_s - want_s).abs().max().item(), tol_s)
        assert _rel(got_q.cpu(), want_q.cpu()) <= 1e-5, (u["name"], _rel(got_q.cpu(), want_q.cpu()))
    # which launches carried the statistics: every cout <= 128 layer except the three 16 -> 16 ... all of them here
    from abcnet_b200.train import can_fuse_stats
    fused = sum(1 for k, pk in eng._packs.items() if not k.endswith(".dgrad") and "heads" not in k and ".up." not in k
                and can_fuse_stats(pk, object()))
    print(f"fused BatchNorm statistics verified on {checked} conv units ({fused} of them accumulated in the conv epilogue)")
    assert checked >= 20 and fused >= 14
