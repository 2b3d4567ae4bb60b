"""GPU checks of the pooled slot layout of SparseHeadsPipeline (``peak_pool=S``): a batch shares S slots, so one crowded image
may hold most of them. Records must equal UNet.infer + PeakDecoder bit for bit (positions, classes, omega survivors, rho
bits, counts) and the MOL blocks built from them must be the same text."""
import numpy as np
import pytest
import torch

from oracle import synth, unet_ref

pytestmark = pytest.mark.gpu
HEADS = list(unet_ref.V2_HEADS)
CROWDED = 2                                   # index of the crowded image: groups before and after it share the pool
SCALES = (1.5, 2, 3, 4, 6, 8, 12, 16, 24, 32)


def _model(seed, act_dtype="bf16"):
    import abcnet_b200
    m = abcnet_b200.UNet(1, HEADS, act_dtype=act_dtype).cuda().eval()
    m.load_state_dict(unet_ref.make_state_dict(seed=seed, variant="W1"))
    return m


def _calibrate(m, x, q):
    """Constant offsets on the centre / omega heads so that a fraction (1 - q) of the pixels exceeds the -1 threshold."""
    outs = m(x)
    with torch.no_grad():
        for k in (0, 4, 7):
            m.out_modules[k].conv2.bias += -1.0 - torch.quantile(outs[k].flatten()[:2_000_000].float(), q)


def _images(seed, B, H=512, W=512):
    return torch.from_numpy(synth.binary_images(seed, B, H, W, 0.05)).cuda()


def _dense(B, H4W4):
    import abcnet_b200
    return abcnet_b200.PeakDecoder(B, atom_cap=H4W4, bond_cap=1 << 17)


def _same(want, got):
    for i, ((wa, wb, wn), (ga, gb, gn)) in enumerate(zip(want, got)):
        assert wn == gn, (i, wn, gn)
        assert np.array_equal(wa, ga), f"image {i}: atom records differ"
        assert np.array_equal(wb, gb), f"image {i}: bond records differ"    # structured compare: includes the rho bits
    assert len(want) == len(got)


def _crowd(m, x, dec, **opt):
    """Scale the amplitude of image CROWDED (fp32 input) until its bond-centre map has more than 1024 peaks (several
    rounds of the record kernel), or as far as SCALES go. Returns (input, dense records, counts [B, 4])."""
    best = None
    for s in SCALES:
        xc = x.clone()
        xc[CROWDED] *= s
        want = dec(m.infer(xc, layout="p8f"), **opt)
        counts = dec.h_counts[:x.shape[0]].numpy().copy()
        if best is None or counts[CROWDED, 2] > best[2][CROWDED, 2]:
            best = (xc, want, counts)
        if counts[CROWDED, 2] > 1024:
            break
    return best


def _pool_for(counts):
    total = int(counts[:, 0].sum() + counts[:, 2].sum())
    return total, (total + 63) // 64 * 64


@pytest.mark.parametrize("omega_mode,apply_sigmoid,act_dtype", [("nms", False, "bf16"), ("raw", False, "bf16"),
                                                                 ("nms", True, "bf16"), ("nms", False, "fp16")])
def test_pooled_crowded_image_equals_dense_path(omega_mode, apply_sigmoid, act_dtype):
    import abcnet_b200
    B = 8
    m = _model(31, act_dtype)
    x = _images(41, B)
    _calibrate(m, x, 0.997)
    opt = dict(omega_mode=omega_mode)
    if apply_sigmoid:
        opt.update(thr=0.27, apply_sigmoid=True, thr_omega=-1.0)         # just above sigmoid(-1): the calibrated density
    dense = _dense(B, 128 * 128)
    xc, want, counts = _crowd(m, x, dense, **opt)
    total, S = _pool_for(counts)
    crowded = int(counts[CROWDED, 0] + counts[CROWDED, 2])
    print(f"peaks per image (atoms + bond centres): {(counts[:, 0] + counts[:, 2]).tolist()}, pool {S}")
    assert crowded > 4 * S / B, (crowded, S)                              # far more than its share of the pool
    assert counts[CROWDED, 0] > 128 or counts[CROWDED, 2] > 128           # more than the fixed layout's peak_cap below
    assert sum(len(b) for _, b, _ in want) > 0
    fixed = abcnet_b200.SparseHeadsPipeline(m, B, peak_cap=128, bond_cap=1 << 17)
    with pytest.raises(RuntimeError, match="capacity|peak_cap"):
        fixed.fetch(fixed.launch(xc, **opt))
    pipe = abcnet_b200.SparseHeadsPipeline(m, B, bond_cap=1 << 17, peak_pool=S, atom_cap=128 * 128)
    got = pipe.fetch(pipe.launch(xc, **opt))
    _same(want, got)
    assert pipe.molblocks(B) == dense.molblocks(B)
    # a normal batch through the same buffers afterwards: no stale slot of the crowded one leaks
    x2 = _images(42, B)
    want2 = dense(m.infer(x2, layout="p8f"), **opt)
    _same(want2, pipe.fetch(pipe.launch(x2, **opt)))


def test_partial_batches_in_both_layouts():
    import abcnet_b200
    m = _model(32)
    x = _images(43, 6)
    _calibrate(m, x, 0.995)
    dense = _dense(6, 128 * 128)
    pipes = [abcnet_b200.SparseHeadsPipeline(m, 6, peak_cap=512, bond_cap=1 << 15),
             abcnet_b200.SparseHeadsPipeline(m, 6, bond_cap=1 << 15, peak_pool=2 * 6 * 128)]
    for B in (6, 3, 1):
        want = dense(m.infer(x[:B].contiguous(), layout="p8f"))
        assert sum(len(a) for a, _, _ in want) > 5 * B
        for pipe in pipes:
            got = pipe.fetch(pipe.launch(x[:B].contiguous()))
            assert len(got) == B
            _same(want, got)
            assert pipe.molblocks(B) == dense.molblocks(B)
    with pytest.raises(ValueError, match="up to 6"):
        pipes[1].launch(_images(44, 7))


def test_pool_overflow_raises_and_the_next_batch_is_exact():
    import abcnet_b200
    B = 8
    m = _model(33)
    x = _images(45, B)
    _calibrate(m, x, 0.997)
    dense = _dense(B, 128 * 128)
    xc, _, counts = _crowd(m, x, dense)
    total, S = _pool_for(counts)
    S_small = S - 128
    assert total > S_small
    pipe = abcnet_b200.SparseHeadsPipeline(m, B, bond_cap=1 << 17, peak_pool=S_small, atom_cap=128 * 128)
    with pytest.raises(RuntimeError, match=f"peak_pool {S_small}"):
        pipe.fetch(pipe.launch(xc))
    pipe.fetch_async(pipe.launch(xc))
    with pytest.raises(RuntimeError, match="peak_pool"):
        pipe.collect(B)
    with pytest.raises(RuntimeError, match="peak_pool"):
        pipe.wait(B)
    x2 = _images(46, B)
    want2 = dense(m.infer(x2, layout="p8f"))
    assert int(dense.h_counts[:B, 0].sum() + dense.h_counts[:B, 2].sum()) <= S_small
    _same(want2, pipe.fetch(pipe.launch(x2)))


def test_pooled_launch_replays_from_a_cuda_graph():
    import abcnet_b200
    B = 4
    m = _model(34)
    x = _images(47, B)
    _calibrate(m, x, 0.997)
    dense = _dense(B, 128 * 128)
    pipe = abcnet_b200.SparseHeadsPipeline(m, B, bond_cap=1 << 15, peak_pool=2 * B * 256)
    xs = x.clone()
    for _ in range(2):                                                # eager warm-up: weight packs and buffers exist
        pipe.launch(xs)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        pipe.launch(xs)
    for seed in (48, 49):
        xn = _images(seed, B)
        want = dense(m.infer(xn, layout="p8f"))
        eager = pipe.fetch(pipe.launch(xn))
        _same(want, eager)
        xs.copy_(xn)
        g.replay()
        _same(eager, pipe.fetch(B))


def test_fixed_layout_raises_for_atom_peaks_beyond_peak_cap_under_a_larger_atom_cap():
    """The fixed layout keeps at most peak_cap atom peaks per image, whatever atom_cap is: with atom_cap > peak_cap an image
    with more atom peaks must still make fetch / collect / wait raise instead of returning records that were never written."""
    import abcnet_b200
    B, cap = 2, 64
    m = _model(35)
    x = _images(50, B)
    outs = m(x)
    z = {k: outs[k].flatten()[:2_000_000].float().clone() for k in (0, 4, 7)}
    with torch.no_grad():                                              # few bond-centre peaks, so only the atoms overflow
        for k, q in ((4, 0.9995), (7, 0.997)):
            m.out_modules[k].conv2.bias += -1.0 - torch.quantile(z[k], q)
        b0 = m.out_modules[0].conv2.bias.detach().clone()
    dense = _dense(B, 128 * 128)
    for q in (0.99, 0.98, 0.97, 0.95, 0.9):
        with torch.no_grad():
            m.out_modules[0].conv2.bias.copy_(b0 - 1.0 - torch.quantile(z[0], q))
        want = dense(m.infer(x, layout="p8f"))
        counts = dense.h_counts[:B].numpy().copy()
        if counts[:, 0].max() > cap:
            break
    assert counts[:, 0].max() > cap >= counts[:, 2].max(), counts
    fixed = abcnet_b200.SparseHeadsPipeline(m, B, peak_cap=cap, atom_cap=1024, bond_cap=1 << 15)
    with pytest.raises(RuntimeError, match=f"atom peaks in one image exceed peak_cap {cap}"):
        fixed.fetch(fixed.launch(x))
    fixed.fetch_async(fixed.launch(x))
    with pytest.raises(RuntimeError, match="peak_cap"):
        fixed.collect(B)
    with pytest.raises(RuntimeError, match="peak_cap"):
        fixed.wait(B)
    roomy = abcnet_b200.SparseHeadsPipeline(m, B, peak_cap=1024, atom_cap=1024, bond_cap=1 << 15)
    _same(want, roomy.fetch(roomy.launch(x)))
