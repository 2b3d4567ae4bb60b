"""abc_heads_fused (hidden maps kept in tensor memory, the default inference path) against the separate conv1 / conv2
launches, bit for bit: both compute the same 16-bit hidden values and accumulate conv2 over K in the same order. Head
lists of every shape the kernel takes, partial tiles, B = 1, both output layouts and both activation formats; the decoded
records; and a CUDA-graph replay against the eager call."""
import numpy as np
import pytest
import torch

from oracle import synth, unet_ref

pytestmark = pytest.mark.gpu

V2 = list(unet_ref.V2_HEADS)


def _model(heads, act_dtype, seed=9):
    import abcnet_b200
    sd = unet_ref.make_state_dict(seed=seed, heads=tuple(heads), variant="W1")
    m = abcnet_b200.UNet(1, list(heads), act_dtype=act_dtype).cuda().eval()
    m.load_state_dict(sd)
    return m


@pytest.mark.parametrize("act_dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("heads,B,H,W", [(V2, 2, 96, 64), ([1, 21, 5, 1, 4, 2], 1, 64, 96), ([1, 14, 3], 1, 96, 32),
                                         ([360], 2, 64, 64), ([5, 60, 2, 360, 1], 1, 32, 96)])
def test_fused_heads_equal_separate_launches(heads, B, H, W, act_dtype):
    m = _model(heads, act_dtype)
    x = torch.from_numpy(synth.binary_images(9, B, H, W, 0.08)).cuda()
    sep = [o.clone() for o in m.infer(x, fused=False)]
    assert m._packed.get("heads.fused") is not None
    fus = [o.clone() for o in m.infer(x)]                  # the default is the fused kernel
    fus_p8 = m.infer(x, layout="p8f", fused=True).to_nchw()
    sep_p8 = m.infer(x, layout="p8f", fused=False).to_nchw()
    torch.cuda.synchronize()
    for i, (a, b, c, d) in enumerate(zip(sep, fus, fus_p8, sep_p8)):
        assert a.shape == b.shape == c.shape
        assert torch.equal(a, b), f"head {i}: fused NCHW differs by {(a - b).abs().max().item()}"
        assert torch.equal(c, d), f"head {i}: fused planar-8 differs by {(c - d).abs().max().item()}"
        assert torch.equal(a, c)


def test_fused_heads_records_and_graph_replay():
    import abcnet_b200
    m = _model(V2, "bf16", seed=1)
    x = torch.from_numpy(synth.binary_images(5, 2, 512, 512, 0.05)).cuda()
    sep = m.infer(x, layout="p8f", fused=False)            # each call without `outs` returns new buffers
    fus = m.infer(x, layout="p8f")
    for a, b in zip(sep.to_nchw(), fus.to_nchw()):
        assert torch.equal(a, b)
    # shift the centre / omega maps so that there are peaks to decode, identically in both
    for k in (0, 4, 7):
        off = -1.0 - torch.quantile(sep.to_nchw()[k].flatten()[:1_000_000], 0.995)
        sep[k] += off
        fus[k] += off
    dec = abcnet_b200.PeakDecoder(2, atom_cap=16384, bond_cap=262144)
    r_sep = dec(sep)
    r_fus = dec(fus)
    assert sum(len(a) for a, _, _ in r_fus) > 10
    for (a1, b1, n1), (a2, b2, n2) in zip(r_sep, r_fus):
        assert n1 == n2 and np.array_equal(a1, a2) and np.array_equal(b1, b2)
    # one CUDA graph of the fused forward + decode against the eager call on the same input
    g = abcnet_b200.InferGraph(m, 2, 512, 512, atom_cap=16384, bond_cap=262144, dtype=x.dtype)
    r_graph = g(x)
    eager = m.infer(x, layout="p8f")
    r_eager = abcnet_b200.PeakDecoder(2, atom_cap=16384, bond_cap=262144)(eager)
    for a, b in zip(g.outs.to_nchw(), eager.to_nchw()):
        assert torch.equal(a, b)
    for (a1, b1, n1), (a2, b2, n2) in zip(r_graph, r_eager):
        assert n1 == n2 and np.array_equal(a1, a2) and np.array_equal(b1, b2)
