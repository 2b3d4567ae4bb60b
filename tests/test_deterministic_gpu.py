"""Bit-reproducible training under torch.use_deterministic_algorithms(True): every reduction of the step (split-K weight
gradients, BatchNorm statistics and backward sums, bias sums, loss sums) stores per-block partials to workspace slots that one
kernel adds in a fixed order. Checked per kernel (two deterministic launches are torch.equal and agree with the atomic path
within reordering tolerance), for the whole TrainStep (eager and graph), for the autograd path and across processes."""
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

from oracle import synth, unet_ref

pytestmark = pytest.mark.gpu
HEADS = list(unet_ref.V2_HEADS)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def det_mode():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev)


def _p8(seed, N, planes, H, W, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn((N, planes, H, W, 8), generator=g) * scale).to(torch.bfloat16).cuda()


def _rel(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _ws(n):
    return torch.empty(max(int(n), 1), dtype=torch.uint8, device="cuda")


# ------------------------------------------------------------------------------------------------ per kernel
WGRAD_CASES = [  # (cout, cin, H, W, taps, row_boxes): the shapes of test_train_ops_gpu.py::test_wgrad_conv3x3
    (16, 16, 64, 64, 9, 0), (16, 16, 64, 64, 9, 1), (32, 16, 32, 48, 9, 0), (64, 32, 32, 32, 9, 1), (128, 128, 16, 16, 9, 0),
    (256, 256, 8, 8, 9, 0), (24, 128, 16, 24, 1, 0), (1024, 128, 16, 16, 9, 0), (128, 64, 24, 16, 4, 0),
]


@pytest.mark.parametrize("cout,cin,H,W,ntaps,row_boxes", WGRAD_CASES)
def test_wgrad_deterministic(cout, cin, H, W, ntaps, row_boxes):
    from abcnet_b200._lib import AbcWgradDesc, check, lib
    N = 3
    dz, a = _p8(1, N, cout // 8, H, W), _p8(2, N, cin // 8, H, W)
    taps = [(dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)][:ntaps] if ntaps != 1 else [(0, 0)]
    if ntaps == 4:
        taps = [(0, 0), (0, -1), (-1, 0), (-1, -1)]

    def run(det):
        dw = torch.zeros((ntaps, cout, cin), dtype=torch.float32, device="cuda")
        d = AbcWgradDesc()
        d.dz, d.dz_planes, d.dz_plane_off, d.cout = dz.data_ptr(), cout // 8, 0, cout
        d.in_, d.in_planes, d.in_plane_off, d.cin = a.data_ptr(), cin // 8, 0, cin
        d.N, d.H, d.W, d.ntaps, d.row_boxes = N, H, W, ntaps, row_boxes
        for i, (dy, dx) in enumerate(taps):
            d.tap_dy[i], d.tap_dx[i] = dy, dx
        d.dw = dw.data_ptr()
        ws = None
        if det:
            ws = torch.full((lib.abc_conv_wgrad_workspace_bytes(C.byref(d)) // 4,), float("nan"), device="cuda")
            d.ws = ws.data_ptr()
        check(lib.abc_conv_wgrad(C.byref(d), _st()), "abc_conv_wgrad")
        torch.cuda.synchronize()
        return dw
    d1, d2, ref = run(True), run(True), run(False)
    assert torch.equal(d1, d2)
    assert torch.isfinite(d1).all()
    assert _rel(d1, ref) <= 1e-6


@pytest.mark.parametrize("N,C_,H,W", [(2, 16, 64, 64), (4, 64, 32, 32), (1, 8, 1, 1), (3, 24, 7, 5)])
def test_bn_stats_and_channel_sum_deterministic(N, C_, H, W):
    from abcnet_b200._lib import check, lib
    z = _p8(3, N, C_ // 8 + 1, H, W)

    def run(det):
        s = torch.empty(C_, dtype=torch.float64, device="cuda")
        q = torch.empty(C_, dtype=torch.float64, device="cuda")
        if det:
            ws = _ws(lib.abc_bn_stats_workspace_bytes(N, H, W, C_))
            check(lib.abc_bn_stats_det(z.data_ptr(), N, H, W, C_ // 8 + 1, 1, C_, s.data_ptr(), q.data_ptr(), ws.data_ptr(), _st()), "det")
        else:
            check(lib.abc_bn_stats(z.data_ptr(), N, H, W, C_ // 8 + 1, 1, C_, s.data_ptr(), q.data_ptr(), _st()), "bn_stats")
        torch.cuda.synchronize()
        return s, q
    (s1, q1), (s2, q2), (sr, qr) = run(True), run(True), run(False)
    assert torch.equal(s1, s2) and torch.equal(q1, q2)
    assert torch.allclose(s1, sr, rtol=1e-12, atol=1e-9) and torch.allclose(q1, qr, rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("pool", [False, True])
def test_bn_act_backward_deterministic(pool):
    from abcnet_b200._lib import AbcBnActBwdDesc, check, lib
    N, C_, H, W = 4, 32, 32, 32
    z, dA = _p8(4, N, C_ // 8, H, W), _p8(5, N, C_ // 8, H, W)
    dP = _p8(6, N, C_ // 8, H // 2, W // 2) if pool else None
    g = torch.Generator().manual_seed(7)
    st = [(torch.rand(C_, generator=g) + 0.5).cuda(), (torch.randn(C_, generator=g) * 0.1).cuda(),
          (torch.randn(C_, generator=g) * 0.1).cuda(), (torch.rand(C_, generator=g) + 0.5).cuda()]

    def run(det):
        s1 = torch.empty(C_, dtype=torch.float64, device="cuda")
        s2 = torch.empty(C_, dtype=torch.float64, device="cuda")
        dz = torch.empty_like(z)
        d = AbcBnActBwdDesc()
        d.z, d.z_planes, d.z_plane_off = z.data_ptr(), C_ // 8, 0
        d.dA, d.dA_planes, d.dA_plane_off = dA.data_ptr(), C_ // 8, 0
        if pool:
            d.dP, d.dP_planes, d.dP_plane_off = dP.data_ptr(), C_ // 8, 0
        d.dz, d.dz_planes, d.dz_plane_off = dz.data_ptr(), C_ // 8, 0
        d.N, d.H, d.W, d.C = N, H, W, C_
        d.scale, d.shift, d.mean, d.invstd = [t.data_ptr() for t in st]
        d.act, d.s1, d.s2 = 1, s1.data_ptr(), s2.data_ptr()
        ws = _ws(lib.abc_bn_act_backward_workspace_bytes(C.byref(d))) if det else None
        if det:
            d.ws = ws.data_ptr()
        check(lib.abc_bn_act_backward(C.byref(d), _st()), "abc_bn_act_backward")
        torch.cuda.synchronize()
        return s1, s2, dz
    a, b, r = run(True), run(True), run(False)
    for x, y, ref in zip(a, b, r):
        assert torch.equal(x, y)
    assert torch.allclose(a[0], r[0], rtol=1e-12, atol=1e-9) and torch.allclose(a[1], r[1], rtol=1e-12, atol=1e-9)
    assert _rel(a[2].float(), r[2].float()) <= 1e-2          # dz: bf16 of values computed from reordered sums


def test_nchw_to_p8_ex_deterministic():
    from abcnet_b200._lib import check, lib
    N, C_, H, W, planes = 4, 60, 32, 32, 8
    g = torch.randn((N, C_, H, W), generator=torch.Generator().manual_seed(8)).cuda()
    sc = torch.tensor([0.37], device="cuda")

    def run(det):
        dst = torch.empty((N, planes, H, W, 8), dtype=torch.bfloat16, device="cuda")
        db = torch.empty(C_, dtype=torch.float64, device="cuda")
        if det:
            ws = _ws(lib.abc_nchw_to_p8_ex_workspace_bytes(N, C_, H, W, planes))
            check(lib.abc_nchw_to_p8_ex_det(g.data_ptr(), dst.data_ptr(), N, C_, H, W, planes, sc.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                            _st()), "det")
        else:
            check(lib.abc_nchw_to_p8_ex(g.data_ptr(), dst.data_ptr(), N, C_, H, W, planes, sc.data_ptr(), db.data_ptr(), _st()), "ex")
        torch.cuda.synchronize()
        return dst, db
    (x1, b1), (x2, b2), (xr, br) = run(True), run(True), run(False)
    assert torch.equal(x1, xr) and torch.equal(b1, b2)
    assert torch.allclose(b1, br, rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("cin", [1, 3])
def test_stem_wgrad_deterministic(cin):
    from abcnet_b200._lib import check, lib
    N, H, W = 4, 64, 64
    dz = _p8(9, N, 2, H, W)
    if cin == 1:
        img = torch.from_numpy(synth.binary_images(9, N, H, W, 0.08)).to(torch.uint8).cuda().contiguous()
    else:
        img = torch.rand((N, cin, H, W), generator=torch.Generator().manual_seed(9)).cuda()

    def run(det):
        dw = torch.zeros(144 * cin, dtype=torch.float32, device="cuda")
        ws = _ws(lib.abc_conv3x3_wgrad_workspace_bytes(cin)) if det else None
        if cin == 1:
            if det:
                check(lib.abc_conv3x3_c1_wgrad_det(img.data_ptr(), 1, dz.data_ptr(), 2, 0, N, H, W, dw.data_ptr(), ws.data_ptr(), _st()), "c1")
            else:
                check(lib.abc_conv3x3_c1_wgrad(img.data_ptr(), 1, dz.data_ptr(), 2, 0, N, H, W, dw.data_ptr(), _st()), "c1")
        else:
            if det:
                check(lib.abc_conv3x3_cn_wgrad_det(img.data_ptr(), cin, dz.data_ptr(), 2, 0, N, H, W, dw.data_ptr(), ws.data_ptr(), _st()), "cn")
            else:
                check(lib.abc_conv3x3_cn_wgrad(img.data_ptr(), cin, dz.data_ptr(), 2, 0, N, H, W, dw.data_ptr(), _st()), "cn")
        torch.cuda.synchronize()
        return dw
    a, b, r = run(True), run(True), run(False)
    assert torch.equal(a, b)
    assert _rel(a, r) <= 1e-5


def _targets(seed, B, h, w):
    return [torch.from_numpy(t).cuda().contiguous() for t in synth.dense_targets(seed, B, h, w)]


@pytest.mark.parametrize("p8", [False, True])
def test_loss_deterministic(p8, det_mode):
    """Both loss entry points under the flag: bit-identical twice, and within reordering tolerance of the atomic path."""
    from abcnet_b200 import loss as L
    from abcnet_b200.loss import head_grad_planes
    B, h, w = 4, 64, 64
    tg = _targets(12, B, h, w)
    gen = torch.Generator().manual_seed(12)
    logits = [torch.randn((B, c, h, w), generator=gen).cuda() for c in HEADS]
    s = torch.zeros(10, device="cuda")

    def run():
        if p8:
            dz = [torch.empty((B, head_grad_planes(c), h, w, 8), dtype=torch.bfloat16, device="cuda") for c in HEADS]
            db = [torch.empty(c, dtype=torch.float64, device="cuda") for c in HEADS]
            total, parts, ds, hs = L.loss_forward_p8(s, None, tg, logits, dz, db)
            out = [total, parts, ds, hs] + dz + db
        else:
            total, parts, ds, dl, _ = L.loss_forward_backward(s, None, tg, logits)
            out = [total, parts, ds] + dl
        torch.cuda.synchronize()
        return [t.clone() for t in out]
    a, b = run(), run()
    torch.use_deterministic_algorithms(False)
    r = run()
    torch.use_deterministic_algorithms(True)
    for x, y, ref in zip(a, b, r):
        assert torch.equal(x, y)
        assert not torch.isnan(x.double()).any()
        if x.dtype == torch.float64:
            assert torch.allclose(x, ref, rtol=1e-10, atol=1e-12), (x, ref)


# ------------------------------------------------------------------------------------------------ whole step
def _model(seed, p_drop):
    import abcnet_b200
    m = abcnet_b200.UNet(1, HEADS).cuda()
    m.load_state_dict(unet_ref.make_state_dict(seed=seed, variant="W1"))
    m.train()
    m.dropout_p = p_drop
    return m


def _state(m, opt, losses):
    """Everything a step produces: loss values, gradients, parameters, buffers (running statistics), optimiser moments."""
    out = {"loss": torch.stack([l.double().reshape(()) for l in losses])}
    for n, p in m.named_parameters():
        out["p:" + n] = p.detach().clone()
        if p.grad is not None:
            out["g:" + n] = p.grad.detach().clone()
    for n, b in m.named_buffers():
        out["b:" + n] = b.detach().clone()
    if opt is not None:
        for i, p in enumerate(m.parameters()):
            for k, v in opt.state.get(p, {}).items():
                if torch.is_tensor(v):
                    out[f"o:{i}:{k}"] = v.detach().clone()
    return out


def _run_steps(seed, B, H, W, use_graph, seed_buf=None, steps=3, p_drop=0.2):
    import abcnet_b200
    m = _model(seed, p_drop)
    x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08)).cuda()
    tg = _targets(seed, B, H // 4, W // 4)
    if seed_buf is not None:                      # same dropout stream as the first engine (each engine draws its own seed);
        # a graph run draws two counters in its warm-up before the replays, so it starts two counters earlier
        m._train_engine().bufs["seed"] = seed_buf.clone() - (2 * 0x5DEECE66D if use_graph else 0)
    opt = abcnet_b200.make_optimizer(m, capturable=use_graph)
    step = abcnet_b200.TrainStep(m, opt, class_weights=True, use_graph=use_graph)
    losses = [step(x, tg) for _ in range(steps)]
    torch.cuda.synchronize()
    st = _state(m, opt, losses)
    st["parts"] = step.parts.clone()
    return st, m._train_engine().bufs["seed"]


def test_train_step_bit_reproducible_eager_and_graph(det_mode):
    B, H, W, seed = 4, 128, 128, 21
    ref, sbuf = _run_steps(seed, B, H, W, False)
    sbuf0 = sbuf.clone() - 3 * 0x5DEECE66D            # the counter before the three forwards advanced it
    runs = {"eager2": _run_steps(seed, B, H, W, False, sbuf0)[0], "graph": _run_steps(seed, B, H, W, True, sbuf0)[0]}
    runs["graph2"] = _run_steps(seed, B, H, W, True, sbuf0)[0]
    for name, st in runs.items():
        assert st.keys() == ref.keys()
        for k in ref:
            assert torch.equal(st[k], ref[k]), (name, k)
    for k, v in ref.items():
        assert not torch.isnan(v.double()).any(), k           # torch's NaN fill of torch.empty must not reach any result
    # against the default (atomic) step: one step (later Adam steps amplify last-bit differences), dropout off so that both
    # see the same function, the first-step tolerances of test_train_gpu.py
    det = _run_steps(seed, B, H, W, False, p_drop=0.0, steps=1)[0]
    torch.use_deterministic_algorithms(False)
    nd = _run_steps(seed, B, H, W, False, p_drop=0.0, steps=1)[0]
    torch.use_deterministic_algorithms(True)
    assert abs(det["loss"][0].item() - nd["loss"][0].item()) <= 1e-6 * abs(nd["loss"][0].item())
    names = [k for k in nd if k.startswith("g:") and nd[k].abs().max().item() != 0.0]
    flat = torch.cat([det[k].flatten().double() for k in names])
    flat_nd = torch.cat([nd[k].flatten().double() for k in names])
    assert _rel(flat, flat_nd) <= 5e-2
    assert max(_rel(det[k], nd[k]) for k in names) <= 1e-1


def test_autograd_path_bit_reproducible(det_mode):
    import abcnet_b200
    B, H, W, seed = 4, 128, 128, 22

    def run():
        m = _model(seed, 0.0)
        x = torch.from_numpy(synth.binary_images(seed, B, H, W, 0.08)).cuda()
        tg = _targets(seed, B, H // 4, W // 4)
        crit = abcnet_b200.HeatmapLoss(class_weights=True)
        loss = crit(m(x), tg, m.s)
        loss.backward()
        torch.cuda.synchronize()
        return _state(m, None, [loss.detach()])
    a, b = run(), run()
    for k in a:
        assert torch.equal(a[k], b[k]), k
        assert not torch.isnan(a[k].double()).any(), k


_CHILD = r"""
import hashlib, sys, torch
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
torch.use_deterministic_algorithms(True)
torch.manual_seed(5)
import test_deterministic_gpu as T
st, _ = T._run_steps(31, 8, 256, 256, True)
h = hashlib.sha256()
for k in sorted(st):
    h.update(k.encode()); h.update(st[k].detach().cpu().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes())
print("DIGEST", h.hexdigest())
"""


def test_train_step_reproducible_across_processes():
    """The public contract: two processes with the flag on and the same seed give the same SHA-256 of the loss, parts,
    gradients, parameters, running statistics and Adam moments after 3 graph steps at B = 8, 256 x 256."""
    code = _CHILD.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    digests = []
    for _ in range(2):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        digests.append([l for l in r.stdout.splitlines() if l.startswith("DIGEST")][-1])
    assert digests[0] == digests[1], digests
