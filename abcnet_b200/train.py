"""Training-mode U-Net pass (forward with batch-statistics BatchNorm + dropout, and the full backward) on the sm_100a
kernels. Replaces what autograd + cuDNN do for ``/root/reference/src/train.py:94`` (forward in ``model.train()``) and
``:139-140`` (``loss.backward()``) for the model of ``/root/reference/src/unet.py``.

Forward per conv unit:  z = conv(a_in) + b  (tcgen05 implicit GEMM, bf16 P8)  ->  batch statistics (fp64 accumulation)
->  a = act(gamma * (z - mean) * invstd + beta) [* dropout]  (+ fused 2x2 max-pool output).
Backward per conv unit: (dA and/or pooled dP) -> dz (BN / act / dropout / pool-routing backward, also dgamma, dbeta)
->  dW = wgrad(dz, a_in) on tensor cores  ->  dA_in = conv(dz, W^T flipped) with the forward kernel.
The up-sampling convolution is differentiated phase-wise (de-interleave + one K-segmented implicit GEMM for the data
gradient, one wgrad per phase). Gradients of conv biases that feed a train-mode BatchNorm are identically zero.
"""
from __future__ import annotations

import ctypes as C
import itertools
import os

import torch

from . import _lib
from ._lib import AbcBnActBwdDesc, AbcBnActDesc, AbcConvDesc, AbcWgradDesc, check, lib
from .unet import fold_rows, fold_rows_swap, pair_pack, row_fold_for, swap_fold_for, use_cta_pair, use_swap

TAPS3 = [(ky - 1, kx - 1) for ky in range(3) for kx in range(3)]
_seed_counter = itertools.count(0)


def _initial_dropout_seed():
    """First value of an engine's dropout counter: torch's global seed (so ``torch.manual_seed`` controls the masks, as it
    does for nn.Dropout in the reference), mixed with the data-parallel rank (every replica must draw its own masks) and
    an engine ordinal."""
    import torch.distributed as dist
    rank = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
    z = (torch.initial_seed() + 0x9E3779B97F4A7C15 * (rank + 1) + 0xBF58476D1CE4E5B9 * next(_seed_counter)) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return (z ^ (z >> 31)) & 0x3FFFFFFFFFFFFFFF                       # positive int64


timing = None   # set to a list to collect (label, start event, end event) around every conv / wgrad launch (tools only)


class _timed:
    def __init__(self, label):
        self.label = label

    def __enter__(self):
        if timing is not None:
            self.a, self.b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if timing is not None:
            self.b.record()
            timing.append((self.label, self.a, self.b))
        return False


def _st():
    return _lib.current_stream_ptr()


def deterministic():
    """torch.use_deterministic_algorithms(True) (warn_only too): every reduction of the training step then runs in a fixed
    order (per-block slots of a workspace summed by one small kernel instead of atomics), read when the work is enqueued."""
    return torch.are_deterministic_algorithms_enabled()


def _n_tile(cout):
    c16 = (cout + 15) // 16 * 16
    if c16 <= 128:
        return c16
    return 256 if cout % 256 == 0 else 128


class Packed:
    """Packed bf16 weight blocks in the kernel's consumption order (see include/abcnet_b200.h)."""

    def __init__(self, w_taps, bias, taps, n_tile=None, segments=None, fold=1, fold_swap=False):
        # w_taps: [ntaps, cout, K] fp32; without segments every tap sees all K channels. With segments =
        # [(tap0, ntaps), ...] the K axis of tap t covers only its segment's channels (K = channels per segment).
        self.fold, real_cout = fold, w_taps.shape[1]
        self.fold_swap = bool(fold_swap) and fold > 1                  # folded rows in the operand-swap order (unet.swap_fold_for)
        if fold > 1:                                                   # row folding (AbcConvDesc.row_fold): Toeplitz along y
            w_taps, bias = (fold_rows_swap if self.fold_swap else fold_rows)(w_taps, bias, taps, fold)
            n_tile = fold * real_cout
        ntaps, cout, K = w_taps.shape
        n_tile = n_tile or _n_tile(cout)
        n_tiles = (cout + n_tile - 1) // n_tile
        pad = n_tiles * n_tile - cout
        if pad:
            w_taps = torch.cat([w_taps, w_taps.new_zeros(ntaps, pad, K)], 1)
            bias = torch.cat([bias, bias.new_zeros(pad)])
        kc = min(K, 64)
        w = w_taps.view(ntaps, n_tiles, n_tile, K // kc, kc // 8, 8)
        self.pair = segments is None and fold == 1 and use_cta_pair(K, ntaps, n_tile)
        if self.pair:                                                  # CTA-pair mode: blocks as two halves of n_tile / 2 rows
            blocks = pair_pack(w_taps, n_tiles, n_tile)
            self.cin = K
        elif segments is None:
            blocks = w.permute(1, 3, 0, 4, 2, 5)                      # [nt][chunk][tap][kp][n_tile][8]
            self.cin = K
        else:
            parts = []
            for (t0, nt) in segments:
                parts.append(w[t0:t0 + nt].permute(1, 3, 0, 4, 2, 5).reshape(n_tiles, -1, kc // 8, n_tile, 8))
            blocks = torch.cat(parts, 1)                               # [nt][blocks in consumption order][kp][n_tile][8]
            self.cin = K * len(segments)
        # index mode (PackArena): float64 "codes" instead of values -- the layout code above only moves elements around, so
        # running it on element indices yields the gather map of the packed block; no cast then
        raw = w_taps.dtype == torch.float64
        self.w = blocks.contiguous() if raw else blocks.contiguous().to(torch.bfloat16)
        self.bias = bias.contiguous() if raw else bias.contiguous().float()
        self.taps, self.n_tile, self.cout, self.segments = taps, n_tile, real_cout, segments


class PackArena:
    """Packed weights of every convolution of the training pass (forward and backward), rebuilt from the fp32 master
    parameters by ONE ``abc_gather_pack`` launch per dtype and iteration (SURVEY.md section 8f, N3).

    The gather maps are derived by running the ordinary packing code (``Packed``: tap stacking, BN-free layouts, row folding,
    K segmentation, zero padding) once on tensors of element *codes* ``(parameter id << 22 | offset) + 1`` (0 = zero
    padding) instead of values. Views into the arenas are stable, so the launch sequence is CUDA-graph replayable."""

    CAP_W = 48 * 1024 * 1024          # bf16 elements (the v2 network needs ~24 M: forward + data-gradient packs)
    CAP_B = 1024 * 1024               # fp32 elements (biases)

    def __init__(self, params, device):
        self.params = list(params)
        assert len(self.params) < 1024 and all(p.numel() < (1 << 22) and p.dtype == torch.float32 for p in self.params)
        self.pid = {id(p): i for i, p in enumerate(self.params)}
        self.key = tuple(p.data_ptr() for p in self.params)
        self.ptrs = torch.tensor(self.key, dtype=torch.int64, device=device)
        self.dev = device
        self.w = torch.zeros(self.CAP_W, dtype=torch.bfloat16, device=device)
        self.wc = torch.full((self.CAP_W,), -1, dtype=torch.int32, device=device)
        self.b = torch.zeros(self.CAP_B, dtype=torch.float32, device=device)
        self.bc = torch.full((self.CAP_B,), -1, dtype=torch.int32, device=device)
        self.used = {"w": 0, "b": 0}

    def codes_of(self, p):
        base = float((self.pid[id(p)] << 22) + 1)
        return (torch.arange(p.numel(), dtype=torch.float64, device=self.dev) + base).view(p.shape)

    def add(self, codes, kind):
        """Append a block given by its float64 code tensor; returns the arena view (filled right away)."""
        arena, carena = (self.w, self.wc) if kind == "w" else (self.b, self.bc)
        n = codes.numel()
        n_pad = (n + 63) // 64 * 64                                    # 128-byte aligned bf16 blocks
        off = self.used[kind]
        if off + n_pad > arena.numel():
            raise RuntimeError("PackArena: capacity exceeded")
        carena[off:off + n].copy_((codes.reshape(-1).to(torch.int64) - 1).to(torch.int32))     # 0 -> -1 = 0xFFFFFFFF = zero
        self.used[kind] = off + n_pad
        self._gather(kind, off, n_pad)
        return arena[off:off + n].view(codes.shape)

    def _gather(self, kind, off, n):
        arena, carena = (self.w, self.wc) if kind == "w" else (self.b, self.bc)
        check(lib.abc_gather_pack(self.ptrs.data_ptr(), carena[off:].data_ptr(), arena[off:].data_ptr(), n, 1 if kind == "w" else 0,
                                  _st()), "abc_gather_pack")

    def refresh(self):
        for kind in ("w", "b"):
            if self.used[kind]:
                self._gather(kind, 0, self.used[kind])


def can_fuse_stats(pk, dst):
    """Fused BatchNorm statistics exist in the operand-swap epilogue and in the row-folded 16 -> 16 epilogue (AbcConvDesc.stat_sum)."""
    return use_swap(pk, 0, dst, None) or (pk.fold == 4 and not pk.fold_swap and pk.cout == 16 and pk.cin == 16 and not pk.pair)


def conv(pk, src, in_plane_off, dst, out_plane_off=0, act=0, out_mode=0, out_scale=(1, 0, 1, 0), pool=None, pool_plane_off=0,
         stats=None, ws=None):
    """stats: (sum, sumsq) fp64 [cout] tensors -> fused BatchNorm statistics of the output (AbcConvDesc.stat_sum / stat_sq).
    ws: ``nbytes -> tensor`` (TrainEngine.det_ws): the statistics are summed in a fixed order (AbcConvDesc.stat_ws)."""
    d = AbcConvDesc()
    N, in_planes, H, W, _ = src.shape
    d.in_, d.N, d.H, d.W = src.data_ptr(), N, H, W
    d.in_planes, d.in_plane_off, d.cin = in_planes, in_plane_off, pk.cin
    d.wpack, d.bias = pk.w.data_ptr(), pk.bias.data_ptr()
    d.cout, d.n_tile, d.ntaps = pk.cout, pk.n_tile, len(pk.taps)
    for i, (dy, dx) in enumerate(pk.taps):
        d.tap_dy[i], d.tap_dx[i] = dy, dx
    if pk.segments:
        d.k_segments = len(pk.segments)
        for i, (t0, nt) in enumerate(pk.segments):
            d.seg_tap0[i], d.seg_ntaps[i] = t0, nt
    d.row_fold, d.cta_pair = pk.fold, int(pk.pair)
    d.subpixel = getattr(pk, "subpixel", 0)
    d.swap_mn = int(use_swap(pk, out_mode, dst, pool)) if not d.subpixel else 0
    d.act, d.out_mode = act, out_mode
    d.out_sy, d.out_oy, d.out_sx, d.out_ox = out_scale
    if dst is not None:
        d.out = dst.data_ptr()
        d.out_H, d.out_W = dst.shape[2], dst.shape[3]
        d.out_planes = dst.shape[1] if out_mode in (0, 2) else 0
        d.out_plane_off = out_plane_off
    else:
        d.out_H, d.out_W = H, W
    if pool is not None:
        d.pool_out, d.pool_planes, d.pool_plane_off = pool.data_ptr(), pool.shape[1], pool_plane_off
    if stats is not None:
        d.stat_sum, d.stat_sq = stats[0].data_ptr(), stats[1].data_ptr()
        if ws is not None:
            d.stat_ws = ws(lib.abc_conv_stat_workspace_bytes(C.byref(d))).data_ptr()
    with _timed(f"conv {pk.cin}->{pk.cout} t{len(pk.taps)} @{H}x{W} nt{pk.n_tile}"):
        check(lib.abc_conv_igemm(C.byref(d), _st()), "abc_conv_igemm")


def wgrad(dz, dz_off, cout, a, a_off, cin, taps, ws=None):
    """-> fp32 [ntaps, cout, cin]; ws as in conv(): fixed-order split-K sum (AbcWgradDesc.ws)."""
    N, _, H, W, _ = a.shape
    dw = torch.zeros((len(taps), cout, cin), dtype=torch.float32, device=a.device)
    d = AbcWgradDesc()
    d.dz, d.dz_planes, d.dz_plane_off, d.cout = dz.data_ptr(), dz.shape[1], dz_off, cout
    d.in_, d.in_planes, d.in_plane_off, d.cin = a.data_ptr(), a.shape[1], a_off, cin
    d.N, d.H, d.W, d.ntaps = N, H, W, len(taps)
    for i, (dy, dx) in enumerate(taps):
        d.tap_dy[i], d.tap_dx[i] = dy, dx
    d.dw = dw.data_ptr()
    d.row_boxes = 1 if os.environ.get("ABCNET_WGRAD_ROWBOX") else 0
    if ws is not None:
        d.ws = ws(lib.abc_conv_wgrad_workspace_bytes(C.byref(d))).data_ptr()
    with _timed(f"wgrad {cin}->{cout} t{len(taps)} @{H}x{W}"):
        check(lib.abc_conv_wgrad(C.byref(d), _st()), "abc_conv_wgrad")
    return dw


def phase_taps(parity, crop_first):
    """(kernel index, input offset) pairs of one output parity of ConvTranspose2d(k=3, s=2) + crop (SURVEY App. A.3)."""
    if crop_first:
        return [(1, 0)] if parity == 0 else [(0, 1), (2, 0)]
    return [(0, 0), (2, -1)] if parity == 0 else [(1, 0)]


def upconv_backward(du, du_off, cout, x, w, crop_first, eng=None, key=None, ws=None):
    """Backward of the up-sampling convolution. du: P8 gradient of the cropped output (planes [du_off, du_off+cout/8) of a
    [N, planes, 2H, 2W, 8] buffer); x: P8 input [N, cin/8, H, W, 8]; w: [cin, cout, 3, 3] fp32.
    Returns (dx P8 [N, cin/8, H, W, 8], dw fp32 [cin, cout, 3, 3])."""
    N, _, H, W, _ = x.shape
    cin = w.shape[0]
    dev = x.device
    dph = torch.empty((N, 4 * cout // 8, H, W, 8), dtype=torch.bfloat16, device=dev)
    check(lib.abc_deinterleave2(du.data_ptr(), du.shape[1], du_off, cout, dph.data_ptr(), N, H, W, _st()), "abc_deinterleave2")
    taps, mats, segments = [], [], []
    dw = torch.zeros_like(w, dtype=torch.float32)
    for py in (0, 1):
        for px in (0, 1):
            ys, xs = phase_taps(py, crop_first), phase_taps(px, crop_first)
            t0 = len(taps)
            fwd_taps = []
            for (ky, dy) in ys:
                for (kx, dx) in xs:
                    taps.append((-dy, -dx))                    # data gradient reads the phase map at i - dy
                    mats.append(w[:, :, ky, kx])               # GEMM N = ci, K = co
                    fwd_taps.append((ky, kx, dy, dx))
            segments.append((t0, len(taps) - t0))
            phase = 2 * py + px
            g = wgrad(dph, phase * (cout // 8), cout, x, 0, cin, [(dy, dx) for (_, _, dy, dx) in fwd_taps], ws=ws)
            for i, (ky, kx, _, _) in enumerate(fwd_taps):
                dw[:, :, ky, kx] = g[i].t()
    if eng is None:
        pk = Packed(torch.stack(mats).float().contiguous(), torch.zeros(cin, device=dev), taps, segments=segments)
    else:      # gather-packed from the live parameter (w is then only used for its shape above)
        def make():
            wi = eng._w(eng_param)
            m_i = [wi[:, :, ky, kx] for py in (0, 1) for px in (0, 1) for (ky, dy) in phase_taps(py, crop_first)
                   for (kx, dx_) in phase_taps(px, crop_first)]
            return Packed(torch.stack(m_i).contiguous(), eng._zeros(cin), taps, segments=segments)
        eng_param = key[1]
        pk = eng._pk(key[0], make)
    dx = torch.empty((N, cin // 8, H, W, 8), dtype=torch.bfloat16, device=dev)
    conv(pk, dph, 0, dx)
    return dx, dw


class TrainEngine:
    """Owns the activation / gradient buffers of one UNet for a fixed input shape and runs forward / backward."""

    def __init__(self, model):
        self.m = model
        self.bufs = {}
        self._mask_keys = set()          # BatchNorm keys whose forward pass stored its dropout keep bits (AbcBnActDesc.drop_mask)
        self.saved = {}
        self.arena = None            # PackArena of the current parameter storage (ABCNET_NO_ARENA=1: re-pack with torch ops)
        self._packs = {}
        self._index_mode = False

    # ------------------------------------------------------------------ packed weights
    def _w(self, p):
        """fp32 values of a parameter -- or, while a gather map is being derived, its element codes."""
        return self.arena.codes_of(p) if self._index_mode else p.detach().float()

    def _zeros(self, n):
        return torch.zeros(n, dtype=torch.float64 if self._index_mode else torch.float32, device=self.m.s.device)

    def _pk(self, key, make):
        """Packed weights for ``key``: ``make()`` builds them from ``self._w(...)`` tensors. With the arena the layout is
        derived once (index mode) and afterwards only refreshed by the per-iteration gather."""
        if self.arena is None:
            return make()
        pk = self._packs.get(key)
        if pk is None:
            self._index_mode = True
            try:
                pk = make()
            finally:
                self._index_mode = False
            pk.w = self.arena.add(pk.w, "w")
            pk.bias = self.arena.add(pk.bias, "b")
            self._packs[key] = pk
        return pk

    def _sync_arena(self):
        """Called at the start of every forward: (re)build the arena when the parameter storage changed, else refresh it."""
        if os.environ.get("ABCNET_NO_ARENA"):
            self.arena, self._packs = None, {}
            return
        params = [p for p in self.m.parameters()]
        key = tuple(p.data_ptr() for p in params)
        if self.arena is None or self.arena.key != key:
            self.arena, self._packs = PackArena(params, self.m.s.device), {}
        else:
            self.arena.refresh()

    # ------------------------------------------------------------------ buffers
    def buf(self, key, shape, dtype=torch.bfloat16, zero=False):
        t = self.bufs.get(key)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            # deterministic mode: torch fills torch.empty with NaN there, and a region no kernel writes (padding / halo planes)
            # would turn into NaN * 0 in the gradients; zeroed once, such regions stay zero
            t = (torch.zeros if zero or deterministic() else torch.empty)(shape, dtype=dtype, device=self.m.s.device)
            self.bufs[key] = t
        return t

    def det_ws(self, nbytes):
        """The workspace of the deterministic reductions: one buffer shared by all of them (they run in stream order, each
        producer followed by its reduction), grown to the largest request -- reached in the warm-up before a graph capture."""
        t = self.bufs.get("det:ws")
        if t is None or t.numel() < nbytes:
            t = self.bufs["det:ws"] = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.m.s.device)
        return t

    def _ws(self):
        return self.det_ws if deterministic() else None

    # ------------------------------------------------------------------ layer helpers
    def _stat_bufs(self, key, Cc):
        return self.buf(key + ".sum", (Cc,), torch.float64), self.buf(key + ".sq", (Cc,), torch.float64)

    def _bn_forward(self, key, z, z_off, Cc, bn_params, act, out, out_off, pool, drop_p, seed, have_stats=False):
        """have_stats: the producing convolution already accumulated the batch statistics into ``_stat_bufs(key)``."""
        N, _, H, W, _ = z.shape
        dev = z.device
        gamma, beta, rmean, rvar = bn_params
        s, q = self._stat_bufs(key, Cc)
        if not have_stats and deterministic():
            ws = self.det_ws(lib.abc_bn_stats_workspace_bytes(N, H, W, Cc))
            check(lib.abc_bn_stats_det(z.data_ptr(), N, H, W, z.shape[1], z_off, Cc, s.data_ptr(), q.data_ptr(), ws.data_ptr(), _st()),
                  "abc_bn_stats_det")
        elif not have_stats:
            check(lib.abc_bn_stats(z.data_ptr(), N, H, W, z.shape[1], z_off, Cc, s.data_ptr(), q.data_ptr(), _st()), "abc_bn_stats")
        st = [self.buf(key + f".st{i}", (Cc,), torch.float32) for i in range(4)]
        check(lib.abc_bn_finalize(s.data_ptr(), q.data_ptr(), Cc, float(N * H * W), gamma.data_ptr(), beta.data_ptr(), 1e-5, 0.1,
                                  rmean.data_ptr(), rvar.data_ptr(), *[t.data_ptr() for t in st], _st()), "abc_bn_finalize")
        d = AbcBnActDesc()
        d.z, d.z_planes, d.z_plane_off = z.data_ptr(), z.shape[1], z_off
        if out is not None:
            d.out, d.out_planes, d.out_plane_off = out.data_ptr(), out.shape[1], out_off
        if pool is not None:
            d.pool, d.pool_planes, d.pool_plane_off = pool.data_ptr(), pool.shape[1], 0
        d.N, d.H, d.W, d.C = N, H, W, Cc
        d.scale, d.shift = st[0].data_ptr(), st[1].data_ptr()
        d.act, d.drop_p, d.seed = act, drop_p, 0
        d.seed_dev = seed.data_ptr() if (seed is not None and drop_p > 0) else None
        if drop_p > 0 and pool is None and not os.environ.get("ABCNET_NO_DROP_MASK"):
            # 1 byte of keep bits per P8 vector (+3 % traffic) saves the backward passes the mask hash they were co-bound by
            d.drop_mask = self.buf(key + ".mask", (N * (Cc // 8) * H * W,), torch.uint8).data_ptr()
            self._mask_keys.add(key)
        else:
            self._mask_keys.discard(key)
        check(lib.abc_bn_act(C.byref(d), _st()), "abc_bn_act")
        return st

    def _bwd_sum_bufs(self, key, Cc):
        return self.buf(key + ".s1", (Cc,), torch.float64), self.buf(key + ".s2", (Cc,), torch.float64)

    def _bn_backward(self, key, z, Cc, st, act, dA, dA_off, dP, dz, drop_p, seed, gscale=None):
        N, _, H, W, _ = z.shape
        s1, s2 = self._bwd_sum_bufs(key, Cc)
        d = AbcBnActBwdDesc()
        d.z, d.z_planes, d.z_plane_off = z.data_ptr(), z.shape[1], 0
        if dA is not None:
            d.dA, d.dA_planes, d.dA_plane_off = dA.data_ptr(), dA.shape[1], dA_off
        if dP is not None:
            d.dP, d.dP_planes, d.dP_plane_off = dP.data_ptr(), dP.shape[1], 0
        d.dz, d.dz_planes, d.dz_plane_off = dz.data_ptr(), dz.shape[1], 0
        d.N, d.H, d.W, d.C = N, H, W, Cc
        d.scale, d.shift, d.mean, d.invstd = [t.data_ptr() for t in st]
        d.act, d.drop_p, d.seed = act, drop_p, 0
        d.seed_dev = seed.data_ptr() if (seed is not None and drop_p > 0) else None
        d.s1, d.s2 = s1.data_ptr(), s2.data_ptr()
        d.gscale = gscale.data_ptr() if gscale is not None else None
        if drop_p > 0 and key in self._mask_keys:                      # the keep bits the forward pass of this step stored
            d.drop_mask = self.bufs[key + ".mask"].data_ptr()
        if deterministic():
            d.ws = self.det_ws(lib.abc_bn_act_backward_workspace_bytes(C.byref(d))).data_ptr()
        check(lib.abc_bn_act_backward(C.byref(d), _st()), "abc_bn_act_backward")
        return s1, s2

    # ------------------------------------------------------------------ network description
    def _double(self, prefix, holder, src, src_off, cin, cout, hw, dst2=None, dst2_off=0, pool2=None, keep2=True):
        """Two conv units of a DoubleConv. Returns the list of unit dicts."""
        seq = holder.double_conv
        u1 = dict(name=prefix + ".0", conv=seq[0], bn=seq[1], act=1, src=src, src_off=src_off, cin=cin, cout=cout, hw=hw,
                  dst=("a", prefix + ".0"), dst_off=0, pool=None, keep=True)
        u2 = dict(name=prefix + ".3", conv=seq[3], bn=seq[4], act=1, src=("a", prefix + ".0"), src_off=0, cin=cout, cout=cout, hw=hw,
                  dst=dst2 if dst2 is not None else ("a", prefix + ".3"), dst_off=dst2_off, pool=pool2, keep=keep2)
        return [u1, u2]

    def _plan(self, H, W):
        m = self.m
        L = []
        # first conv handled separately (direct kernel): unit 0
        seq = m.inc1.double_conv
        L.append(dict(name="inc1.0", conv=seq[0], bn=seq[1], act=1, src=("img", None), src_off=0, cin=m.n_channels, cout=16, hw=(H, W),
                      dst=("a", "inc1.0"), dst_off=0, pool=None, keep=True, first=True))
        L.append(dict(name="inc1.3", conv=seq[3], bn=seq[4], act=1, src=("a", "inc1.0"), src_off=0, cin=16, cout=16, hw=(H, W),
                      dst=("a", "inc1.3"), dst_off=0, pool=None, keep=True))
        L += self._double("inc2", m.inc2, ("a", "inc1.3"), 0, 16, 16, (H, W), pool2=("p", 1), keep2=False)
        L += self._double("down1", m.down1.maxpool_conv[1], ("p", 1), 0, 16, 32, (H // 2, W // 2), pool2=("p", 2), keep2=False)
        L += self._double("down2", m.down2.maxpool_conv[1], ("p", 2), 0, 32, 64, (H // 4, W // 4))
        L += self._double("inc3", m.inc3, ("a", "down2.3"), 0, 64, 64, (H // 4, W // 4), dst2=("cat", 3), pool2=("p", 3))
        L += self._double("down3", m.down3.maxpool_conv[1], ("p", 3), 0, 64, 128, (H // 8, W // 8), dst2=("cat", 2), pool2=("p", 4))
        L += self._double("down4", m.down4.maxpool_conv[1], ("p", 4), 0, 128, 256, (H // 16, W // 16), dst2=("cat", 1), pool2=("p", 5))
        L += self._double("down5", m.down5.maxpool_conv[1], ("p", 5), 0, 256, 512, (H // 32, W // 32))
        L.append(dict(name="up1.up", up=m.up1.up, src=("a", "down5.3"), cin=512, cout=256, hw=(H // 32, W // 32), dst=("cat", 1), dst_off=32))
        L += self._double("up1.conv", m.up1.conv, ("cat", 1), 0, 512, 256, (H // 16, W // 16))
        L.append(dict(name="up2.up", up=m.up2.up, src=("a", "up1.conv.3"), cin=256, cout=128, hw=(H // 16, W // 16), dst=("cat", 2), dst_off=16))
        L += self._double("up2.conv", m.up2.conv, ("cat", 2), 0, 256, 128, (H // 8, W // 8))
        L.append(dict(name="up3.up", up=m.up3.up, src=("a", "up2.conv.3"), cin=128, cout=64, hw=(H // 8, W // 8), dst=("cat", 3), dst_off=8))
        L += self._double("up3.conv", m.up3.conv, ("cat", 3), 0, 128, 128, (H // 4, W // 4))
        L += self._double("dconv1", m.dconv1, ("a", "up3.conv.3"), 0, 128, 128, (H // 4, W // 4))
        L += self._double("dconv2", m.dconv2, ("a", "dconv1.3"), 0, 128, 128, (H // 4, W // 4))
        return L

    def _shape_of(self, ref, B, H, W):
        kind, key = ref
        if kind == "p":
            c = {1: 16, 2: 32, 3: 64, 4: 128, 5: 256}[key]
            s = 2 ** key
            return (B, c // 8, H // s, W // s, 8)
        if kind == "cat":
            c = {3: 128, 2: 256, 1: 512}[key]
            s = {3: 4, 2: 8, 1: 16}[key]
            return (B, c // 8, H // s, W // s, 8)
        raise KeyError(ref)

    def _tensor(self, ref, B, H, W, shape=None, grad=False):
        kind, key = ref
        name = ("g:" if grad else "") + f"{kind}:{key}"
        if shape is None or kind in ("p", "cat"):
            shape = self._shape_of(ref, B, H, W)
        return self.buf(name, shape, zero=grad and kind == "cat")

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, x):
        m = self.m
        if not x.is_cuda:
            raise RuntimeError("abcnet_b200 training forward needs a CUDA tensor (no CPU fallback)")
        _lib.require_device()
        if x.dim() != 4 or x.shape[1] != m.n_channels or x.shape[2] % 32 or x.shape[3] % 32:
            raise ValueError(f"expected [B,{m.n_channels},H,W] with H, W multiples of 32, got {tuple(x.shape)}")
        u8 = x.dtype in (torch.uint8, torch.bool) and m.n_channels == 1
        x = x.contiguous().view(torch.uint8) if u8 else x.contiguous().float()
        B, _, H, W = x.shape
        plan = self._plan(H, W)
        m.invalidate_packed()                                        # the eval-mode weight cache is stale after any training pass
        self._sync_arena()
        # dropout stream: a device-resident counter, advanced by a device op so that CUDA-graph replays draw new masks
        seed_t = self.bufs.get("seed")
        if seed_t is None:
            seed_t = self.bufs["seed"] = torch.full((1,), _initial_dropout_seed(), dtype=torch.int64, device=x.device)
        seed_t.add_(0x5DEECE66D)
        fuse = bool(getattr(m, "fuse_bn", True)) and not os.environ.get("ABCNET_NO_BN_FUSE")
        sv = self.saved = dict(x=x, u8=u8, B=B, H=H, W=W, plan=plan, units={}, seed=seed_t, fuse=fuse)
        for u in plan:
            h, w = u["hw"]
            if "up" in u:                                            # up-sampling conv: 4 sub-pixel phases, bias, no BN
                src = self._tensor(u["src"], B, H, W, (B, u["cin"] // 8, h, w, 8))
                cat = self._tensor(u["dst"], B, H, W)

                def make(up=u["up"], cout=u["cout"]):
                    # the four sub-pixel phases as blocks of the GEMM N axis (AbcConvDesc.subpixel): one launch, zero blocks where
                    # a phase does not use an input offset (same layout as UNet._pack_subpixel)
                    wt = self._w(up.weight)
                    offs = sorted({(dy, dx) for py in (0, 1) for px in (0, 1) for (_, dy) in phase_taps(py, m.crop_first)
                                   for (_, dx) in phase_taps(px, m.crop_first)})
                    mats = wt.new_zeros(len(offs), 4 * cout, wt.shape[0])
                    for py in (0, 1):
                        for px in (0, 1):
                            ph = 2 * py + px
                            for (ky, dy) in phase_taps(py, m.crop_first):
                                for (kx, dx) in phase_taps(px, m.crop_first):
                                    mats[offs.index((dy, dx)), ph * cout:(ph + 1) * cout] = wt[:, :, ky, kx].t()
                    pk = Packed(mats, self._w(up.bias).repeat(4), offs, n_tile=256 if cout % 64 == 0 else 128)
                    pk.subpixel = cout
                    return pk
                conv(self._pk(u["name"] + ".sub", make), src, 0, cat, out_plane_off=u["dst_off"], out_scale=(2, 0, 2, 0))
                continue
            cout = u["cout"]
            z = self.buf("z:" + u["name"], (B, cout // 8, h, w, 8))
            fused_stats = False
            if u.get("first"):                                       # direct kernel, raw conv + bias (BN / ReLU follow)
                w9 = u["conv"].weight.detach().float().reshape(16, m.n_channels * 9).contiguous()
                bias = u["conv"].bias.detach().float()
                if m.n_channels == 1:
                    check(lib.abc_conv3x3_c1_raw(x.data_ptr(), 1 if u8 else 0, w9.data_ptr(), bias.data_ptr(), z.data_ptr(), B, h, w, 2, 0,
                                                 _st()), "abc_conv3x3_c1_raw")
                else:
                    check(lib.abc_conv3x3_cn(x.data_ptr(), m.n_channels, w9.data_ptr(), bias.data_ptr(), z.data_ptr(), B, h, w, 2, 0, 0,
                                             _st()), "abc_conv3x3_cn")
            else:
                src = self._tensor(u["src"], B, H, W, (B, u["cin"] // 8, h, w, 8))

                def make(cv=u["conv"], cin=u["cin"], cout=cout):
                    wt = self._w(cv.weight)
                    mats = torch.stack([wt[:, :, dy + 1, dx + 1] for dy, dx in TAPS3])
                    js = swap_fold_for(cin, cout)                      # train-mode convolutions write plain maps (pooling is in bn_act)
                    return Packed(mats, self._w(cv.bias), TAPS3, fold=js or row_fold_for(cin, cout), fold_swap=bool(js))
                pk = self._pk(u["name"], make)
                fused_stats = fuse and can_fuse_stats(pk, z)
                conv(pk, src, u["src_off"], z, stats=self._stat_bufs("bn:" + u["name"], cout) if fused_stats else None, ws=self._ws())
            dst = self._tensor(u["dst"], B, H, W, (B, cout // 8, h, w, 8)) if u["keep"] or u["dst"][0] == "cat" else None
            pool = self._tensor(u["pool"], B, H, W) if u["pool"] else None
            bn = u["bn"]
            st = self._bn_forward("bn:" + u["name"], z, 0, cout, (bn.weight, bn.bias, bn.running_mean, bn.running_var), 1,
                                  dst, u["dst_off"], pool, 0.0, None, have_stats=fused_stats)
            bn.num_batches_tracked += 1
            sv["units"][u["name"]] = dict(z=z, st=st)
        # heads: fused conv1 (N = 128 * heads) -> BN -> LeakyReLU -> Dropout -> per-head 1x1
        trunk = self._tensor(("a", "dconv2.3"), B, H, W, (B, 16, H // 4, W // 4, 8))
        nh = len(m.heads)
        zh = self.buf("z:heads", (B, 16 * nh, H // 4, W // 4, 8))

        # n-tile 128 = operand-swap mode with the BatchNorm statistics fused into the epilogue: 38.9 -> 38.5 ms per step against the
        # n-tile 256 launch + a separate 0.33 ms statistics pass (A/B on one box, round 2); ABCNET_TRAIN_HEADS_NT256=1 restores that
        def make_h1():
            w1 = torch.cat([self._w(om.conv1.weight) for om in m.out_modules], 0)
            b1 = torch.cat([self._w(om.conv1.bias) for om in m.out_modules])
            return Packed(torch.stack([w1[:, :, dy + 1, dx + 1] for dy, dx in TAPS3]), b1, TAPS3,
                          n_tile=256 if ((128 * nh) % 256 == 0 and os.environ.get("ABCNET_TRAIN_HEADS_NT256")) else 128)
        pk_h1 = self._pk("heads.conv1", make_h1)
        h1_stats = fuse and can_fuse_stats(pk_h1, zh)
        conv(pk_h1, trunk, 0, zh, stats=self._stat_bufs("bn:heads", 128 * nh) if h1_stats else None, ws=self._ws())
        gam = torch.cat([om.bn.weight.detach() for om in m.out_modules]).float().contiguous()
        bet = torch.cat([om.bn.bias.detach() for om in m.out_modules]).float().contiguous()
        rme = torch.cat([om.bn.running_mean for om in m.out_modules]).float().contiguous()
        rva = torch.cat([om.bn.running_var for om in m.out_modules]).float().contiguous()
        hid = self.buf("a:hid", (B, 16 * nh, H // 4, W // 4, 8))
        p_drop = float(m.dropout_p)
        st = self._bn_forward("bn:heads", zh, 0, 128 * nh, (gam, bet, rme, rva), 2, hid, 0, None, p_drop, sv["seed"], have_stats=h1_stats)
        for i, om in enumerate(m.out_modules):                       # write the updated running statistics back
            om.bn.running_mean.copy_(rme[128 * i:128 * (i + 1)])
            om.bn.running_var.copy_(rva[128 * i:128 * (i + 1)])
            om.bn.num_batches_tracked += 1
        sv["heads"] = dict(z=zh, st=st, hid=hid, trunk=trunk, p_drop=p_drop)
        outs = []
        for i, (h_, om) in enumerate(zip(m.heads, m.out_modules)):
            o = torch.empty((B, h_, H // 4, W // 4), dtype=torch.float32, device=x.device)
            n_tile = 16 if h_ <= 16 else (64 if h_ <= 64 else 128)

            def make_h2(om=om, h_=h_, n_tile=n_tile):
                w2 = self._w(om.conv2.weight).reshape(h_, -1)
                return Packed(w2.unsqueeze(0).contiguous(), self._w(om.conv2.bias), [(0, 0)], n_tile=n_tile)
            conv(self._pk(f"heads.{i}.conv2", make_h2), hid, 16 * i, o, out_mode=1)
            outs.append(o)
        return outs

    # ------------------------------------------------------------------ backward
    @torch.no_grad()
    def head_grad_buffers(self):
        """The bf16 P8 gradient operands and fp64 bias-gradient vectors of the eight heads (the buffers ``backward`` itself uses): a
        loss that writes them directly (loss.loss_forward_p8) passes them back as ``backward(None, sink, head_scale, p8=...)``."""
        from .loss import head_grad_planes
        sv = self.saved
        B, H4, W4 = sv["B"], sv["H"] // 4, sv["W"] // 4
        dl = [self.buf(f"g:logit{i}", (B, head_grad_planes(h_), H4, W4, 8)) for i, h_ in enumerate(self.m.heads)]
        db = [self.buf(f"g:bias{i}", (h_,), torch.float64) for i, h_ in enumerate(self.m.heads)]
        return dl, db

    @torch.no_grad()
    def backward(self, dlogits, sink, head_scale=None, p8=None):
        """dlogits: 8 fp32 NCHW gradients (times ``head_scale[i]``, an fp32 device tensor [8], when given).
        ``p8 = head_grad_buffers()`` already filled with the UNSCALED gradient (dlogits is ignored; head_scale required): the
        factor is applied to the head weight / bias gradients and, per channel, inside the BatchNorm backward of the heads.
        ``sink(param, grad_tensor)`` receives every parameter gradient as soon as it is complete (reverse layer order)
        -- e.g. GradBuckets-aware accumulation."""
        m, sv = self.m, self.saved
        B, H, W = sv["B"], sv["H"], sv["W"]
        H4, W4 = H // 4, W // 4
        ws = self._ws()
        dev = sv["x"].device
        hd = sv["heads"]
        nh = len(m.heads)
        dhid = self.buf("g:hid", (B, 16 * nh, H4, W4, 8))
        if p8 is not None and head_scale is None:
            raise ValueError("backward(p8=...): the unscaled P8 gradient needs head_scale")
        for i, (h_, om) in enumerate(zip(m.heads, m.out_modules)):
            c16 = (h_ + 15) // 16 * 16 if h_ <= 64 else (h_ + 63) // 64 * 64     # K of the data-gradient GEMM
            dl = self.buf(f"g:logit{i}", (B, c16 // 8, H4, W4, 8))
            db = self.buf(f"g:bias{i}", (h_,), torch.float64)
            if p8 is not None:
                if p8[0][i].data_ptr() != dl.data_ptr() or p8[1][i].data_ptr() != db.data_ptr():
                    raise ValueError("backward(p8=...): pass the buffers of head_grad_buffers()")
            else:
                g = dlogits[i]
                if g is None:
                    g = torch.zeros((B, h_, H4, W4), dtype=torch.float32, device=dev)
                g = g.contiguous().float()
                # one pass: (optional per-head loss scale) * dlogits -> bf16 P8 with zero K padding, + conv2 bias gradient
                sc = head_scale[i:i + 1].data_ptr() if head_scale is not None else None
                if ws is not None:
                    w_ = ws(lib.abc_nchw_to_p8_ex_workspace_bytes(B, h_, H4, W4, c16 // 8))
                    check(lib.abc_nchw_to_p8_ex_det(g.data_ptr(), dl.data_ptr(), B, h_, H4, W4, c16 // 8, sc, db.data_ptr(), w_.data_ptr(),
                                                    _st()), "abc_nchw_to_p8_ex_det")
                else:
                    check(lib.abc_nchw_to_p8_ex(g.data_ptr(), dl.data_ptr(), B, h_, H4, W4, c16 // 8, sc, db.data_ptr(), _st()),
                          "abc_nchw_to_p8_ex")
            c8 = (h_ + 7) // 8 * 8
            dw2 = wgrad(dl, 0, c8, hd["hid"], 16 * i, 128, [(0, 0)], ws=ws)[0][:h_]
            dbf = db.float()
            if p8 is not None:                                    # the factor the loss kernel left out (linear in the gradient)
                dw2 = dw2 * head_scale[i]
                dbf = dbf * head_scale[i]
            sink(om.conv2.weight, dw2.reshape(h_, 128, 1, 1))
            sink(om.conv2.bias, dbf)
            def make_d2(om=om, h_=h_, c16=c16):
                w2 = self._w(om.conv2.weight).reshape(h_, 128)
                w2p = torch.cat([w2, w2.new_zeros(c16 - h_, 128)], 0)        # K = padded logits channels
                return Packed(w2p.t().contiguous().unsqueeze(0), self._zeros(128), [(0, 0)], n_tile=128)
            conv(self._pk(f"heads.{i}.conv2.dgrad", make_d2), dl, 0, dhid, out_plane_off=16 * i)
        dzh = self.buf("g:zheads", (B, 16 * nh, H4, W4, 8))
        gscale = head_scale.float().view(-1, 1).expand(-1, 128).reshape(-1).contiguous() if p8 is not None else None    # per hidden channel
        s1, s2 = self._bn_backward("bn:heads", hd["z"], 128 * nh, hd["st"], 2, dhid, 0, None, dzh, hd["p_drop"], sv["seed"], gscale=gscale)
        dw1 = wgrad(dzh, 0, 128 * nh, hd["trunk"], 0, 128, TAPS3, ws=ws)     # [9][128*nh][128]
        for i, om in enumerate(m.out_modules):
            sl = slice(128 * i, 128 * (i + 1))
            sink(om.conv1.weight, dw1[:, sl].permute(1, 2, 0).reshape(128, 128, 3, 3))
            sink(om.conv1.bias, torch.zeros(128, device=dev))
            sink(om.bn.weight, s2[sl].float())
            sink(om.bn.bias, s1[sl].float())
        g_trunk = self._tensor(("a", "dconv2.3"), B, H, W, (B, 16, H4, W4, 8), grad=True)
        def make_d1():
            w1 = torch.cat([self._w(om.conv1.weight) for om in m.out_modules], 0)
            mats = torch.stack([w1[:, :, dy + 1, dx + 1].t() for dy, dx in TAPS3]).contiguous()   # [9][ci=128][co=1024]
            return Packed(mats, self._zeros(128), [(-dy, -dx) for dy, dx in TAPS3], n_tile=128)
        conv(self._pk("heads.conv1.dgrad", make_d1), dzh, 0, g_trunk)

        for u in reversed(sv["plan"]):
            h, w = u["hw"]
            if "up" in u:
                gcat = self._tensor(u["dst"], B, H, W, grad=True)
                xin = self._tensor(u["src"], B, H, W, (B, u["cin"] // 8, h, w, 8))
                wt = u["up"].weight.detach().float()
                dx, dwu = upconv_backward(gcat, u["dst_off"], u["cout"], xin, wt, m.crop_first,
                                          eng=self if self.arena is not None else None, key=(u["name"] + ".dgrad", u["up"].weight), ws=ws)
                sink(u["up"].weight, dwu)
                sm = self.buf("up.sum", (u["cout"],), torch.float64)
                sq = self.buf("up.sq", (u["cout"],), torch.float64)
                if ws is not None:
                    w_ = ws(lib.abc_bn_stats_workspace_bytes(B, 2 * h, 2 * w, u["cout"]))
                    check(lib.abc_channel_sum_det(gcat.data_ptr(), B, 2 * h, 2 * w, gcat.shape[1], u["dst_off"], u["cout"], sm.data_ptr(),
                                                  sq.data_ptr(), w_.data_ptr(), _st()), "abc_channel_sum_det")
                else:
                    check(lib.abc_channel_sum(gcat.data_ptr(), B, 2 * h, 2 * w, gcat.shape[1], u["dst_off"], u["cout"], sm.data_ptr(),
                                              sq.data_ptr(), _st()), "abc_channel_sum")
                sink(u["up"].bias, sm.float())
                gsrc = self._tensor(u["src"], B, H, W, (B, u["cin"] // 8, h, w, 8), grad=True)
                gsrc.copy_(dx)
                continue
            cout, cin = u["cout"], u["cin"]
            su = sv["units"][u["name"]]
            dA = None
            if u["keep"] or u["dst"][0] == "cat":
                dA = self._tensor(u["dst"], B, H, W, (B, cout // 8, h, w, 8), grad=True)
            dP = self._tensor(u["pool"], B, H, W, grad=True) if u["pool"] else None
            dz = self.buf("g:z:" + u["name"], (B, cout // 8, h, w, 8))
            s1, s2 = self._bn_backward("bn:" + u["name"], su["z"], cout, su["st"], 1, dA, u["dst_off"] if dA is not None else 0, dP, dz, 0.0, None)
            sink(u["bn"].weight, s2.float())
            sink(u["bn"].bias, s1.float())
            sink(u["conv"].bias, torch.zeros(cout, device=dev))
            if u.get("first"):
                dwf = torch.zeros(144 * m.n_channels, dtype=torch.float32, device=dev)
                if ws is not None:
                    w_ = ws(lib.abc_conv3x3_wgrad_workspace_bytes(m.n_channels))
                    if m.n_channels == 1:
                        check(lib.abc_conv3x3_c1_wgrad_det(sv["x"].data_ptr(), 1 if sv["u8"] else 0, dz.data_ptr(), 2, 0, B, h, w, dwf.data_ptr(),
                                                           w_.data_ptr(), _st()), "abc_conv3x3_c1_wgrad_det")
                    else:
                        check(lib.abc_conv3x3_cn_wgrad_det(sv["x"].data_ptr(), m.n_channels, dz.data_ptr(), 2, 0, B, h, w, dwf.data_ptr(),
                                                           w_.data_ptr(), _st()), "abc_conv3x3_cn_wgrad_det")
                elif m.n_channels == 1:
                    check(lib.abc_conv3x3_c1_wgrad(sv["x"].data_ptr(), 1 if sv["u8"] else 0, dz.data_ptr(), 2, 0, B, h, w, dwf.data_ptr(), _st()),
                          "abc_conv3x3_c1_wgrad")
                else:
                    check(lib.abc_conv3x3_cn_wgrad(sv["x"].data_ptr(), m.n_channels, dz.data_ptr(), 2, 0, B, h, w, dwf.data_ptr(), _st()),
                          "abc_conv3x3_cn_wgrad")
                sink(u["conv"].weight, dwf.reshape(16, m.n_channels, 3, 3))
                continue
            src = self._tensor(u["src"], B, H, W, (B, cin // 8, h, w, 8))
            dwt = wgrad(dz, 0, cout, src, u["src_off"], cin, TAPS3, ws=ws)        # [9][cout][cin]
            sink(u["conv"].weight, dwt.permute(1, 2, 0).reshape(cout, cin, 3, 3))
            gsrc = self._tensor(u["src"], B, H, W, (B, cin // 8, h, w, 8), grad=True)
            def make_d(cv=u["conv"], cin=cin, cout=cout):
                wt = self._w(cv.weight)
                mats = torch.stack([wt[:, :, dy + 1, dx + 1].t() for dy, dx in TAPS3]).contiguous()    # [9][ci][co]
                js = swap_fold_for(cout, cin)
                return Packed(mats, self._zeros(cin), [(-dy, -dx) for dy, dx in TAPS3], fold=js or row_fold_for(cout, cin), fold_swap=bool(js))
            conv(self._pk(u["name"] + ".dgrad", make_d), dz, 0, gsrc, out_plane_off=u["src_off"])

class _UNetTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, x, *params):
        eng = model._train_engine()
        outs = eng.forward(x)
        ctx.model, ctx.eng, ctx.n_params = model, eng, len(params)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *dlogits):
        model = ctx.model
        params = [p for p in model.parameters()]
        index = {id(p): i for i, p in enumerate(params)}
        grads = [None] * len(params)
        buckets = getattr(model, "grad_buckets", None)

        def sink(p, g):
            if not p.requires_grad:
                return
            if buckets is not None:                      # gradient lives in a contiguous bucket; notify for overlapped all-reduce
                p.grad.add_(g.to(p.grad.dtype).view_as(p.grad))
                buckets.grad_ready(p)
            else:
                grads[index[id(p)]] = g.to(p.dtype).reshape(p.shape)

        ctx.eng.backward(list(dlogits), sink)
        return (None, None) + tuple(grads)
