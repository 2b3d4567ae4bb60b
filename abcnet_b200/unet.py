"""Host-side mirror of the reference model interface, driving the sm_100a kernels through the C-ABI.

Drop-in for ``from unet import UNet`` of the reference (``/root/reference/src/unet.py:77-119``):

    model = UNet(in_channels=1, heads=[1, 14, 3, 2, 1, 360, 60, 60])
    outs = model(imgs)            # list of len(heads) contiguous fp32 NCHW tensors [B, heads[i], H/4, W/4]

* same constructor signature, same ``state_dict()`` keys / shapes (261 entries for the v2 heads, loadable with or
  without the ``module.`` prefix written by ``train.py:435``), same ``model.s`` parameter (``unet.py:82``);
* ``eval()`` forward = BatchNorm folded into the convolutions at (re)load time, bf16 activations in the planar-8
  layout, fp32 accumulation in TMEM, fp32 logits out;
* no CPU fallback and no PyTorch/cuDNN compute on this path: every layer is one of the kernels behind
  ``include/abcnet_b200.h``. A CPU tensor, a missing library or a non-sm_100 device raises.

The parameters live in plain torch containers only so that checkpoints, optimizers and DDP wrappers keep working.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict

import torch
import torch.nn as nn

from . import _lib
from ._lib import AbcConvDesc, AbcHeadsFusedDesc, check, lib

BN_EPS = 1e-5
_TAPS3 = [(ky - 1, kx - 1, ky, kx) for ky in range(3) for kx in range(3)]          # (dy, dx, ky, kx)


def _bn(c):
    return nn.BatchNorm2d(c)


def _conv_bn_pair(cin, cout):
    """Parameter container with the reference's key names '<prefix>.double_conv.{0,1,3,4}.*' (unet.py:11-18)."""
    holder = nn.Module()
    holder.double_conv = nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), _bn(cout), nn.ReLU(inplace=True),
                                       nn.Conv2d(cout, cout, 3, padding=1), _bn(cout), nn.ReLU(inplace=True))
    return holder


def _down(cin, cout):
    holder = nn.Module()                                   # keys '<prefix>.maxpool_conv.1.double_conv.*' (unet.py:29-32)
    holder.maxpool_conv = nn.Sequential(nn.MaxPool2d(2), _conv_bn_pair(cin, cout))
    return holder


def _up(cin, cout):
    holder = nn.Module()                                   # keys '<prefix>.up.*', '<prefix>.conv.double_conv.*' (unet.py:44-46)
    holder.up = nn.ConvTranspose2d(cin, cin // 2, kernel_size=3, stride=2)
    holder.conv = _conv_bn_pair(cin, cout)
    return holder


def _head(cin, cout):
    holder = nn.Module()                                   # keys 'out_modules.i.{conv1,bn,conv2}.*' (unet.py:66-70)
    holder.conv1 = nn.Conv2d(cin, cin, 3, padding=1)
    holder.bn = _bn(cin)
    holder.conv2 = nn.Conv2d(cin, cout, 1)
    return holder


def row_fold_for(cin, cout):
    """Row-folding factor of a 3x3 layer (include/abcnet_b200.h, AbcConvDesc.row_fold): the 16 / 32-channel layers are
    bound by the shared-memory operand fetch of their small-N MMAs; folding J rows into the GEMM N axis (N = J * cout = 64)
    cuts the MMA count per pixel by 3J / (J + 2)."""
    if os.environ.get("ABCNET_NO_FOLD"):
        return 1
    if cout == 16 and cin <= 32:
        return 4
    if cout == 32 and cin <= 32:
        return 2
    return 1


def k_chunk_for(cin):
    """Channels per pipeline stage (AbcConvDesc.k_chunk). Default min(cin, 64); ABCNET_KC64=32 selects 32 for the cin = 64
    layers (experiment: deeper rings for the pipeline-depth-bound 64-channel layers at 128 x 128)."""
    if cin == 64 and os.environ.get("ABCNET_KC64"):
        return int(os.environ["ABCNET_KC64"])
    return min(cin, 64)


def use_cta_pair(cin, ntaps, n_tile):
    """CTA-pair (cta_group::2) mode for the layers whose weights of one n-tile do not fit in shared memory and are streamed
    (Cin >= 128 3x3 layers, the 8-head conv1, the large up-sampling phases): see AbcConvDesc.cta_pair.
    Opt-in (ABCNET_PAIR=1). Measured on B200 (tools/layer_bench.py pair / pairdbg): bit-identical results, but the peer CTA
    reports "operands landed" to the leader through a relayed mbarrier arrival per weight block, which costs ~1300 clk per
    block and makes the mode 1.4 - 1.8x slower; with that relay removed (timing experiment only) the pair mode merely ties
    the single-CTA kernel (7.7 vs 7.3 ms for the 8-head conv1, 1.01 vs 1.05 ms for 128 -> 128 @128x128): these layers sit
    at ~95 % / ~85 % of the cuBLAS bf16 rate the 1 kW power cap sustains, not on a shared-memory or L2 limit."""
    if os.environ.get("ABCNET_PAIR", "0") != "1":
        return False
    return cin % 64 == 0 and n_tile % 32 == 0 and cin * ntaps * n_tile * 2 > 160 * 1024


def swap_fold_for(cin, cout, plain_output=True):
    """Row folding combined with the operand swap for the 32- and 64-channel 3x3 layers whose output is a plain P8 map:
    J = 128 / cout vertically adjacent pixels share one pixel column and the 128 GEMM rows are (row j, channel) -- one
    M = 128 x N = 256 MMA per (tap, 16 channels) covers 256 * J pixels with 3 (J + 2) taps instead of 9 J.
    Returns J (0 = not applicable). ABCNET_NO_SWAP / ABCNET_NO_FOLD disable."""
    if os.environ.get("ABCNET_NO_SWAP") or os.environ.get("ABCNET_NO_FOLD") or os.environ.get("ABCNET_NO_SWAPFOLD") or not plain_output:
        return 0
    J = {64: 2, 32: 4}.get(cout, 0)
    if J == 4 and cin > 32:          # a 128-row halo tile of 64 channels (166 KB per pipeline stage) does not fit twice in shared memory
        return 0
    return J


def use_swap(pk, out_mode, dst, pool):
    """Operand-swap mode (AbcConvDesc.swap_mn) for the launches whose n-tile is exactly 128 output channels and whose output is
    a plain bf16 P8 map: the mid-U-Net 128 -> 128 layers, the cout = 128 decoder layers, their data gradients and the data
    gradient of the 8-head conv1. One N = 256-pixel MMA replaces two N = 128-channel ones. ABCNET_NO_SWAP=1 disables."""
    if os.environ.get("ABCNET_NO_SWAP"):
        return False
    return (pk.n_tile == 128 and (pk.fold == 1 or getattr(pk, "fold_swap", False)) and not pk.pair
            and not getattr(pk, "segments", None) and out_mode == 0 and dst is not None and pool is None)


def pair_pack(w_taps, n_tiles, n_tile):
    """Weight blocks of the CTA-pair mode: [n_tiles][cin/64][ntaps][2 halves][n_tile/2 rows][64 channels], each row 128-byte
    swizzled (16-byte chunk c of row r at chunk position c ^ (r % 8)); w_taps: [ntaps, n_tiles * n_tile, cin] fp32."""
    ntaps, _, cin = w_taps.shape
    w = w_taps.view(ntaps, n_tiles, 2, n_tile // 16, 8, cin // 64, 8, 8)          # [t][nt][half][row group][r8][chunk][c][e]
    r8 = torch.arange(8, device=w_taps.device).view(8, 1)
    pos = torch.arange(8, device=w_taps.device).view(1, 8)
    src = (pos ^ r8).view(1, 1, 1, 1, 8, 1, 8, 1).expand(ntaps, n_tiles, 2, n_tile // 16, 8, cin // 64, 8, 8)
    w = torch.gather(w, 6, src)                                                     # out[..., r8, :, pos, :] = in[..., r8, :, pos ^ r8, :]
    return w.permute(1, 5, 0, 2, 3, 4, 6, 7)                                        # [nt][chunk][t][half][row group][r8][pos][e]


def fold_rows_swap(w_taps, bias, taps, J):
    """Toeplitz expansion along y for the operand-swap kernel: like ``fold_rows`` but GEMM row m = j * cout + co
    (AbcConvDesc.swap_mn with row_fold). Returns (w [3 (J + 2), J * cout, cin], bias [J * cout])."""
    ntaps, cout, cin = w_taps.shape
    assert ntaps == 9 and J * cout == 128 and sorted(taps) == sorted((dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    by_off = {t: w_taps[i] for i, t in enumerate(taps)}
    out = w_taps.new_zeros(3 * (J + 2), J, cout, cin)
    for r in range(J + 2):
        for c in range(3):
            for j in range(J):
                dy = r - 1 - j
                if -1 <= dy <= 1:
                    out[r * 3 + c, j] = by_off[(dy, c - 1)]
    return out.view(3 * (J + 2), J * cout, cin), bias.view(1, cout).expand(J, cout).reshape(-1)


def fold_rows(w_taps, bias, taps, J):
    """Toeplitz expansion along y of a 3x3 kernel: w_taps [9, cout, cin] for ``taps`` (dy, dx) -> folded
    [3 * (J + 2), J * cout, cin] in (row offset r, column offset c) order, column n = (b * J + j) * 16 + i for output
    channel 16 b + i of folded row j; tap (r, c) contributes W[(dy = r - 1 - j, dx = c - 1)]. Returns (w, bias)."""
    ntaps, cout, cin = w_taps.shape
    assert ntaps == 9 and cout % 16 == 0 and sorted(taps) == sorted((dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    by_off = {t: w_taps[i] for i, t in enumerate(taps)}
    out = w_taps.new_zeros(3 * (J + 2), cout // 16, J, 16, cin)
    for r in range(J + 2):
        for c in range(3):
            for j in range(J):
                dy = r - 1 - j
                if -1 <= dy <= 1:
                    out[r * 3 + c, :, j] = by_off[(dy, c - 1)].view(cout // 16, 16, cin)
    b = bias.view(cout // 16, 1, 16).expand(cout // 16, J, 16).reshape(-1)
    return out.view(3 * (J + 2), J * cout, cin), b


class _Packed:
    """Device-resident, kernel-ready form of one convolution: packed bf16 weights + fp32 bias + tap list."""

    def __init__(self, w_taps, bias, taps, n_tile, cout, fold=1, pair=None, fold_swap=False, kc=None, dtype=torch.bfloat16):
        # w_taps: fp32 [ntaps, cout, cin] (already BN-folded); taps: list of (dy, dx)
        # pair: CTA-pair mode (AbcConvDesc.cta_pair); None = decide from the layer size (weights too large to stay resident)
        # fold_swap: row folding in the row order of the operand-swap kernel (the launch must then use swap_mn)
        self.fold, self.fold_swap = fold, bool(fold_swap) and fold > 1
        if fold > 1:
            w_taps, bias = (fold_rows_swap if fold_swap else fold_rows)(w_taps, bias, taps, fold)
            n_tile = fold * cout
        ntaps, co, cin = w_taps.shape
        kc = kc or k_chunk_for(cin)
        self.kc = kc
        n_tiles = (cout + n_tile - 1) // n_tile
        pad = n_tiles * n_tile - co
        if pad:
            w_taps = torch.cat([w_taps, w_taps.new_zeros(ntaps, pad, cin)], 1)
            bias = torch.cat([bias, bias.new_zeros(pad)])
        if pair is None:
            pair = use_cta_pair(cin, ntaps, n_tile) and fold == 1
        self.pair = bool(pair)
        if self.pair:      # every (n-tile, chunk, tap) block as two halves of n_tile / 2 rows: one per CTA of the pair
            w = pair_pack(w_taps, n_tiles, n_tile)
        else:
            w = w_taps.view(ntaps, n_tiles, n_tile, cin // kc, kc // 8, 8).permute(1, 3, 0, 4, 2, 5)
        self.fp16 = dtype == torch.float16            # AbcConvDesc.act_fp16: weights AND activations of the launch are fp16
        self.w = (w.contiguous().clamp(-65504.0, 65504.0) if self.fp16 else w.contiguous()).to(dtype)
        assert self.w.numel() * 2 == lib.abc_conv_wpack_bytes(cin, co, ntaps, n_tile)
        self.bias = bias.contiguous().float()
        self.taps, self.n_tile, self.cout, self.cin = taps, n_tile, cout, cin


def _fold(conv_w, conv_b, bn):
    """Inference BatchNorm fold (SURVEY App. A.2): W' = W * g / sqrt(var + eps), b' = (b - mean) * g / sqrt(var + eps) + beta."""
    # sqrt through fp64 and back = the correctly rounded fp32 sqrt on every backend (CUDA's sqrtf already is; torch's vectorised CPU
    # sqrt is not always), so the packs are the same bytes wherever they are built -- and the same as csrc/unet_plan.cu's sqrtf
    scale = bn.weight.detach().float() / torch.sqrt((bn.running_var.detach().float() + bn.eps).double()).float()
    w = conv_w.detach().float() * scale.view(-1, 1, 1, 1)
    b = (conv_b.detach().float() - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()
    return w, b


def _default_n_tile(cin, cout):
    env = os.environ.get(f"ABCNET_NTILE_{cin}x{cout}")
    if env:
        return int(env)
    c16 = (cout + 15) // 16 * 16
    if c16 <= 128:
        return c16
    return 256 if (cout % 256 == 0 and cin >= 128) else 128


class HeadMaps(list):
    """The 8 head outputs plus their channel counts (needed to interpret planar-8 maps)."""

    def __init__(self, heads):
        super().__init__()
        self.heads = list(heads)

    def to_nchw(self):
        out = []
        for t, h in zip(self, self.heads):
            if t.dim() == 5:
                N, P_, H, W, _ = t.shape
                t = t.permute(0, 1, 4, 2, 3).reshape(N, P_ * 8, H, W)[:, :h].contiguous()
            out.append(t)
        return out


class _LaunchTimer:
    """Context manager recording CUDA events around a launch group when ``model.timing`` is a list."""

    def __init__(self, sink, name):
        self.sink, self.name = sink, name

    def __enter__(self):
        if self.sink is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.sink is not None:
            self.b.record()
            self.sink.append((self.name, self.a, self.b))
        return False


class UNet(nn.Module):
    def __init__(self, in_channels, heads=[1, 21, 5, 1, 4, 2], crop_first=True, act_dtype="bf16"):
        """``act_dtype``: storage format of the eval-mode activations and packed weights. "bf16" (default; the format north_star
        names and the only one the training pass uses) or "fp16": IEEE half, 8 x smaller rounding error per stored value at the
        same tensor-core rate -- the decision-stable inference mode (fewer threshold / NMS / omega ties flip against the fp32
        reference, DESIGN.md section 2); values saturate at +-65504."""
        super().__init__()
        if act_dtype not in ("bf16", "fp16"):
            raise ValueError("act_dtype must be 'bf16' or 'fp16'")
        self.act_dtype = act_dtype
        # in_channels = 1: the binarised drawings of the reference's datasets (utils.py:80-81), table-driven stem kernel;
        # 2..8 real-valued channels (unet.py:127 self-checks in_channels=3): general fp32 stem kernel (abc_conv3x3_cn)
        if not (1 <= int(in_channels) <= 8):
            raise ValueError("abcnet_b200.UNet: in_channels must be in 1..8")
        self.n_channels = int(in_channels)
        self.heads = list(heads)
        # torch >= 1.13 floor-divides the negative crop in unet.py:54-55 -> the FIRST row / column is dropped (SURVEY D1)
        self.crop_first = bool(crop_first)
        self.s = nn.Parameter(torch.randn(10) / 100)
        self.inc1 = _conv_bn_pair(in_channels, 16)
        self.inc2 = _conv_bn_pair(16, 16)
        self.down1 = _down(16, 32)
        self.down2 = _down(32, 64)
        self.inc3 = _conv_bn_pair(64, 64)
        self.down3 = _down(64, 128)
        self.down4 = _down(128, 256)
        self.down5 = _down(256, 512)
        self.up1 = _up(512, 256)
        self.up2 = _up(256, 128)
        self.up3 = _up(128, 128)
        self.dconv1 = _conv_bn_pair(128, 128)
        self.dconv2 = _conv_bn_pair(128, 128)
        self.out_modules = nn.ModuleList([_head(128, h) for h in self.heads])
        self._packed = None
        self._packed_key = None
        self._pack_gen = 0
        self._bufs = {}
        self.timing = None        # set to a list to collect (layer name, start event, end event) per launch group
        self.dropout_p = 0.2      # nn.Dropout(0.2) of OutConv (unet.py:69); train mode only
        self.grad_buckets = None  # optional abcnet_b200.ddp.GradBuckets: gradients are accumulated into its buckets
        self.fuse_bn = True       # training pass: BatchNorm statistics / backward reductions fused into the conv epilogues
        self._engine = None

    # ------------------------------------------------------------------ checkpoints
    def load_state_dict(self, state_dict, strict=True, **kw):
        if any(k.startswith("module.") for k in state_dict):
            state_dict = OrderedDict((k[7:] if k.startswith("module.") else k, v) for k, v in state_dict.items())
        self._packed = None
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def _param_key(self):
        return tuple((p.data_ptr(), p._version) for p in list(self.parameters()) + list(self.buffers()))

    def invalidate_packed(self):
        """Drop the eval-mode cache of BN-folded, packed weights. ``_param_key`` only sees updates that bump a tensor's
        ``_version``; a CUDA-graph replay (``TrainStep`` + ``FusedAdam``) rewrites weights and BatchNorm running statistics
        through raw pointers without doing so, hence the training entry points and every ``train()`` / ``eval()`` mode
        change call this explicitly (train.py:89,218 alternates the two every epoch)."""
        self._packed = None
        self._packed_key = None

    def train(self, mode=True):
        self.invalidate_packed()
        return super().train(mode)

    # ------------------------------------------------------------------ weight preparation (cold path)
    def _dc_layers(self, holder):
        seq = holder.double_conv
        return [(seq[0], seq[1]), (seq[3], seq[4])]

    @property
    def _act_torch_dtype(self):
        return torch.float16 if self.act_dtype == "fp16" else torch.bfloat16

    @torch.no_grad()
    def prepare(self, _inspect_on_cpu=False):
        """Fold BatchNorm (running statistics) and pack every convolution for the kernels. Called lazily by forward.
        ``_inspect_on_cpu``: build the packs from CPU parameters (pure data movement, no kernel) so that tests can compare them
        with the C++ packing of ``abc_unet_pack_host``; the forward pass itself still refuses to run without a CUDA device."""
        dev = self.s.device
        adt = self._act_torch_dtype
        if dev.type != "cuda" and not _inspect_on_cpu:
            raise RuntimeError("abcnet_b200.UNet runs on a CUDA (sm_100) device only; call .cuda() first -- there is no CPU path")
        P = {}

        pooled = {"inc2.3", "down1.3", "inc3.3", "down3.3", "down4.3"}       # layers with a fused 2x2 max-pool output (see trunk())

        def pack3(name, conv, bn):
            w, b = _fold(conv.weight, conv.bias, bn)
            cout, cin = w.shape[:2]
            wt = torch.stack([w[:, :, ky, kx] for (_, _, ky, kx) in _TAPS3])
            js = swap_fold_for(cin, cout, name not in pooled)
            P[name] = _Packed(wt, b, [(dy, dx) for (dy, dx, _, _) in _TAPS3], _default_n_tile(cin, cout), cout,
                              fold=js or row_fold_for(cin, cout), fold_swap=bool(js), dtype=adt)

        # first conv (1 -> 16): direct kernel, fp32 folded weights [16][9]
        c0, b0 = self.inc1.double_conv[0], self.inc1.double_conv[1]
        w, b = _fold(c0.weight, c0.bias, b0)
        P["inc1.0"] = (w.reshape(16, self.n_channels * 9).contiguous(), b.contiguous())        # [16][cin][9]
        pack3("inc1.3", self.inc1.double_conv[3], self.inc1.double_conv[4])
        for name, holder in (("inc2", self.inc2), ("down1", self.down1.maxpool_conv[1]), ("down2", self.down2.maxpool_conv[1]),
                             ("inc3", self.inc3), ("down3", self.down3.maxpool_conv[1]), ("down4", self.down4.maxpool_conv[1]),
                             ("down5", self.down5.maxpool_conv[1]), ("up1.conv", self.up1.conv), ("up2.conv", self.up2.conv),
                             ("up3.conv", self.up3.conv), ("dconv1", self.dconv1), ("dconv2", self.dconv2)):
            (ca, ba), (cb, bb) = self._dc_layers(holder)
            pack3(name + ".0", ca, ba)
            pack3(name + ".3", cb, bb)
        # up-sampling convolutions: 4 sub-pixel phases each (SURVEY App. A.3) -- as ONE launch with the phases as blocks of the
        # GEMM N axis (AbcConvDesc.subpixel), and as four separate launches (kept for comparison: ABCNET_UP_PHASES=1)
        for name, holder in (("up1", self.up1), ("up2", self.up2), ("up3", self.up3)):
            w = holder.up.weight.detach().float()          # [Cin, Cout, 3, 3]
            b = holder.up.bias.detach().float()
            cin, cout = w.shape[:2]
            P[f"{name}.up"] = self._pack_subpixel(w, b)
            for py in (0, 1):
                for px in (0, 1):
                    ys = self._phase_taps(py)
                    xs = self._phase_taps(px)
                    taps = [(dy, dx) for (ky, dy) in ys for (kx, dx) in xs]
                    wt = torch.stack([w[:, :, ky, kx].t() for (ky, dy) in ys for (kx, dx) in xs])
                    P[f"{name}.up.{py}{px}"] = _Packed(wt.contiguous(), b, taps, _default_n_tile(cin, cout), cout, dtype=adt)
        # heads: the eight conv1 share their input -> one GEMM with N = 128 * len(heads); conv2 is a per-head 1x1
        ws, bs = [], []
        for om in self.out_modules:
            w, b = _fold(om.conv1.weight, om.conv1.bias, om.bn)
            ws.append(w)
            bs.append(b)
        w = torch.cat(ws, 0)
        wt = torch.stack([w[:, :, ky, kx] for (_, _, ky, kx) in _TAPS3])
        nt = int(os.environ.get("ABCNET_NTILE_HEADS", "256"))       # N = 256 tiles: measured 1.4x faster than N = 128
        P["heads.conv1"] = _Packed(wt, torch.cat(bs), [(dy, dx) for (dy, dx, _, _) in _TAPS3], nt, w.shape[0], dtype=adt)
        P["heads.conv1.plain"] = P["heads.conv1"] if not P["heads.conv1"].pair else None   # abc_heads_fused reads the unpaired pack
        self._heads_w1 = (wt, torch.cat(bs), w.shape[0])
        self._packed_heads_ntile = nt
        for i, om in enumerate(self.out_modules):
            w2 = om.conv2.weight.detach().float().reshape(om.conv2.weight.shape[0], -1)
            h = w2.shape[0]
            # n-tile of the 1x1 head convolutions (HBM class). Measured stand-alone at B = 256 (tools/layer_bench.py conv2): the
            # small heads run at 6.5 - 6.7 TB/s, 60 channels at 5.4; for 360 channels two tiles of 192 (4.63 TB/s) beat three of
            # 128 (4.36) and two of 256 (3.9): fewer re-reads of the hidden tile at the same padding.
            n_tile = 16 if h <= 16 else (64 if h <= 64 else (128 if h <= 128 else (192 if (h + 191) // 192 * 192 <= (h + 127) // 128 * 128 else 128)))
            P[f"heads.{i}.conv2"] = _Packed(w2.unsqueeze(0).contiguous(), om.conv2.bias.detach().float(), [(0, 0)], n_tile, h, dtype=adt)
        P["heads.fused"] = self._pack_fused_heads(dev)
        self._packed = P
        self._packed_key = self._param_key()
        self._pack_gen += 1                  # consumers that derive their own packs (SparseHeadsPipeline) key on this
        return self

    def _pack_fused_heads(self, dev):
        """conv2 weights / biases in the (head, chunk) order of abc_heads_fused (include/abcnet_b200.h); None when the head list
        is outside the fused kernel's limits (then conv1 and the per-head conv2 run as separate launches)."""
        heads = self.heads
        if len(heads) > 16 or self._packed_heads_ntile != 256:
            return None
        for i in range(0, len(heads), 2):
            pair = heads[i:i + 2]
            chunks = sum((h + 127) // 128 for h in pair)
            cols = sum(sum(((min(h - c0, 128) + 15) // 16) * 16 for c0 in range(0, h, 128)) for h in pair)
            if chunks > 6 or cols > 512:
                return None
        adt = self._act_torch_dtype
        blocks, biases = [], []
        for om, h in zip(self.out_modules, heads):
            w2 = om.conv2.weight.detach().float().reshape(h, -1)
            b2 = om.conv2.bias.detach().float()
            for c0 in range(0, h, 128):
                cnt = min(h - c0, 128)
                nc = (cnt + 15) // 16 * 16
                wb = w2.new_zeros(nc, 128)
                wb[:cnt] = w2[c0:c0 + cnt]
                wb = wb.view(nc, 16, 8).permute(1, 0, 2).contiguous()
                blocks.append((wb.clamp(-65504.0, 65504.0) if adt == torch.float16 else wb).to(adt).reshape(-1))   # as _Packed
                bb = b2.new_zeros(nc)
                bb[:cnt] = b2[c0:c0 + cnt]
                biases.append(bb)
        w2pack = torch.cat(blocks).contiguous()
        bias2 = torch.cat(biases).contiguous()
        nb, nl = C.c_int64(0), C.c_int(0)
        check(lib.abc_heads_fused_pack_sizes(len(heads), (C.c_int * len(heads))(*heads), C.byref(nb), C.byref(nl)), "abc_heads_fused_pack_sizes")
        assert w2pack.numel() * 2 == nb.value and bias2.numel() == nl.value
        return w2pack, bias2

    def _pack_subpixel(self, w, b):
        """All four sub-pixel phases of ConvTranspose2d(k3, s2) + crop as one N = 4 * cout GEMM over the union of the phases'
        input offsets: w [Cin, Cout, 3, 3] -> taps [(dy, dx)], weights [ntaps, 4 * cout, cin] with zero blocks."""
        cin, cout = w.shape[:2]
        offs = sorted({(dy, dx) for py in (0, 1) for px in (0, 1) for (_, dy) in self._phase_taps(py) for (_, dx) in self._phase_taps(px)})
        wt = w.new_zeros(len(offs), 4 * cout, cin)
        for py in (0, 1):
            for px in (0, 1):
                ph = 2 * py + px
                for (ky, dy) in self._phase_taps(py):
                    for (kx, dx) in self._phase_taps(px):
                        wt[offs.index((dy, dx)), ph * cout:(ph + 1) * cout] = w[:, :, ky, kx].t()
        pk = _Packed(wt, b.repeat(4), offs, 256 if cout % 64 == 0 else 128, 4 * cout, pair=False, dtype=self._act_torch_dtype)
        pk.subpixel = cout
        return pk

    def _phase_taps(self, parity):
        """(kernel index, input offset) pairs of one output parity of ConvTranspose2d(k=3, s=2) + crop."""
        if self.crop_first:      # kept[y] = U[y + 1]
            return [(1, 0)] if parity == 0 else [(0, 1), (2, 0)]
        return [(0, 0), (2, -1)] if parity == 0 else [(1, 0)]   # kept[y] = U[y]

    # ------------------------------------------------------------------ launch helpers
    def _buf(self, key, shape):
        t = self._bufs.get(key)
        dt = self._act_torch_dtype
        if t is None or tuple(t.shape) != tuple(shape) or t.device != self.s.device or t.dtype != dt:
            t = torch.empty(shape, dtype=dt, device=self.s.device)
            self._bufs[key] = t
        return t

    @staticmethod
    def _conv(pk, src, in_plane_off, dst, out_plane_off=0, act=1, pool=None, pool_plane_off=0, out_mode=0,
              out_scale=(1, 0, 1, 0), stream=0):
        d = AbcConvDesc()
        N, in_planes, H, W, _ = src.shape
        d.in_, d.N, d.H, d.W = src.data_ptr(), N, H, W
        d.in_planes, d.in_plane_off, d.cin = in_planes, in_plane_off, pk.cin
        d.wpack, d.bias = pk.w.data_ptr(), pk.bias.data_ptr()
        d.cout, d.n_tile, d.ntaps = pk.cout, pk.n_tile, len(pk.taps)
        for i, (dy, dx) in enumerate(pk.taps):
            d.tap_dy[i], d.tap_dx[i] = dy, dx
        d.row_fold, d.cta_pair = pk.fold, int(pk.pair)
        d.k_chunk = getattr(pk, "kc", 0) if getattr(pk, "kc", 0) != min(pk.cin, 64) else 0
        d.act_fp16 = int(getattr(pk, "fp16", False))
        d.subpixel = getattr(pk, "subpixel", 0)
        d.swap_mn = int(use_swap(pk, out_mode, dst, pool)) if not d.subpixel else 0
        d.act, d.out_mode = act, out_mode
        sy, oy, sx, ox = out_scale
        d.out_sy, d.out_oy, d.out_sx, d.out_ox = sy, oy, sx, ox
        if dst is not None:
            d.out = dst.data_ptr()
            if out_mode in (0, 2):
                d.out_planes, d.out_H, d.out_W = dst.shape[1], dst.shape[2], dst.shape[3]
            else:
                d.out_planes, d.out_H, d.out_W = 0, dst.shape[2], dst.shape[3]
            d.out_plane_off = out_plane_off
        else:
            d.out, d.out_H, d.out_W = None, H, W
        if pool is not None:
            d.pool_out, d.pool_planes, d.pool_plane_off = pool.data_ptr(), pool.shape[1], pool_plane_off
        check(lib.abc_conv_igemm(C.byref(d), stream), "abc_conv_igemm")

    def _timed(self, name):
        return _LaunchTimer(self.timing, name)

    # ------------------------------------------------------------------ forward
    def forward(self, x):
        if self.training:
            from .train import _UNetTrainFn
            return list(_UNetTrainFn.apply(self, x, *self.parameters()))
        return self.infer(x)

    def _train_engine(self):
        if self._engine is None:
            from .train import TrainEngine
            self._engine = TrainEngine(self)
        return self._engine

    @torch.no_grad()
    def trunk_and_hidden(self, x):
        """Runs everything up to the 8-head conv1 as a separate launch; returns (trunk P8, hidden P8)."""
        k2 = self.trunk(x)
        B, _, H4, W4, _ = k2.shape
        hid = self._buf("hid", (B, 16 * len(self.heads), H4, W4, 8))
        with self._timed("heads.conv1"):
            self._conv(self._packed["heads.conv1"], k2, 0, hid, act=2, stream=_lib.current_stream_ptr())   # BN fold + LeakyReLU(0.01)
        return k2, hid

    @torch.no_grad()
    def trunk(self, x):
        """Encoder + decoder up to dconv2 (unet.py:101-115): the 128-channel stride-4 trunk, P8 bf16."""
        if not x.is_cuda:
            raise RuntimeError("abcnet_b200.UNet.forward needs a CUDA tensor (no CPU fallback)")
        _lib.require_device()
        if x.dim() != 4 or x.shape[1] != self.n_channels or x.shape[2] % 32 or x.shape[3] % 32:
            raise ValueError(f"expected [B,{self.n_channels},H,W] with H, W multiples of 32, got {tuple(x.shape)}")
        if self._packed is None or self._packed_key != self._param_key():
            self.prepare()
        P = self._packed
        # fp32 {0,1} images as the reference's DataLoader delivers them, or the same bits as uint8 / bool
        u8 = self.n_channels == 1 and x.dtype in (torch.uint8, torch.bool)
        x = x.contiguous().view(torch.uint8) if u8 else x.contiguous().float()
        stem_flags = 1 | (2 if self.act_dtype == "fp16" else 0)           # ReLU | fp16 output

        def first(xp, wp, bp, op, B_, H_, W_, planes, off, st_):
            return lib.abc_conv3x3_stem(xp, int(u8), self.n_channels, wp, bp, op, B_, H_, W_, planes, off, stem_flags, st_)
        B, _, H, W = x.shape
        st = _lib.current_stream_ptr()

        def cv(name, *a, **k):
            with self._timed(name):
                self._conv(P[name], *a, stream=st, **k)

        a = self._buf("a", (B, 2, H, W, 8))
        b = self._buf("b", (B, 2, H, W, 8))
        w0, b0 = P["inc1.0"]
        with self._timed("inc1.0"):
            check(first(x.data_ptr(), w0.data_ptr(), b0.data_ptr(), a.data_ptr(), B, H, W, 2, 0, st), "abc_conv3x3_stem")
        cv("inc1.3", a, 0, b)
        cv("inc2.0", b, 0, a)
        p1 = self._buf("p1", (B, 2, H // 2, W // 2, 8))
        cv("inc2.3", a, 0, None, pool=p1)                                   # x1 is never used as a skip (SURVEY D2)
        d1 = self._buf("d1", (B, 4, H // 2, W // 2, 8))
        cv("down1.0", p1, 0, d1)
        p2 = self._buf("p2", (B, 4, H // 4, W // 4, 8))
        cv("down1.3", d1, 0, None, pool=p2)                                 # x2 neither
        e1 = self._buf("e1", (B, 8, H // 4, W // 4, 8))
        e2 = self._buf("e2", (B, 8, H // 4, W // 4, 8))
        cat3 = self._buf("cat3", (B, 16, H // 4, W // 4, 8))
        cv("down2.0", p2, 0, e1)
        cv("down2.3", e1, 0, e2)
        cv("inc3.0", e2, 0, e1)
        p3 = self._buf("p3", (B, 8, H // 8, W // 8, 8))
        cv("inc3.3", e1, 0, cat3, out_plane_off=0, pool=p3)                 # x3 -> concat slot [0, 64)
        f1 = self._buf("f1", (B, 16, H // 8, W // 8, 8))
        cat2 = self._buf("cat2", (B, 32, H // 8, W // 8, 8))
        p4 = self._buf("p4", (B, 16, H // 16, W // 16, 8))
        cv("down3.0", p3, 0, f1)
        cv("down3.3", f1, 0, cat2, out_plane_off=0, pool=p4)                # x4
        g1 = self._buf("g1", (B, 32, H // 16, W // 16, 8))
        cat1 = self._buf("cat1", (B, 64, H // 16, W // 16, 8))
        p5 = self._buf("p5", (B, 32, H // 32, W // 32, 8))
        cv("down4.0", p4, 0, g1)
        cv("down4.3", g1, 0, cat1, out_plane_off=0, pool=p5)                # x5
        h1 = self._buf("h1", (B, 64, H // 32, W // 32, 8))
        h2 = self._buf("h2", (B, 64, H // 32, W // 32, 8))
        cv("down5.0", p5, 0, h1)
        cv("down5.3", h1, 0, h2)                                            # x6

        merged_up = not os.environ.get("ABCNET_UP_PHASES")

        def up(name, src, cat, half_planes):
            with self._timed(name + ".up"):
                if merged_up:
                    self._conv(P[f"{name}.up"], src, 0, cat, out_plane_off=half_planes, act=0, out_scale=(2, 0, 2, 0), stream=st)
                    return
                for py in (0, 1):
                    for px in (0, 1):
                        self._conv(P[f"{name}.up.{py}{px}"], src, 0, cat, out_plane_off=half_planes, act=0,
                                   out_scale=(2, py, 2, px), stream=st)

        up("up1", h2, cat1, 32)
        i1 = self._buf("i1", (B, 32, H // 16, W // 16, 8))
        i2 = self._buf("i2", (B, 32, H // 16, W // 16, 8))
        cv("up1.conv.0", cat1, 0, i1)
        cv("up1.conv.3", i1, 0, i2)
        up("up2", i2, cat2, 16)
        j1 = self._buf("j1", (B, 16, H // 8, W // 8, 8))
        j2 = self._buf("j2", (B, 16, H // 8, W // 8, 8))
        cv("up2.conv.0", cat2, 0, j1)
        cv("up2.conv.3", j1, 0, j2)
        up("up3", j2, cat3, 8)
        k1 = self._buf("k1", (B, 16, H // 4, W // 4, 8))
        k2 = self._buf("k2", (B, 16, H // 4, W // 4, 8))
        cv("up3.conv.0", cat3, 0, k1)
        cv("up3.conv.3", k1, 0, k2)
        cv("dconv1.0", k2, 0, k1)
        cv("dconv1.3", k1, 0, k2)
        cv("dconv2.0", k2, 0, k1)
        cv("dconv2.3", k1, 0, k2)                                           # trunk
        return k2

    @torch.no_grad()
    def infer(self, x, outs=None, layout="nchw", fused=None):
        """Eval forward. layout="nchw": the reference's list of fp32 NCHW tensors. layout="p8f": a ``HeadMaps`` list in
        which heads with more than one channel are fp32 planar-8 [B, ceil(h/8), H/4, W/4, 8] (padding slots undefined);
        this is the format the fused inference + decode path uses (``PeakDecoder`` accepts both).
        fused=None (default): conv1 + LeakyReLU + conv2 of all heads in one kernel (abc_heads_fused) whenever the head list is
        within its limits, unless ABCNET_FUSED_HEADS=0; fused=True requires it; fused=False: conv1 and the per-head conv2 as
        separate launches (hidden maps materialised in HBM)."""
        if layout not in ("nchw", "p8f"):
            raise ValueError("layout must be 'nchw' or 'p8f'")
        p8f = layout == "p8f"
        k2 = self.trunk(x)
        B, _, H4, W4, _ = k2.shape
        st = _lib.current_stream_ptr()
        if outs is None:
            outs = HeadMaps(self.heads)
            for h in self.heads:
                shape = (B, (h + 7) // 8, H4, W4, 8) if (p8f and h > 1) else (B, h, H4, W4)
                outs.append(torch.empty(shape, dtype=torch.float32, device=k2.device))
        fpack = self._packed.get("heads.fused")
        if fused is None:
            # the hidden maps stay in TMEM, so the fused kernel saves their 2 x 8.6 GB HBM round trip per 256-image batch
            # (DESIGN.md 4.2); ABCNET_FUSED_HEADS=0 selects the separate launches for A/B runs
            fused = fpack is not None and os.environ.get("ABCNET_FUSED_HEADS", "1") != "0"
        if fused:
            if fpack is None:
                raise ValueError("abc_heads_fused is not available for this head list (see include/abcnet_b200.h); use fused=False")
            w2pack, bias2 = fpack
            pk1 = self._packed["heads.conv1.plain"]
            if pk1 is None:
                wt1, b1, c1 = self._heads_w1
                pk1 = self._packed["heads.conv1.plain"] = _Packed(wt1, b1, [(dy, dx) for (dy, dx, _, _) in _TAPS3], 256, c1, pair=False,
                                                                  dtype=self._act_torch_dtype)
            d = AbcHeadsFusedDesc()
            d.in_, d.N, d.H, d.W, d.in_planes, d.in_plane_off = k2.data_ptr(), B, H4, W4, k2.shape[1], 0
            d.w1pack, d.bias1, d.n_heads = pk1.w.data_ptr(), pk1.bias.data_ptr(), len(self.heads)
            d.w2pack, d.w2pack_bytes, d.bias2, d.bias2_len = w2pack.data_ptr(), w2pack.numel() * 2, bias2.data_ptr(), bias2.numel()
            slots = [int(v) for v in os.environ.get("ABCNET_HF_SLOTS", "").split(",") if v.strip()]
            for i in range(6):
                d.item_slot[i] = slots[i] if i < len(slots) else -1
            d.act_fp16 = int(pk1.fp16)
            for i, h in enumerate(self.heads):
                d.cout[i], d.out[i] = h, outs[i].data_ptr()
                d.out_mode[i] = 2 if outs[i].dim() == 5 else 1
                d.out_planes[i] = outs[i].shape[1] if outs[i].dim() == 5 else 0
            with self._timed("heads.fused"):
                check(lib.abc_heads_fused(C.byref(d), st), "abc_heads_fused")
            return outs
        hid = self._buf("hid", (B, 16 * len(self.heads), H4, W4, 8))
        with self._timed("heads.conv1"):
            self._conv(self._packed["heads.conv1"], k2, 0, hid, act=2, stream=st)   # BN fold + LeakyReLU(0.01); Dropout is identity in eval
        with self._timed("heads.conv2"):
            for i, h in enumerate(self.heads):
                self._conv(self._packed[f"heads.{i}.conv2"], hid, 16 * i, outs[i], act=0,
                           out_mode=2 if outs[i].dim() == 5 else 1, stream=st)
        return outs

    def activation(self, name):
        """Debug / test access to an internal P8 buffer as an NCHW fp32 tensor."""
        t = self._bufs[name]
        N, P_, H, W, _ = t.shape
        return t.float().permute(0, 1, 4, 2, 3).reshape(N, P_ * 8, H, W)
