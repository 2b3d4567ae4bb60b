"""Fused ABC-Net training losses through the C-ABI (``abc_loss_partials`` / ``abc_loss_backward``).

Replaces ``/root/reference/src/train.py:95-137`` (``class_weights=True``) and
``/root/reference/src/multi_gpu_train2.py:140-192`` (``class_weights=False``): activations, the eight losses, the
learned uncertainty weighting with ``model.s`` and -- through ``torch.autograd.Function`` -- their gradients with
respect to the eight logit maps and to ``s``. Two bandwidth-bound passes over logits + targets instead of ~120 ATen
kernels; numerators / denominators are accumulated in fp64 on the device, no host synchronisation.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import AbcLossDesc, AbcLossP8Out, check, lib

ATOM_TYPE_WEIGHTS = [1, 0.1, 0.1, 0.1, 1, 1, 1, 1, 1, 10, 10, 10, 10, 10]          # train.py:16
# kernel order: atom, bond, type, charge, btype, rho, omega, hs  ->  index into model.s (train.py:127-135)
_S_INDEX = [0, 1, 2, 3, 4, 6, 7, 9]
NAMES = ["atom_targets", "bond_targets", "atom_types", "atom_charges", "bond_types", "bond_rhos", "bond_omega_types", "atom_hs"]


def _desc(logits, targets, type_w, sums, scale, dlogits):
    d = AbcLossDesc()
    N, _, H, W = logits[0].shape
    n_omega = logits[7].shape[1]
    for i in range(8):
        d.logits[i] = logits[i].data_ptr()
        d.targets[i] = targets[i].data_ptr()
        d.dlogits[i] = dlogits[i].data_ptr() if dlogits is not None else None
    d.tgt_f64 = 1 if targets[6].dtype == torch.float64 else 0
    d.N, d.H, d.W = N, H, W
    d.c_type, d.c_charge, d.c_hs = logits[1].shape[1], logits[2].shape[1], logits[3].shape[1]
    d.n_omega, d.n_btype = n_omega, logits[5].shape[1] // n_omega
    d.type_weights = type_w.data_ptr() if type_w is not None else None
    d.sums = sums.data_ptr() if sums is not None else None
    d.scale = scale.data_ptr() if scale is not None else None
    return d


def _det_ws(d, p8, dev):
    """Under torch.use_deterministic_algorithms: a workspace for the fixed-order sums of the loss pass (AbcLossDesc.ws)."""
    if not torch.are_deterministic_algorithms_enabled():
        return None
    ws = torch.empty(lib.abc_loss_workspace_bytes(C.byref(d), p8), dtype=torch.uint8, device=dev)
    d.ws = ws.data_ptr()
    return ws


_IDX_CACHE = {}


def _s_index(dev):
    """Device-resident index / constant tensors (created once per device: no host -> device copy inside a CUDA-graph capture)."""
    t = _IDX_CACHE.get(dev)
    if t is None:
        half = [1.0] * 8
        half[5] = 0.5                                                      # train.py:133 (rho term: 0.5 * exp(-s) + s)
        t = _IDX_CACHE[dev] = (torch.tensor(_S_INDEX, dtype=torch.long, device=dev),
                               torch.tensor(half, dtype=torch.float64, device=dev),
                               torch.tensor(_HEAD_TO_LOSS, dtype=torch.long, device=dev))
    return t


# head i of UNet.forward -> loss index of the kernels (AbcLossIndex): atom, type, charge, hs, bond, btype, rho, omega
_HEAD_TO_LOSS = [0, 2, 3, 7, 1, 4, 5, 6]


def loss_forward_backward(s, type_w, targets, logits, scaled=True):
    """Losses + gradients without autograd. Returns (total fp64 scalar, 8 weighted parts, dL/ds [10] fp64, 8 dlogits fp32,
    head_scale). ``scaled=True``: two passes, dlogits are dL/dlogits and head_scale is None. ``scaled=False``: ONE fused
    pass, dlogits are unscaled and dL/dlogits[i] = head_scale[i] * dlogits[i] (fp32 device tensor [8]; the consumer --
    TrainEngine.backward -- folds the factor into its fp32 -> bf16 conversion). No host synchronisation: capturable."""
    _lib.require_device()
    logits = [z.contiguous() for z in logits]
    for z in logits:
        if not (z.is_cuda and z.dtype == torch.float32):
            raise ValueError("loss inputs must be fp32 CUDA tensors (no CPU fallback)")
    # kernel target order: atom, type, charge, hs, bond, btype, rho, omega  (= the reference's argument order)
    if targets[6].dtype != targets[7].dtype:
        raise ValueError("rho / omega targets must share a dtype (fp32 or fp64, utils.py:91-92)")
    for i, t in enumerate(targets):
        want = (torch.float32, torch.float64) if i >= 6 else (torch.float32,)
        if not (t.is_cuda and t.is_contiguous() and t.dtype in want):
            raise ValueError(f"target {i}: contiguous CUDA tensor of dtype {want} required")
    st = _lib.current_stream_ptr()
    dev = logits[0].device
    sums = torch.empty(16, dtype=torch.float64, device=dev)
    dlogits = [torch.empty_like(z) for z in logits]
    d = _desc(logits, targets, type_w, sums, None, None if scaled else dlogits)
    ws = _det_ws(d, 0, dev)  # noqa: F841  (alive until the call is enqueued)
    check(lib.abc_loss_partials(C.byref(d), st), "abc_loss_partials")
    total, parts, ds, scale, h2l = _weighting(sums, s, dev)
    head_scale = None
    if scaled:
        check(lib.abc_loss_backward(C.byref(_desc(logits, targets, type_w, None, scale, dlogits)), st), "abc_loss_backward")
    else:
        head_scale = scale[h2l]
    return total, parts, ds, dlogits, head_scale


def _weighting(sums, s, dev):
    """Uncertainty weighting of train.py:127-137 from the 8 numerators / 8 denominators: (total, weighted parts, dL/ds [10],
    per-loss gradient factor u_k / denom_k in kernel order, head -> loss index)."""
    num, den = sums[:8], sums[8:].clone()
    den[7] = den[7] + 0.1                                                  # train.py:114
    raw = num / den
    idx, half, h2l = _s_index(dev)
    sk = s.detach().double()[idx]
    u = half * torch.exp(-sk) + sk
    total = (raw * u).sum()
    scale = (u / den).float().contiguous()
    ds = torch.zeros(10, dtype=torch.float64, device=dev)
    ds[idx] = raw * (1.0 - half * torch.exp(-sk))
    return total, (raw * u).detach(), ds, scale, h2l


def head_grad_planes(h):
    """P8 planes of the gradient operand of a head with h logit channels (K of its data-gradient GEMM, zero padded)."""
    c = (h + 15) // 16 * 16 if h <= 64 else (h + 63) // 64 * 64
    return c // 8


def p8_loss_supported(logits):
    """abc_loss_partials_p8 covers the v2 head list (src/train.py:47): 14 / 3 / 2 classes, 6 bond types, n_omega % 4 == 0."""
    n_omega = logits[7].shape[1]
    return ([z.shape[1] for z in logits[:5]] == [1, 14, 3, 2, 1] and n_omega % 4 == 0 and n_omega >= 4
            and logits[5].shape[1] == 6 * n_omega and logits[6].shape[1] == n_omega)


def loss_forward_p8(s, type_w, targets, logits, dz_p8, dbias):
    """One pass over logits + targets (abc_loss_partials_p8): the losses and the UNSCALED gradient written directly as the bf16 P8
    operand of the head weight- / data-gradient GEMMs (``dz_p8[i]``: [B, head_grad_planes(h_i), H, W, 8] bf16) plus its per-channel
    sums (``dbias[i]``: fp64 [h_i]). Returns (total fp64 scalar, 8 weighted parts, dL/ds [10] fp64, head_scale fp32 [8]) with
    dL/dlogits[i] = head_scale[i] * dz_p8[i]. No fp32 gradient maps, no conversion pass, no host synchronisation."""
    _lib.require_device()
    logits = [z.contiguous() for z in logits]
    if targets[6].dtype != targets[7].dtype:
        raise ValueError("rho / omega targets must share a dtype (fp32 or fp64, utils.py:91-92)")
    for i, t in enumerate(targets):
        want = (torch.float32, torch.float64) if i >= 6 else (torch.float32,)
        if not (t.is_cuda and t.is_contiguous() and t.dtype in want):
            raise ValueError(f"target {i}: contiguous CUDA tensor of dtype {want} required")
    dev = logits[0].device
    B, _, H, W = logits[0].shape
    out = AbcLossP8Out()
    for i, z in enumerate(logits):
        if not (z.is_cuda and z.dtype == torch.float32):
            raise ValueError("loss inputs must be fp32 CUDA tensors (no CPU fallback)")
        g, b = dz_p8[i], dbias[i]
        if not (g.dtype == torch.bfloat16 and g.is_contiguous() and tuple(g.shape) == (B, g.shape[1], H, W, 8) and g.shape[1] * 8 >= z.shape[1]):
            raise ValueError(f"dz_p8[{i}]: contiguous bf16 [B, planes, H, W, 8] with planes * 8 >= {z.shape[1]} required")
        if not (b.dtype == torch.float64 and b.numel() >= z.shape[1]):
            raise ValueError(f"dbias[{i}]: fp64 [{z.shape[1]}] required")
        out.dz[i], out.planes[i], out.dbias[i] = g.data_ptr(), g.shape[1], b.data_ptr()
    sums = torch.empty(16, dtype=torch.float64, device=dev)
    d = _desc(logits, targets, type_w, sums, None, None)
    ws = _det_ws(d, 1, dev)  # noqa: F841  (alive until the call is enqueued)
    check(lib.abc_loss_partials_p8(C.byref(d), C.byref(out), _lib.current_stream_ptr()), "abc_loss_partials_p8")
    total, parts, ds, scale, h2l = _weighting(sums, s, dev)
    return total, parts, ds, scale[h2l]


class _HeatmapLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, type_w, targets, *logits):
        total, parts, ds, dlogits, _ = loss_forward_backward(s, type_w, targets, logits)
        ctx.save_for_backward(ds.to(s.dtype), *dlogits)
        ctx.parts = parts
        return total

    @staticmethod
    def backward(ctx, g):
        ds, *dlogits = ctx.saved_tensors
        gf = g.float()
        return (g.to(ds.dtype) * ds, None, None) + tuple(gf * d for d in dlogits)


class HeatmapLoss(torch.nn.Module):
    """loss = HeatmapLoss(class_weights=True)(outs, targets, model.s)

    outs: the 8 tensors returned by UNet.forward; targets: (atom_targets, atom_types, atom_charges, atom_hs,
    bond_targets, bond_types, bond_rhos, bond_omega_types) as produced by the reference's collate_fn
    (utils.py:254-300). Returns the float64 scalar of train.py:137; ``.last_parts`` holds the 8 weighted terms."""

    def __init__(self, class_weights: bool = True):
        super().__init__()
        self.class_weights = class_weights
        self.register_buffer("type_w", torch.tensor(ATOM_TYPE_WEIGHTS, dtype=torch.float32), persistent=False)
        self.last_parts = None

    def forward(self, outs, targets, s):
        tw = None
        if self.class_weights:
            if self.type_w.device != outs[0].device:
                self.type_w = self.type_w.to(outs[0].device)
            tw = self.type_w
        total = _HeatmapLossFn.apply(s, tw, list(targets), *outs)
        return total
