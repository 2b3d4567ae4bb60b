"""Fused inference + decode with SPARSE class / offset heads (SURVEY.md section 8f, N4) -- an opt-in fast path.

The reference evaluates all eight ``OutConv`` heads densely (``/root/reference/src/unet.py:116-118``) and then reads six of
them only at the atom / bond centre peaks (``/root/reference/src/img2smiles.py:115-124, :134-193``). Here only the two
centre heads (outputs 0 and 4) are evaluated densely; after the peak search the 3x3 trunk neighbourhoods of the peaks are
gathered into a compact tensor and the SAME head kernels with the SAME packed weights run on it:

    trunk -> conv1+conv2 of heads 0, 4 (dense) -> peak lists -> gather 3x3 patches -> conv1 (as a 1x1 GEMM over K = 9 x 128
    in the dense kernel's K order) -> conv2 of heads 1, 2, 3, 5, 6, 7 on the compact hidden map -> records

Per output element the tensor cores execute the same MMA sequence on the same operands as in the dense path, so the logits
at the peaks -- and therefore the records -- are bit-identical to ``UNet.infer`` + ``PeakDecoder``
(``tests/test_sparse_gpu.py``), while 6/8 of the head FLOPs (29 of 94 GFLOP per image) and the 8.4 GB of dense logits per
256-image batch are never produced. ``model(x)`` / ``UNet.infer`` keep returning the dense maps.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import AbcDecodeDesc, check, lib
from .decode import PeakDecoder
from .unet import _Packed, _TAPS3

V2_HEADS = [1, 14, 3, 2, 1, 360, 60, 60]
_CLASS_HEADS = (1, 2, 3, 5, 6, 7)


class SparseHeadsPipeline:
    """pipe = SparseHeadsPipeline(model, batch, peak_cap=128, bond_cap=2048, peak_pool=None, atom_cap=None)
    n = pipe.launch(x)            # enqueue everything on the current stream (no synchronisation); x holds 1 .. batch images
    recs = pipe.fetch(n)          # same per-image (atoms, bonds, n_bond_peaks) records as PeakDecoder.fetch

    Slot layouts of the compact tensors the class / offset heads run on:

    * ``peak_pool=None`` (fixed): ``peak_cap`` slots per image and peak kind (multiple of 64, <= 1024). An image with more
      atom or bond-centre peaks than that makes ``fetch`` raise (the dense path has no such limit).
    * ``peak_pool=S`` (pooled, a multiple of 64): the batch shares S slots, handed out on the device in image order. An image
      may have any number of peaks; ``fetch`` / ``collect`` / ``wait`` raise only when the batch's atom plus bond-centre
      peaks exceed S. The per-step work is that of S slots whatever the peaks, so S = 2 * batch * peak_cap costs what the
      fixed layout costs. ``peak_cap`` is not used.

    ``atom_cap`` sizes the atom record arrays: ``peak_cap`` by default in the fixed layout, 1024 in the pooled one."""

    def __init__(self, model, batch, peak_cap=128, bond_cap=2048, device=None, peak_pool=None, atom_cap=None):
        if list(model.heads) != V2_HEADS:
            raise NotImplementedError("SparseHeadsPipeline: the v2 head list [1, 14, 3, 2, 1, 360, 60, 60] only")
        if peak_pool is None:
            if peak_cap % 64 or not (64 <= peak_cap <= 1024):
                raise ValueError("peak_cap must be a multiple of 64 in [64, 1024]")
            P = 2 * batch * peak_cap
        else:
            if peak_pool % 64 or not (64 <= peak_pool < 1 << 30):
                raise ValueError("peak_pool must be a positive multiple of 64 (below 2^30)")
            P = peak_pool
        self.m, self.batch, self.cap, self.pool = model, batch, peak_cap, peak_pool
        self.dev = device or model.s.device
        if atom_cap is None:
            atom_cap = peak_cap if peak_pool is None else 1024
        self.dec = PeakDecoder(batch, atom_cap=atom_cap, bond_cap=bond_cap, device=self.dev)
        self.P = P
        dev = self.dev
        if peak_pool is None:
            self.peak_pix = torch.zeros((batch, 2, peak_cap), dtype=torch.int32, device=dev)
        else:
            self.peak_pix = None                                          # untruncated lists [batch][2][H * W], sized at launch
            self.peak_off = torch.zeros(2 * batch + 1, dtype=torch.int32, device=dev)
        self.peak_cnt = torch.zeros((batch, 2), dtype=torch.int32, device=dev)
        rows = self.P // 8
        adt = model._act_torch_dtype                                                              # 16-bit storage format of the model
        self.patches = torch.zeros((1, 144, rows, 8, 8), dtype=adt, device=dev)                  # unused slots stay finite
        self.hid_c = torch.zeros((1, 128, rows, 8, 8), dtype=adt, device=dev)
        self.logits_c = {k: torch.zeros((1, (V2_HEADS[k] + 7) // 8, rows, 8, 8), dtype=torch.float32, device=dev) for k in _CLASS_HEADS}
        self._bufs = {}
        self._centre_pack = None
        self._centre_key = None

    def _buf(self, key, shape, dtype):
        t = self._bufs.get(key)
        if t is None or tuple(t.shape) != tuple(shape):
            t = self._bufs[key] = torch.empty(shape, dtype=dtype, device=self.dev)
        return t

    @torch.no_grad()
    def launch(self, x, thr=-1.0, omega_mode="nms", apply_sigmoid=False, thr_omega=-1.0):
        """Same decoding options as ``PeakDecoder.launch``."""
        m = self.m
        k2 = m.trunk(x)                                                  # also (re)packs the weights when they changed
        B, _, H4, W4, _ = k2.shape
        if not 1 <= B <= self.batch:
            raise ValueError(f"SparseHeadsPipeline was built for batches of up to {self.batch} images, got {B}")
        st = _lib.current_stream_ptr()
        P_ = m._packed
        if self._centre_pack is None or self._centre_key != m._pack_gen:
            wt, bias, _ = m._heads_w1                                    # [9, 1024, 128] BN-folded conv1 of all heads
            sel = torch.cat([torch.arange(0, 128), torch.arange(512, 640)]).to(wt.device)       # heads 0 and 4
            self._centre_pack = _Packed(wt[:, sel].contiguous(), bias[sel].contiguous(), [(dy, dx) for (dy, dx, _, _) in _TAPS3], 256, 256,
                                        dtype=m._act_torch_dtype)
            self._centre_key = m._pack_gen
        # dense centre heads
        hid2 = self._buf("hid2", (B, 32, H4, W4, 8), m._act_torch_dtype)
        m._conv(self._centre_pack, k2, 0, hid2, act=2, stream=st)
        za = self._buf("za", (B, 1, H4, W4), torch.float32)
        zb = self._buf("zb", (B, 1, H4, W4), torch.float32)
        m._conv(P_["heads.0.conv2"], hid2, 0, za, act=0, out_mode=1, stream=st)
        m._conv(P_["heads.4.conv2"], hid2, 16, zb, act=0, out_mode=1, stream=st)
        # peak lists (pooled: untruncated, plus the slot offsets of every image and peak kind)
        if self.pool is None:
            plist, P = self.peak_pix, 2 * B * self.cap
        else:
            plist, P = self._buf("plist", (self.batch, 2, H4 * W4), torch.int32), self.pool
        d = self._desc(B, H4, W4, thr, omega_mode, apply_sigmoid, thr_omega, plist)
        d.maps[0], d.maps[4] = za.data_ptr(), zb.data_ptr()
        d.sparse_mode = 1
        check(lib.abc_decode_peaks(C.byref(d), st), "abc_decode_peaks[find]")
        # 3x3 trunk patches of the peaks -> compact K-ordered tensor -> conv1 (all heads' weights, same pack as the dense layer)
        patches = _slots(self.patches, P)
        if self.pool is None:
            check(lib.abc_gather_patches(k2.data_ptr(), B, H4, W4, 16, plist.data_ptr(), self.peak_cnt.data_ptr(), self.cap,
                                         patches.data_ptr(), st), "abc_gather_patches")
        else:
            check(lib.abc_gather_patches_pooled(k2.data_ptr(), B, H4, W4, 16, plist.data_ptr(), self.peak_cnt.data_ptr(),
                                                self.peak_off.data_ptr(), self.pool, patches.data_ptr(), st), "abc_gather_patches_pooled")
        pk1 = P_["heads.conv1"]
        if pk1.pair:
            raise RuntimeError("SparseHeadsPipeline does not support the CTA-pair weight pack (ABCNET_PAIR=1)")
        hid_c = _slots(self.hid_c, P)
        self._conv1x1_k(pk1, patches, hid_c, st)
        for k in _CLASS_HEADS:
            m._conv(P_[f"heads.{k}.conv2"], hid_c, 16 * k, _slots(self.logits_c[k], P), act=0, out_mode=2, stream=st)
        # records
        d = self._desc(B, H4, W4, thr, omega_mode, apply_sigmoid, thr_omega, plist)
        for k in _CLASS_HEADS:
            d.maps[k] = self.logits_c[k].data_ptr()
        d.p8f_mask = sum(1 << k for k in _CLASS_HEADS)
        d.sparse_mode = 2
        check(lib.abc_decode_peaks(C.byref(d), st), "abc_decode_peaks[finish]")
        return B

    def _conv1x1_k(self, pk, src, dst, st):
        """The dense 3x3 conv1 pack consumed as a 1x1 convolution over K = 9 x 128 gathered channels (same block order)."""
        view = _PackView(pk)
        self.m._conv(view, src, 0, dst, act=2, stream=st)

    def _desc(self, B, H4, W4, thr, omega_mode, apply_sigmoid, thr_omega, plist):
        d = AbcDecodeDesc()
        d.N, d.H, d.W = B, H4, W4
        d.c_type, d.c_charge, d.c_hs, d.n_omega, d.n_btype = 14, 3, 2, 60, 6
        d.thr, d.thr_omega = float(thr), float(thr_omega)
        d.centre_prob = int(bool(apply_sigmoid))
        d.omega_mode = {"nms": 0, "raw": 1}[omega_mode]
        d.atoms, d.atom_cap = self.dec.d_atoms.data_ptr(), self.dec.atom_cap
        d.bonds, d.bond_cap = self.dec.d_bonds.data_ptr(), self.dec.bond_cap
        d.counts = self.dec.d_counts.data_ptr()
        d.peak_pix, d.peak_cnt, d.peak_cap = plist.data_ptr(), self.peak_cnt.data_ptr(), self.cap
        if self.pool is not None:
            d.peak_off, d.pool_slots = self.peak_off.data_ptr(), self.pool
        return d

    def _check_slots(self, N):
        """Every peak of the batch had a slot, so the records are complete (from the counts already copied back): in the
        fixed layout no image has more than peak_cap atom or bond-centre peaks, in the pooled one the batch fits the pool.
        Checked before the record capacities, which may be larger than peak_cap."""
        counts = self.dec.h_counts[:N].numpy()
        if self.pool is None:
            for col, kind in ((2, "bond-centre"), (0, "atom")):
                if (counts[:, col] > self.cap).any():
                    raise RuntimeError(f"sparse heads: {int(counts[:, col].max())} {kind} peaks in one image exceed peak_cap "
                                       f"{self.cap}; use a larger peak_cap, a peak_pool or the dense path")
            return
        total = int(counts[:, 0].sum(dtype="int64") + counts[:, 2].sum(dtype="int64"))
        if total > self.pool:
            raise RuntimeError(f"sparse heads: {total} atom + bond-centre peaks in the batch exceed peak_pool {self.pool}; "
                               "use a larger peak_pool or the dense path")

    def fetch(self, N):
        self.dec.fetch_async(N)
        return self.collect(N)

    def fetch_async(self, N):
        return self.dec.fetch_async(N)

    def collect(self, N):
        self.dec.wait_copy()
        self._check_slots(N)
        return self.dec.collect(N)                                       # raises when a count exceeds atom_cap / bond_cap

    def wait(self, N):
        self.dec.wait_copy()
        self._check_slots(N)
        return self.dec.wait(N)

    def molblocks(self, N, n_threads=0):
        return self.dec.molblocks(N, n_threads)


def _slots(t, P):
    """The first P slots of a compact tensor [1][planes][rows][8][8]: the layout a convolution over P slots reads / writes."""
    return t.view(-1)[: t.shape[1] * P * 8].view(1, t.shape[1], P // 8, 8, 8)


class _PackView:
    """A 3x3 pack [n-tile][chunk][tap] seen as the 1x1 pack [n-tile][chunk * 9 + tap] over 9x the channels: same bytes."""

    def __init__(self, pk):
        self.w, self.bias, self.n_tile, self.cout = pk.w, pk.bias, pk.n_tile, pk.cout
        self.cin = pk.cin * len(pk.taps)
        self.taps = [(0, 0)]
        self.fold, self.pair = 1, False
        self.fp16 = getattr(pk, "fp16", False)
