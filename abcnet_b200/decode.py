"""Heat-map decoding through the C-ABI (``abc_decode_peaks``) plus the thin adapter that rebuilds the reference's
Python lists, so that the unchanged host assembly of ``img2smiles*.py`` (lines 195-318) can consume them.

Replaces ``/root/reference/src/img2smiles.py:62-80, :115-124`` and the gather loop ``:134-182`` (hundreds of
``.cpu().item()`` synchronisations per image) by ONE kernel launch and ONE device->host copy per batch.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import AbcDecodeDesc, check, lib

ATOM_DT = np.dtype([("x", "<u2"), ("y", "<u2"), ("type", "u1"), ("charge", "u1"), ("hs", "u1"), ("pad", "u1")])
BOND_DT = np.dtype([("x", "<u2"), ("y", "<u2"), ("omega", "u1"), ("type", "u1"), ("pad", "<u2"), ("rho", "<f4")])

# utils.py:12-14 inverted as in img2smiles.py:24-26 (index 0 -> 'C')
ATOM_SYMBOLS = ['C', 'C', 'N', 'O', 'P', 'F', 'Cl', 'S', 'Br', 'B', 'Se', 'I', 'H', 'Si']
CHARGE_VALUES = [0, 1, -1]


class PeakDecoder:
    """Reusable decoder: owns the (pinned) host and device record buffers for a fixed batch size and capacity."""

    def __init__(self, batch, atom_cap=512, bond_cap=2048, device=None):
        self.batch, self.atom_cap, self.bond_cap = batch, atom_cap, bond_cap
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        self.d_atoms = torch.empty((batch, atom_cap, 8), dtype=torch.uint8, device=self.device)
        self.d_bonds = torch.empty((batch, bond_cap, 12), dtype=torch.uint8, device=self.device)
        self.d_counts = torch.empty((batch, 4), dtype=torch.int32, device=self.device)
        self.h_atoms = torch.empty((batch, atom_cap, 8), dtype=torch.uint8).pin_memory()
        self.h_bonds = torch.empty((batch, bond_cap, 12), dtype=torch.uint8).pin_memory()
        self.h_counts = torch.empty((batch, 4), dtype=torch.int32).pin_memory()

    def launch(self, outs, thr=-1.0, omega_mode="nms", apply_sigmoid=False, thr_omega=-1.0):
        """Enqueue the decode kernel on the current stream (no synchronisation).

        ``apply_sigmoid=True`` selects the training-time metric definition of a centre peak (train.py:95,100,145-151):
        threshold ``thr`` (0.25 there) and 3x3 NMS on ``clamp(sigmoid(z), 1e-5, 1 - 1e-5)`` instead of on the raw logit
        (img2smiles.py:62-68, ``thr = -1``); the omega NMS then uses the logit threshold ``thr_omega``."""
        if len(outs) != 8:
            raise ValueError("decode needs the 8 head outputs of the v2 model")
        for o in outs:
            if not (o.is_cuda and o.dtype == torch.float32 and o.is_contiguous()):
                raise ValueError("decode inputs must be contiguous fp32 CUDA tensors -- there is no CPU path")
        _lib.require_device()
        # NCHW tensors [N,C,H,W] (the reference's format) or planar-8 maps [N,ceil(C/8),H,W,8] from UNet.infer(layout="p8f")
        heads = getattr(outs, "heads", None)
        mask, chans = 0, []
        for i, o in enumerate(outs):
            if o.dim() == 5:
                if heads is None:
                    raise ValueError("planar-8 maps need the channel counts (use the HeadMaps returned by UNet.infer)")
                mask |= 1 << i
                chans.append(heads[i])
            else:
                chans.append(o.shape[1])
        N, H, W = outs[0].shape[0], outs[0].shape[2], outs[0].shape[3]
        if N > self.batch:
            raise ValueError(f"batch {N} exceeds decoder capacity {self.batch}")
        n_omega = chans[7]
        d = AbcDecodeDesc()
        for i, o in enumerate(outs):
            d.maps[i] = o.data_ptr()
        d.N, d.H, d.W = N, H, W
        d.c_type, d.c_charge, d.c_hs = chans[1], chans[2], chans[3]
        d.n_omega, d.n_btype = n_omega, chans[5] // n_omega
        d.p8f_mask = mask
        d.thr = float(thr)
        d.omega_mode = {"nms": 0, "raw": 1}[omega_mode]
        d.centre_prob, d.thr_omega = int(bool(apply_sigmoid)), float(thr_omega)
        d.atoms, d.atom_cap = self.d_atoms.data_ptr(), self.atom_cap
        d.bonds, d.bond_cap = self.d_bonds.data_ptr(), self.bond_cap
        d.counts = self.d_counts.data_ptr()
        check(lib.abc_decode_peaks(C.byref(d), _lib.current_stream_ptr()), "abc_decode_peaks")
        return N

    def fetch_async(self, N):
        """Enqueue the D2H copy of the compact records behind the decode kernel and record an event; ``collect`` waits for
        that event only, so the host can already enqueue the next batch on the same stream (use one PeakDecoder per batch in
        flight)."""
        self.h_counts[:N].copy_(self.d_counts[:N], non_blocking=True)
        self.h_atoms[:N].copy_(self.d_atoms[:N], non_blocking=True)
        self.h_bonds[:N].copy_(self.d_bonds[:N], non_blocking=True)
        if getattr(self, "_done", None) is None:
            self._done = torch.cuda.Event()
        self._done.record(torch.cuda.current_stream())
        return N

    def wait_copy(self):
        """Wait for the copy enqueued by ``fetch_async``; no capacity check (``h_counts`` is then valid)."""
        self._done.synchronize()

    def collect(self, N):
        """Wait for the copy enqueued by ``fetch_async`` and return per-image numpy record arrays."""
        self.wait_copy()
        return self._parse(N)

    def wait(self, N):
        """Wait for the copy enqueued by ``fetch_async`` and check the capacities, without building per-image arrays (for
        callers that go straight to ``molblocks``). Returns the [N, 4] counts."""
        self.wait_copy()
        counts = self.h_counts[:N].numpy()
        if (counts[:, 0] > self.atom_cap).any() or (counts[:, 1] > self.bond_cap).any():
            raise RuntimeError(f"decode capacity exceeded: max atoms {counts[:, 0].max()} (cap {self.atom_cap}), "
                               f"max bond records {counts[:, 1].max()} (cap {self.bond_cap}); enlarge the capacities")
        return counts

    def fetch(self, N):
        """One async D2H of the compact records + a single stream sync; returns per-image numpy record arrays."""
        self.h_counts[:N].copy_(self.d_counts[:N], non_blocking=True)
        self.h_atoms[:N].copy_(self.d_atoms[:N], non_blocking=True)
        self.h_bonds[:N].copy_(self.d_bonds[:N], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._parse(N)

    def molblocks(self, N, n_threads=0):
        """MOL-block text of the N images whose records were fetched last (``fetch`` / ``collect``), or ``None`` per image
        without a molecule -- native multi-threaded host assembly, see ``assemble_molblocks``."""
        counts = self.h_counts[:N].numpy()
        if (counts[:, 0] > self.atom_cap).any() or (counts[:, 1] > self.bond_cap).any():
            raise RuntimeError("decode capacity exceeded; enlarge the capacities")
        return assemble_molblocks(self.h_atoms, self.h_bonds, self.h_counts[:N], n_threads=n_threads)

    def _parse(self, N):
        counts = self.h_counts[:N].numpy()
        if (counts[:, 0] > self.atom_cap).any() or (counts[:, 1] > self.bond_cap).any():
            raise RuntimeError(f"decode capacity exceeded: max atoms {counts[:, 0].max()} (cap {self.atom_cap}), "
                               f"max bond records {counts[:, 1].max()} (cap {self.bond_cap}); enlarge the capacities")
        atoms = self.h_atoms[:N].numpy().view(ATOM_DT).reshape(N, self.atom_cap)
        bonds = self.h_bonds[:N].numpy().view(BOND_DT).reshape(N, self.bond_cap)
        return [(atoms[i, :counts[i, 0]].copy(), bonds[i, :counts[i, 1]].copy(), int(counts[i, 2])) for i in range(N)]

    def __call__(self, outs, thr=-1.0, omega_mode="nms", apply_sigmoid=False, thr_omega=-1.0):
        return self.fetch(self.launch(outs, thr, omega_mode, apply_sigmoid, thr_omega))


_OMEGA_TABLES = {}


def omega_tables(n_omega=60):
    """(cos, sin) of the bin angles omega_w = w * pi / (n_omega / 2) + pi / n_omega - pi / 2 (img2smiles.py:160), float64."""
    t = _OMEGA_TABLES.get(n_omega)
    if t is None:
        w = np.arange(n_omega, dtype=np.int64)
        omega = w * (np.pi / (n_omega // 2)) + np.pi / n_omega - np.pi / 2
        t = _OMEGA_TABLES[n_omega] = (np.ascontiguousarray(np.cos(omega)), np.ascontiguousarray(np.sin(omega)))
    return t


def assemble_molblocks(atoms, bonds, counts, n_omega=60, n_threads=0):
    """Decoded records of a batch -> list of V2000 MOL-block strings (``None`` where the reference yields no molecule), through
    the native multi-threaded assembler ``abc_assemble_molblocks``: the host loop of ``img2smiles.py:183-318`` plus the text
    builder of ``generate_smiles.py:18-105`` (the string RDKit parses at ``:115-118``), byte-identical to feeding
    ``records_to_lists`` into the unchanged Python statements.

    atoms: uint8 [N, atom_cap, 8], bonds: uint8 [N, bond_cap, 12], counts: int32 [N, 4] -- host arrays / CPU tensors as filled
    by ``PeakDecoder`` (``h_atoms`` / ``h_bonds`` / ``h_counts``)."""
    def as_np(t, dt):
        a = t.numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
        if a.dtype != dt or not a.flags.c_contiguous:
            raise ValueError(f"assemble_molblocks: expected a C-contiguous {dt} host array")
        return a
    a, b, c = as_np(atoms, np.uint8), as_np(bonds, np.uint8), as_np(counts, np.int32)
    N = c.shape[0]
    if N == 0:
        return []
    if a.ndim != 3 or b.ndim != 3 or a.shape[2] != 8 or b.shape[2] != 12 or a.shape[0] < N or b.shape[0] < N or c.shape[1] != 4:
        raise ValueError("assemble_molblocks: bad record array shapes")
    cos_t, sin_t = omega_tables(n_omega)
    n_at, n_bd = int(c[:, 0].max()), int(c[:, 1].max())
    stride = 96 + 80 * n_at + 16 * n_bd + 230 * min(n_at, 2 * n_bd)          # header + atom lines + bond lines + CHG + implicit-H blocks
    text = np.empty((N, stride), dtype=np.uint8)
    lens = np.empty(N, dtype=np.int32)
    check(lib.abc_assemble_molblocks(a.ctypes.data, a.shape[1], b.ctypes.data, b.shape[1], c.ctypes.data, N, cos_t.ctypes.data,
                                     sin_t.ctypes.data, n_omega, n_threads, text.ctypes.data, stride, lens.ctypes.data),
          "abc_assemble_molblocks")
    return [None if lens[i] < 0 else text[i, :lens[i]].tobytes().decode("ascii") for i in range(N)]


def records_to_lists(atoms, bonds, n_bond_peaks=None, n_omega=60):
    """Rebuild the lists of img2smiles.py:131-193 from one image's records; ``None`` when the image has no atom or
    no bond-centre peak (img2smiles.py:126-129). The greedy de-duplication of :183-187 is applied here."""
    if len(atoms) == 0 or (n_bond_peaks == 0 if n_bond_peaks is not None else len(bonds) == 0):
        return None
    w = bonds["omega"].astype(np.int64)
    omega = w * (np.pi / (n_omega // 2)) + np.pi / n_omega - np.pi / 2
    rho = bonds["rho"].astype(np.float64)
    out = dict(
        bonds_position_list=np.stack([bonds["x"], bonds["y"]], -1).astype(np.int64).tolist(),
        bonds_property_list=bonds["type"].astype(np.int64).tolist(),
        bonds_delta_list=np.stack([rho * np.cos(omega), rho * np.sin(omega)], -1).tolist(),
        atoms_position_list=[], atoms_type_list=[], atoms_charge_list=[], atoms_hs_list=[])
    kept = np.empty((len(atoms), 2), np.int64)
    k = 0
    for a in atoms:
        x, y = int(a["x"]), int(a["y"])
        if k and ((kept[:k] - (x, y)) ** 2).sum(-1).min() < 4:
            continue
        kept[k] = (x, y)
        k += 1
        out["atoms_position_list"].append([x, y])
        out["atoms_type_list"].append(ATOM_SYMBOLS[a["type"]])
        out["atoms_charge_list"].append(CHARGE_VALUES[a["charge"]])
        out["atoms_hs_list"].append(int(a["hs"]))
    return out
