"""ctypes binding of ``libabcnet_b200.so`` (the C-ABI declared in ``include/abcnet_b200.h``).

There is no CPU / PyTorch fallback: if the shared library is missing or a call fails, an exception
is raised. Build the library with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C abcnet_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libabcnet_b200.so")

EXPORTS = (
    "abc_last_error", "abc_version", "abc_device_ok", "abc_sm_count", "abc_launch_count",
    "abc_conv3x3_c1", "abc_conv3x3_c1_u8", "abc_conv3x3_cn", "abc_conv3x3_cn_wgrad", "abc_conv3x3_stem", "abc_conv_igemm", "abc_conv_wpack_bytes", "abc_decode_peaks",
    "abc_loss_partials", "abc_loss_backward", "abc_loss_partials_p8",
    "abc_bn_stats", "abc_bn_finalize", "abc_bn_act", "abc_bn_act_backward", "abc_nchw_to_p8", "abc_channel_sum",
    "abc_nchw_to_p8_ex", "abc_deinterleave2", "abc_conv_wgrad", "abc_conv3x3_c1_wgrad", "abc_conv3x3_c1_raw",
    "abc_heads_fused", "abc_heads_fused_pack_sizes", "abc_gather_pack", "abc_adam_step", "abc_adam_chunk_elems", "abc_assemble_molblocks", "abc_gather_patches", "abc_gather_patches_pooled", "abc_rasterise_targets",
    "abc_unet_wpack_bytes", "abc_unet_workspace_bytes", "abc_unet_create", "abc_unet_forward_infer", "abc_unet_destroy", "abc_unet_pack_host",
    # deterministic reductions (torch.use_deterministic_algorithms)
    "abc_bn_stats_det", "abc_channel_sum_det", "abc_bn_stats_workspace_bytes", "abc_bn_act_backward_workspace_bytes",
    "abc_nchw_to_p8_ex_det", "abc_nchw_to_p8_ex_workspace_bytes", "abc_conv3x3_c1_wgrad_det", "abc_conv3x3_cn_wgrad_det",
    "abc_conv3x3_wgrad_workspace_bytes", "abc_conv_wgrad_workspace_bytes", "abc_conv_stat_workspace_bytes", "abc_loss_workspace_bytes",
)


class AbcConvDesc(C.Structure):
    _fields_ = [
        ("in_", C.c_void_p), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("in_planes", C.c_int), ("in_plane_off", C.c_int), ("cin", C.c_int),
        ("wpack", C.c_void_p), ("bias", C.c_void_p),
        ("cout", C.c_int), ("n_tile", C.c_int), ("ntaps", C.c_int),
        ("tap_dy", C.c_int * 9), ("tap_dx", C.c_int * 9),
        ("act", C.c_int), ("out_mode", C.c_int),
        ("out", C.c_void_p), ("out_planes", C.c_int), ("out_plane_off", C.c_int),
        ("out_H", C.c_int), ("out_W", C.c_int),
        ("out_sy", C.c_int), ("out_oy", C.c_int), ("out_sx", C.c_int), ("out_ox", C.c_int),
        ("pool_out", C.c_void_p), ("pool_planes", C.c_int), ("pool_plane_off", C.c_int),
        ("k_segments", C.c_int), ("seg_tap0", C.c_int * 4), ("seg_ntaps", C.c_int * 4),
        ("row_fold", C.c_int), ("cta_pair", C.c_int), ("swap_mn", C.c_int),
        ("stat_sum", C.c_void_p), ("stat_sq", C.c_void_p), ("subpixel", C.c_int), ("k_chunk", C.c_int), ("act_fp16", C.c_int),
        ("stat_ws", C.c_void_p),
    ]


class AbcUNetConfig(C.Structure):
    _fields_ = [("in_channels", C.c_int), ("n_heads", C.c_int), ("heads", C.c_int * 16), ("crop_first", C.c_int), ("act_fp16", C.c_int)]


class AbcNamedTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_int64)]


class AbcAtomRec(C.Structure):
    _fields_ = [("x", C.c_uint16), ("y", C.c_uint16), ("type", C.c_uint8), ("charge", C.c_uint8),
                ("hs", C.c_uint8), ("pad", C.c_uint8)]


class AbcBondRec(C.Structure):
    _fields_ = [("x", C.c_uint16), ("y", C.c_uint16), ("omega", C.c_uint8), ("type", C.c_uint8),
                ("pad", C.c_uint16), ("rho", C.c_float)]


class AbcDecodeDesc(C.Structure):
    _fields_ = [
        ("maps", C.c_void_p * 8), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("c_type", C.c_int), ("c_charge", C.c_int), ("c_hs", C.c_int), ("n_omega", C.c_int), ("n_btype", C.c_int),
        ("thr", C.c_float), ("omega_mode", C.c_int),
        ("atoms", C.c_void_p), ("atom_cap", C.c_int),
        ("bonds", C.c_void_p), ("bond_cap", C.c_int),
        ("counts", C.c_void_p), ("p8f_mask", C.c_int), ("centre_prob", C.c_int), ("thr_omega", C.c_float),
        ("peak_pix", C.c_void_p), ("peak_cnt", C.c_void_p), ("peak_cap", C.c_int), ("sparse_mode", C.c_int),
        ("peak_off", C.c_void_p), ("pool_slots", C.c_int),
    ]


class AbcTargetsDesc(C.Structure):
    _fields_ = [
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("n_omega", C.c_int), ("n_btype", C.c_int), ("c_type", C.c_int),
        ("c_charge", C.c_int), ("c_hs", C.c_int),
        ("atoms", C.c_void_p), ("atom_off", C.c_void_p), ("bonds", C.c_void_p), ("bond_rho", C.c_void_p), ("bond_off", C.c_void_p),
        ("atom_target", C.c_void_p), ("atom_type", C.c_void_p), ("atom_charge", C.c_void_p), ("atom_hs", C.c_void_p),
        ("bond_target", C.c_void_p), ("bond_type", C.c_void_p), ("bond_rho_map", C.c_void_p), ("bond_omega", C.c_void_p),
        ("f64", C.c_int), ("zero_first", C.c_int),
    ]


class AbcHeadsFusedDesc(C.Structure):
    _fields_ = [
        ("in_", C.c_void_p), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("in_planes", C.c_int), ("in_plane_off", C.c_int),
        ("w1pack", C.c_void_p), ("bias1", C.c_void_p), ("n_heads", C.c_int), ("cout", C.c_int * 16),
        ("w2pack", C.c_void_p), ("w2pack_bytes", C.c_int64), ("bias2", C.c_void_p), ("bias2_len", C.c_int),
        ("out", C.c_void_p * 16), ("out_mode", C.c_int * 16), ("out_planes", C.c_int * 16),
        ("act_fp16", C.c_int), ("trace", C.c_void_p),
    ]


class AbcBnActDesc(C.Structure):
    _fields_ = [
        ("z", C.c_void_p), ("z_planes", C.c_int), ("z_plane_off", C.c_int),
        ("out", C.c_void_p), ("out_planes", C.c_int), ("out_plane_off", C.c_int),
        ("pool", C.c_void_p), ("pool_planes", C.c_int), ("pool_plane_off", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("C", C.c_int),
        ("scale", C.c_void_p), ("shift", C.c_void_p),
        ("act", C.c_int), ("drop_p", C.c_float), ("seed", C.c_uint64), ("seed_dev", C.c_void_p), ("drop_mask", C.c_void_p),
    ]


class AbcBnActBwdDesc(C.Structure):
    _fields_ = [
        ("z", C.c_void_p), ("z_planes", C.c_int), ("z_plane_off", C.c_int),
        ("dA", C.c_void_p), ("dA_planes", C.c_int), ("dA_plane_off", C.c_int),
        ("dP", C.c_void_p), ("dP_planes", C.c_int), ("dP_plane_off", C.c_int),
        ("dz", C.c_void_p), ("dz_planes", C.c_int), ("dz_plane_off", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("C", C.c_int),
        ("scale", C.c_void_p), ("shift", C.c_void_p), ("mean", C.c_void_p), ("invstd", C.c_void_p),
        ("act", C.c_int), ("drop_p", C.c_float), ("seed", C.c_uint64),
        ("s1", C.c_void_p), ("s2", C.c_void_p), ("seed_dev", C.c_void_p), ("gscale", C.c_void_p), ("drop_mask", C.c_void_p),
        ("ws", C.c_void_p),
    ]


class AbcWgradDesc(C.Structure):
    _fields_ = [
        ("dz", C.c_void_p), ("dz_planes", C.c_int), ("dz_plane_off", C.c_int), ("cout", C.c_int),
        ("in_", C.c_void_p), ("in_planes", C.c_int), ("in_plane_off", C.c_int), ("cin", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("ntaps", C.c_int), ("tap_dy", C.c_int * 9), ("tap_dx", C.c_int * 9),
        ("dw", C.c_void_p), ("row_boxes", C.c_int), ("ws", C.c_void_p),
    ]


class AbcLossDesc(C.Structure):
    _fields_ = [
        ("logits", C.c_void_p * 8), ("targets", C.c_void_p * 8), ("tgt_f64", C.c_int),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("c_type", C.c_int), ("c_charge", C.c_int), ("c_hs", C.c_int), ("n_omega", C.c_int), ("n_btype", C.c_int),
        ("type_weights", C.c_void_p), ("sums", C.c_void_p), ("scale", C.c_void_p),
        ("dlogits", C.c_void_p * 8), ("ws", C.c_void_p),
    ]


class AbcLossP8Out(C.Structure):
    _fields_ = [("dz", C.c_void_p * 8), ("planes", C.c_int * 8), ("dbias", C.c_void_p * 8)]


assert C.sizeof(AbcAtomRec) == 8 and C.sizeof(AbcBondRec) == 12


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the abcnet_b200 CUDA library has not been built "
            "(run __graft_entry__.build() or `make -C abcnet_b200/csrc`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.abc_last_error.restype = C.c_char_p
    lib.abc_launch_count.restype = C.c_int64
    lib.abc_conv_wpack_bytes.restype = C.c_int64
    lib.abc_conv_wpack_bytes.argtypes = [C.c_int] * 4
    lib.abc_conv3x3_c1.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_void_p]
    lib.abc_conv3x3_c1_u8.argtypes = lib.abc_conv3x3_c1.argtypes
    lib.abc_conv3x3_cn.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.abc_conv3x3_stem.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.abc_conv3x3_cn_wgrad.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p]
    lib.abc_conv_igemm.argtypes = [C.POINTER(AbcConvDesc), C.c_void_p]
    lib.abc_decode_peaks.argtypes = [C.POINTER(AbcDecodeDesc), C.c_void_p]
    lib.abc_loss_partials.argtypes = [C.POINTER(AbcLossDesc), C.c_void_p]
    lib.abc_loss_backward.argtypes = [C.POINTER(AbcLossDesc), C.c_void_p]
    lib.abc_loss_partials_p8.argtypes = [C.POINTER(AbcLossDesc), C.POINTER(AbcLossP8Out), C.c_void_p]
    vp, ci = C.c_void_p, C.c_int
    lib.abc_bn_stats.argtypes = [vp, ci, ci, ci, ci, ci, ci, vp, vp, vp]
    lib.abc_channel_sum.argtypes = lib.abc_bn_stats.argtypes
    lib.abc_bn_finalize.argtypes = [vp, vp, ci, C.c_double, vp, vp, C.c_float, C.c_float, vp, vp, vp, vp, vp, vp, vp]
    lib.abc_bn_act.argtypes = [C.POINTER(AbcBnActDesc), vp]
    lib.abc_bn_act_backward.argtypes = [C.POINTER(AbcBnActBwdDesc), vp]
    lib.abc_nchw_to_p8.argtypes = [vp, vp, ci, ci, ci, ci, vp]
    lib.abc_nchw_to_p8_ex.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp]
    lib.abc_deinterleave2.argtypes = [vp, ci, ci, ci, vp, ci, ci, ci, vp]
    lib.abc_conv_wgrad.argtypes = [C.POINTER(AbcWgradDesc), vp]
    lib.abc_conv3x3_c1_wgrad.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, vp, vp]
    lib.abc_conv3x3_c1_raw.argtypes = [vp, ci, vp, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.abc_heads_fused.argtypes = [C.POINTER(AbcHeadsFusedDesc), vp]
    lib.abc_heads_fused_pack_sizes.argtypes = [ci, C.POINTER(C.c_int), C.POINTER(C.c_int64), C.POINTER(C.c_int)]
    lib.abc_gather_pack.argtypes = [vp, vp, vp, C.c_int64, ci, vp]
    lib.abc_adam_step.argtypes = [vp, vp, vp, vp, vp, vp, ci, vp, vp, vp]
    lib.abc_rasterise_targets.argtypes = [C.POINTER(AbcTargetsDesc), vp]
    lib.abc_gather_patches.argtypes = [vp, ci, ci, ci, ci, vp, vp, ci, vp, vp]
    lib.abc_gather_patches_pooled.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, ci, vp, vp]
    lib.abc_unet_wpack_bytes.restype = C.c_int64
    lib.abc_unet_wpack_bytes.argtypes = [C.POINTER(AbcUNetConfig)]
    lib.abc_unet_workspace_bytes.restype = C.c_int64
    lib.abc_unet_workspace_bytes.argtypes = [C.POINTER(AbcUNetConfig), ci, ci, ci]
    lib.abc_unet_create.argtypes = [C.POINTER(AbcUNetConfig), C.POINTER(AbcNamedTensor), ci, vp, C.c_int64, vp, C.POINTER(vp)]
    lib.abc_unet_forward_infer.argtypes = [vp, vp, ci, ci, ci, ci, vp, C.c_int64, C.POINTER(vp), ci, vp]
    lib.abc_unet_destroy.argtypes = [vp]
    lib.abc_unet_pack_host.argtypes = [C.POINTER(AbcUNetConfig), C.POINTER(AbcNamedTensor), ci, vp, C.c_int64, C.POINTER(C.c_int64)]
    lib.abc_assemble_molblocks.argtypes = [vp, ci, vp, ci, vp, ci, vp, vp, ci, ci, vp, C.c_int64, vp]
    lib.abc_bn_stats_det.argtypes = [vp, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp]
    lib.abc_channel_sum_det.argtypes = lib.abc_bn_stats_det.argtypes
    lib.abc_nchw_to_p8_ex_det.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp]
    lib.abc_conv3x3_c1_wgrad_det.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, vp, vp, vp]
    lib.abc_conv3x3_cn_wgrad_det.argtypes = [vp, ci, vp, ci, ci, ci, ci, ci, vp, vp, vp]
    sz = C.c_size_t
    for name, args in (("abc_bn_stats_workspace_bytes", [ci] * 4), ("abc_bn_act_backward_workspace_bytes", [C.POINTER(AbcBnActBwdDesc)]),
                       ("abc_nchw_to_p8_ex_workspace_bytes", [ci] * 5), ("abc_conv3x3_wgrad_workspace_bytes", [ci]),
                       ("abc_conv_wgrad_workspace_bytes", [C.POINTER(AbcWgradDesc)]),
                       ("abc_conv_stat_workspace_bytes", [C.POINTER(AbcConvDesc)]),
                       ("abc_loss_workspace_bytes", [C.POINTER(AbcLossDesc), ci])):
        getattr(lib, name).restype = sz
        getattr(lib, name).argtypes = args
    return lib


lib = _load()


def check(rc: int, what: str = "abcnet_b200") -> None:
    if rc != 0:
        msg = lib.abc_last_error()
        raise RuntimeError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")


def require_device() -> None:
    if not lib.abc_device_ok():
        msg = lib.abc_last_error()
        raise RuntimeError("abcnet_b200 needs an sm_100 (B200) CUDA device and has no CPU fallback: "
                           + (msg.decode() if msg else ""))


def current_stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(lib.abc_launch_count())
