"""ctypes binding of libcstp_b200.so (the C ABI declared in include/cstp_b200.h).

There is no CPU fallback: every compute entry point needs the CUDA library and a B200.  Importing this module
only loads the shared object (which works without a GPU, e.g. to check the exported symbols).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

CSTP_MAX_AMAPS = 4
CSTP_MAX_TAPS = 32
CSTP_MAX_MCHUNKS = 96


class Tensor5(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("dims", C.c_int32 * 5), ("strides", C.c_int64 * 4)]


class Tap(C.Structure):
    _fields_ = [("map_id", C.c_int32), ("dw", C.c_int32), ("dh", C.c_int32), ("dt", C.c_int32), ("k_off", C.c_int32)]


class Prologue(C.Structure):
    """cstp_prologue: BatchNorm affine + ReLU applied to the activation operand inside the kernel."""
    _fields_ = [("scale", C.c_void_p), ("shift", C.c_void_p), ("groups", C.c_int32), ("Cp", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("n_amaps", C.c_int32),
        ("amap", Tensor5 * CSTP_MAX_AMAPS),
        ("a_channels", C.c_int32),
        ("n_taps", C.c_int32),
        ("taps", Tap * CSTP_MAX_TAPS),
        ("w_packed", C.c_void_p),
        ("Np", C.c_int32),
        ("Ktot", C.c_int32),
        ("n_tile", C.c_int32),
        ("Wt", C.c_int32), ("Ht", C.c_int32), ("Tt", C.c_int32), ("Nt", C.c_int32),
        ("bw", C.c_int32), ("bh", C.c_int32), ("bt", C.c_int32), ("bn", C.c_int32),
        ("out_bf16", C.c_void_p),
        ("out_f32", C.c_void_p),
        ("out_off", C.c_int64),
        ("osw", C.c_int64), ("osh", C.c_int64), ("ost", C.c_int64), ("osn", C.c_int64),
        ("bias", C.c_void_p),
        ("accumulate", C.c_int32),
        ("pro", Prologue),
        ("n_classes", C.c_int32),
        ("cls_first_tap", C.c_int32 * 8),
        ("cls_n_taps", C.c_int32 * 8),
        ("cls_out_off", C.c_int64 * 8),
    ]


class MChunk(C.Structure):
    _fields_ = [("map_id", C.c_int32), ("dw", C.c_int32), ("dh", C.c_int32), ("dt", C.c_int32), ("c_off", C.c_int32)]


class WgradDesc(C.Structure):
    _fields_ = [
        ("n_amaps", C.c_int32),
        ("amap", Tensor5 * CSTP_MAX_AMAPS),
        ("n_mchunks", C.c_int32),
        ("mchunks", MChunk * CSTP_MAX_MCHUNKS),
        ("gmap", Tensor5),
        ("Np", C.c_int32),
        ("n_tile", C.c_int32),
        ("Wt", C.c_int32), ("Ht", C.c_int32), ("Tt", C.c_int32), ("Nt", C.c_int32),
        ("bw", C.c_int32), ("bh", C.c_int32), ("bt", C.c_int32), ("bn", C.c_int32),
        ("splits", C.c_int32),
        ("partials", C.c_void_p),
        ("pro", Prologue),
        ("mt_per_cta", C.c_int32),
    ]


class HaloGroup(C.Structure):
    _fields_ = [("dw", C.c_int32), ("dh", C.c_int32), ("dt", C.c_int32), ("first_tap", C.c_int32), ("n_taps", C.c_int32)]


class HaloTap(C.Structure):
    _fields_ = [("a_shift", C.c_uint32), ("k_off", C.c_int32)]


class HaloSlabs(C.Structure):
    _fields_ = [("n_slabs", C.c_int32), ("axis", C.c_int32), ("nslots", C.c_int32)]


class ConvHaloDesc(C.Structure):
    _fields_ = [
        ("amap", Tensor5),
        ("a_channels", C.c_int32),
        ("n_groups", C.c_int32),
        ("groups", HaloGroup * 4),
        ("n_taps", C.c_int32),
        ("taps", HaloTap * 16),
        ("w_packed", C.c_void_p),
        ("Np", C.c_int32), ("Ktot", C.c_int32), ("n_tile", C.c_int32),
        ("Wt", C.c_int32), ("Ht", C.c_int32), ("Tt", C.c_int32), ("Nt", C.c_int32),
        ("bw", C.c_int32), ("bh", C.c_int32), ("bt", C.c_int32), ("bn", C.c_int32),
        ("halo_w", C.c_int32), ("halo_h", C.c_int32), ("halo_t", C.c_int32),
        ("out_bf16", C.c_void_p),
        ("out_f32", C.c_void_p),
        ("out_off", C.c_int64),
        ("osw", C.c_int64), ("osh", C.c_int64), ("ost", C.c_int64), ("osn", C.c_int64),
        ("bias", C.c_void_p),
        ("accumulate", C.c_int32),
        ("allow_resident", C.c_int32),
        ("use_tail_boxes", C.c_int32),
        ("atom_pitch_rows", C.c_int32),
        ("stats_groups", C.c_int32),
        ("stats_partials", C.c_void_p),
        ("pro", Prologue),
        ("slabs", HaloSlabs),
    ]


class XBox(C.Structure):
    _fields_ = [("c_off", C.c_int32), ("dw", C.c_int32), ("dh", C.c_int32), ("dt", C.c_int32)]


class WgradHaloDesc(C.Structure):
    _fields_ = [
        ("xmap", Tensor5), ("gmap", Tensor5),
        ("n_xboxes", C.c_int32),
        ("xboxes", XBox * 16),
        ("n_chunks", C.c_int32),
        ("chunk_off", C.c_uint32 * 32),
        ("Np", C.c_int32), ("n_tile", C.c_int32),
        ("Wt", C.c_int32), ("Ht", C.c_int32), ("Tt", C.c_int32), ("Nt", C.c_int32),
        ("bw", C.c_int32), ("bh", C.c_int32), ("bt", C.c_int32), ("bn", C.c_int32),
        ("halo_w", C.c_int32), ("halo_h", C.c_int32), ("halo_t", C.c_int32),
        ("splits", C.c_int32),
        ("partials", C.c_void_p),
        ("atom_pitch_rows", C.c_int32),
        ("pro", Prologue),
        ("mt_per_class", C.c_int32),
        ("pro_on_b", C.c_int32),
    ]


CSTP_CLIP_T = 64
CSTP_CLIP_S = 224
CSTP_CLIP_KMAX = 24


class ClipView(C.Structure):
    """cstp_clip_view: one output clip of the pretraining clip pipeline (include/cstp_b200.h)."""
    _fields_ = [
        ("video", C.c_void_p), ("out", C.c_void_p), ("coef", C.c_void_p),
        ("W", C.c_int32), ("H", C.c_int32),
        ("frames", C.c_int32 * CSTP_CLIP_T),
        ("rot", C.c_int32),
        ("box", C.c_int32 * 4),
        ("flip", C.c_int32),
        ("rotate", C.c_int32),
        ("rot_fix", C.c_int32 * 6),
        ("n_jitter", C.c_int32),
        ("jitter_op", C.c_int32 * 4),
        ("jitter_f", C.c_float * 4),
        ("hue_shift", C.c_int32),
        ("gray", C.c_int32 * CSTP_CLIP_T),
        ("blur", C.c_int32),
        ("blur_radius", C.c_int32), ("blur_edge_a", C.c_int32), ("blur_edge_b", C.c_int32),
        ("blur_ww", C.c_uint32), ("blur_fw", C.c_uint32),
    ]


class JpegImage(C.Structure):
    """cstp_jpeg_image: one stream of a `cstp_jpeg_decode` batch (include/cstp_b200.h)."""
    _fields_ = [("src_offset", C.c_int64), ("src_bytes", C.c_int64), ("out", C.c_void_p),
                ("width", C.c_int32), ("height", C.c_int32), ("ws_offset", C.c_int64)]


CSTP_JPEG_UNSUPPORTED, CSTP_JPEG_MALFORMED, CSTP_JPEG_SIZE = 1, 2, 3


class AdamHyper(C.Structure):
    """cstp_adam_hyper: the scalars of one Adam / AdamW step (include/cstp_b200.h); ten floats, also as a device vector."""
    _fields_ = [(n, C.c_float) for n in ("step_size", "bc2_sqrt", "one_minus_beta1", "beta2", "one_minus_beta2", "eps",
                                         "l2", "decay", "max_norm", "do_clip")]

_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> (restype, argtypes); the single source of truth for the symbols include/cstp_b200.h declares.
SIGNATURES = {
    "cstp_last_error": (C.c_char_p, []),
    "cstp_version": (_i, []),
    "cstp_launch_count": (C.c_longlong, []),
    "cstp_conv_plan_create": (_i, [C.POINTER(ConvDesc), C.POINTER(_vp)]),
    "cstp_conv_plan_run": (_i, [_vp, _vp]),
    "cstp_conv_plan_cluster": (_i, [_vp]),
    "cstp_conv_plan_destroy": (None, [_vp]),
    "cstp_conv_halo_plan_create": (_i, [C.POINTER(ConvHaloDesc), C.POINTER(_vp)]),
    "cstp_conv_halo_plan_resident": (_i, [_vp]),
    "cstp_conv_halo_plan_stat_blocks": (_i, [_vp]),
    "cstp_conv_halo_plan_run": (_i, [_vp, _vp]),
    "cstp_conv_halo_plan_destroy": (None, [_vp]),
    "cstp_wgrad_plan_create": (_i, [C.POINTER(WgradDesc), C.POINTER(_vp)]),
    "cstp_wgrad_plan_splits": (_i, [_vp]),
    "cstp_wgrad_plan_run": (_i, [_vp, _vp]),
    "cstp_wgrad_plan_destroy": (None, [_vp]),
    "cstp_wgrad_halo_plan_create": (_i, [C.POINTER(WgradHaloDesc), C.POINTER(_vp)]),
    "cstp_wgrad_halo_plan_splits": (_i, [_vp]),
    "cstp_wgrad_halo_plan_run": (_i, [_vp, _vp]),
    "cstp_wgrad_halo_plan_destroy": (None, [_vp]),
    "cstp_wgrad_finalize": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "cstp_wgrad_halo_plan_chunk_splits": (_i, [_vp, _vp, _i]),
    "cstp_pack_weight": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "cstp_pack_weights_batched": (_i, [_vp, _vp, _i, _i64, _vp]),
    "cstp_stem_pack": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "cstp_bn_stats": (_i, [_vp, _i64, _i, _i, _vp, _i, _vp]),
    "cstp_bn_partials_reduce": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "cstp_bn_finalize": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cstp_bn_apply": (_i, [_vp, _i64, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "cstp_bn_bwd_reduce": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "cstp_bn_bwd_finalize": (_i, [_vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "cstp_bn_bwd_apply": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cstp_avgpool_fwd": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _i, _vp]),
    "cstp_avgpool_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "cstp_colsum": (_i, [_vp, _i64, _i, _i, _vp, _i, _vp]),
    "cstp_cast_pad": (_i, [_vp, _i64, _i, _i, _vp, _i, _vp, _vp]),
    "cstp_byol_loss": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "cstp_repr_stats": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp]),
    "cstp_pretext_ce": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _i, _i, _i, _vp, _vp, _vp]),
    "cstp_ntxent_workspace_floats": (C.c_longlong, [_i, _i]),
    "cstp_ntxent": (_i, [_vp, _i, _i, _f, _i, _vp, _vp, _vp, C.c_longlong, _vp]),
    "cstp_l2norm_fwd": (_i, [_vp, _i, _i, _i, _f, _vp, _i, _vp, _vp]),
    "cstp_l2norm_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "cstp_ce_loss": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "cstp_bn_eval_coeffs": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp]),
    "cstp_ema_update": (_i, [_vp, _vp, _i64, _f, _f, _vp]),
    "cstp_sgd_clip_step": (_i, [_vp, _vp, _vp, _i64, _f, _f, _f, _f, _i, _i, _vp, _vp, _vp]),
    "cstp_sgd_clip_step_dev": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "cstp_adam_clip_step": (_i, [_vp, _vp, _vp, _vp, _i64, AdamHyper, _vp, _vp, _vp]),
    "cstp_adam_clip_step_dev": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "cstp_clip_assemble": (_i, [_vp, _i, _i, _i, _i, _vp]),
    "cstp_clip_layout": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "cstp_video_accumulate": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _i, _vp]),
    "cstp_video_finalize": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "cstp_l2_normalize_rows": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "cstp_knn_partial": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "cstp_knn_merge": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "cstp_jpeg_workspace_bytes": (C.c_longlong, [_i, _i]),
    "cstp_jpeg_decode": (_i, [_vp, _vp, _i, _vp, _vp, C.c_longlong, _vp]),
    "cstp_bn_sync_buffer_bytes": (C.c_longlong, [_i, _i, _i]),
    "cstp_bn_sync_exchange": (_i, [_vp, _i, _vp, _i, _i, _i, _i, C.c_uint32, _vp, _vp, _vp, _vp]),
}

_lib = None


class CstpError(RuntimeError):
    """A C-ABI call returned a CSTP_E* code (the message comes from cstp_last_error())."""


def lib_path() -> Path:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Loads (building first if needed) libcstp_b200.so and installs the argtypes of every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not path.exists():
        if not build_if_missing:
            raise CstpError(f"{path} is missing: run `python -m cstp_b200.build` (there is no CPU fallback)")
        _build.build()
    elif build_if_missing and _build.is_stale():      # sources edited since the library was built here
        _build.build()
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().cstp_last_error().decode(errors="replace")
        raise CstpError(f"cstp_b200 call failed (code {rc}): {msg}")
