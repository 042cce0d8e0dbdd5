"""ctypes binding of include/vlg_b200.h.  No fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

F32, BF16 = 0, 1
PAD_ZEROS, PAD_BORDER = 0, 1
COORD_FLOW, COORD_GRID = 0, 1
FLAG_NO_FAR_PATH = 1
FLAG_NO_TMA = 2
FLAG_PASS2_COORDS = 32
FLAG_FAR_WIDE = 64
TERM_L1, TERM_GD, TERM_SSIM, TERM_CE, TERM_TV, TERM_ALL = 1, 2, 4, 8, 16, 31
STATUS_BAD_LABEL, STATUS_FAR_TAPS = 1, 2
CE_NORM_TORCH, CE_NORM_COUNT = 0, 1
NEAR_RADIUS = 3
LOSS_L1, LOSS_GD, LOSS_SSIM, LOSS_CE, LOSS_TV, LOSS_TOTAL, LOSS_NVALID, LOSS_MAXDISP, LOSS_SLOTS = range(9)

ABI_VERSION = 200

EXPORTS = [
    "vlg_version", "vlg_last_error", "vlg_workspace_bytes", "vlg_warp_fwd", "vlg_warp_fwd_labels", "vlg_colorize", "vlg_confusion",
    "vlg_one_hot",
    "vlg_frame_affine", "vlg_ingest", "vlg_warp_loss_labels_fwd_bwd",
    "vlg_warp_loss_bwd_out", "vlg_warp_loss_pass1",
    "vlg_warp_bwd_src", "vlg_reduce_partials", "vlg_warp_loss_fwd_bwd", "vlg_pixel_loss_fwd_bwd",
    "vlg_scale_grads", "vlg_scale_grads_multi", "vlg_read_status", "vlg_launch_count", "vlg_timeline_arm", "vlg_timeline_read",
]


class Problem(C.Structure):
    """Mirror of vlg_problem_t (include/vlg_b200.h).  `struct_size` / `abi_version` are filled in by the
    constructor; the library refuses a descriptor whose size differs from its own (stale binding)."""
    _fields_ = [
        ("struct_size", C.c_uint32), ("abi_version", C.c_uint32),
        ("N", C.c_int64), ("H", C.c_int64), ("W", C.c_int64), ("K", C.c_int64),
        ("dtype", C.c_int32), ("padding", C.c_int32), ("coord_mode", C.c_int32), ("flags", C.c_uint32),
        ("ignore_index", C.c_int64),
        ("w_l1", C.c_float), ("w_gd", C.c_float), ("w_ssim", C.c_float), ("w_ce", C.c_float), ("w_tv", C.c_float),
        ("term_mask", C.c_uint32), ("ce_norm", C.c_uint32),
        ("global_N", C.c_int64), ("ce_class_weight", C.c_void_p),
    ]


    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        if "struct_size" not in kw:
            self.struct_size = C.sizeof(Problem)
        if "abi_version" not in kw:
            self.abi_version = ABI_VERSION


class VlgError(RuntimeError):
    pass


_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Load libvlg_b200.so (building it in-tree first if nvcc is available and it is stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    override = os.environ.get("VLG_B200_LIB")   # kernel-tuning experiments: another build of this same library
    if override:
        path, build_if_missing = override, False
    if build_if_missing and _build.is_stale():
        # A library older than its sources is never used silently: rebuild (atomically, under a file lock) or fail.
        # On a box without nvcc a library that is present is accepted as shipped (the GPU box receives the built .so).
        try:
            have_nvcc = bool(_build._nvcc())
        except RuntimeError:
            have_nvcc = False
        if have_nvcc or not os.path.exists(path):
            try:
                _build.build_library()
            except Exception as exc:
                raise VlgError(f"libvlg_b200.so is stale or missing and could not be rebuilt: {exc}") from exc
    if not os.path.exists(path):
        raise VlgError("libvlg_b200.so is missing; run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    vp, i64p, f32p = C.c_void_p, C.c_void_p, C.c_void_p
    P = C.POINTER(Problem)
    lib.vlg_version.restype = C.c_int
    lib.vlg_last_error.restype = C.c_char_p
    lib.vlg_launch_count.restype = C.c_int64
    lib.vlg_workspace_bytes.restype = C.c_size_t
    lib.vlg_workspace_bytes.argtypes = [P, C.c_int]
    lib.vlg_warp_fwd.argtypes = [P, vp, vp, f32p, vp, vp, i64p, vp, vp]
    lib.vlg_warp_fwd_labels.argtypes = [P, vp, i64p, f32p, vp, i64p, vp]
    lib.vlg_colorize.argtypes = [P, vp, i64p, vp, vp, i64p, vp]
    lib.vlg_colorize.restype = C.c_int
    lib.vlg_confusion.argtypes = [P, vp, C.c_int32, i64p, i64p, vp, vp]
    lib.vlg_confusion.restype = C.c_int
    lib.vlg_one_hot.argtypes = [P, i64p, f32p, vp, vp, vp]
    lib.vlg_one_hot.restype = C.c_int
    lib.vlg_frame_affine.argtypes = [P, f32p, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, C.c_int32, vp, i64p, i64p, vp]
    lib.vlg_frame_affine.restype = C.c_int
    lib.vlg_ingest.argtypes = [P, vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, vp, vp, i64p, f32p, vp, vp, vp]
    lib.vlg_ingest.restype = C.c_int
    lib.vlg_warp_loss_labels_fwd_bwd.argtypes = [P, vp, i64p, f32p, vp, i64p, f32p, f32p, i64p, vp, C.c_size_t, vp]
    lib.vlg_warp_loss_labels_fwd_bwd.restype = C.c_int
    lib.vlg_warp_loss_bwd_out.argtypes = [P, vp, vp, f32p, vp, i64p, f32p, i64p, C.c_int, vp, C.c_size_t, vp]
    lib.vlg_warp_loss_pass1.argtypes = [P, vp, vp, f32p, vp, i64p, f32p, f32p, i64p, C.c_int, vp, C.c_size_t, vp]
    lib.vlg_warp_loss_pass1.restype = C.c_int
    lib.vlg_warp_bwd_src.argtypes = [P, f32p, vp, vp, vp, C.c_size_t, vp]
    lib.vlg_reduce_partials.argtypes = [P, f32p, vp, C.c_size_t, vp]
    lib.vlg_warp_loss_fwd_bwd.argtypes = [P, vp, vp, f32p, vp, i64p, f32p, f32p, vp, vp, i64p, vp, C.c_size_t, vp]
    lib.vlg_pixel_loss_fwd_bwd.argtypes = [P, vp, vp, vp, i64p, f32p, vp, vp, i64p, vp, C.c_size_t, vp]
    lib.vlg_scale_grads.argtypes = [vp, C.c_int64, C.c_int32, f32p, vp]
    lib.vlg_scale_grads_multi.argtypes = [C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32), f32p, vp]
    lib.vlg_read_status.argtypes = [vp, C.c_size_t, C.POINTER(C.c_uint32), vp]
    lib.vlg_timeline_arm.argtypes = [C.c_int]
    lib.vlg_timeline_arm.restype = C.c_int
    lib.vlg_timeline_read.argtypes = [C.POINTER(C.c_float)]
    lib.vlg_timeline_read.restype = C.c_int
    for name in ("vlg_warp_fwd", "vlg_warp_fwd_labels", "vlg_warp_loss_bwd_out", "vlg_warp_bwd_src", "vlg_reduce_partials",
                 "vlg_warp_loss_fwd_bwd", "vlg_pixel_loss_fwd_bwd", "vlg_scale_grads", "vlg_scale_grads_multi", "vlg_read_status"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise VlgError(f"vlg error {rc}: {load().vlg_last_error().decode()}")


def launch_count() -> int:
    return int(load().vlg_launch_count())
