"""Torch-facing operators over the C ABI (include/vlg_b200.h).

Everything here is plumbing: device memory comes from torch's allocator, the stream is torch's
current stream, the arithmetic happens in libvlg_b200.so.  There is NO CPU / eager fallback: a
non-CUDA tensor or a missing library raises.

Call signatures mirror the reference's (SURVEY.md section 8b): image tensors are NCHW-logical
(`[N,3,H,W]`, `[N,K,H,W]`), labels int64 `[N,H,W]` (src/folder.py:100).  Tensors already in
`torch.channels_last` storage are consumed in place; NCHW-contiguous ones get ONE explicit
permute-copy.  `flow` / `grid` are `[N,H,W,2]` fp32 (x first), i.e. the channels_last storage of a
`[N,2,H,W]` flow head.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Tuple

import torch

from . import _cabi
from ._cabi import Problem, VlgError, check

_DTYPES = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16}
_PADDING = {"zeros": _cabi.PAD_ZEROS, "border": _cabi.PAD_BORDER}


@dataclass
class WarpLossConfig:
    """Weights follow src/trainer.py:248-250 (40*L1 + 20*(GD+SSIM) + 10*CE); w_tv is new."""
    w_l1: float = 40.0
    w_gd: float = 20.0
    w_ssim: float = 20.0
    w_ce: float = 10.0
    w_tv: float = 0.0
    padding_mode: str = "border"          # oracle default (SURVEY Appendix A.4)
    coords_are_grid: bool = False         # False: pixel flow; True: normalised sampling grid
    ignore_index: int = -100              # nn.CrossEntropyLoss default (src/trainer.py:124)
    global_batch: int = 0                 # data-parallel: divisor batch (0 = local batch)
    assume_near: bool = False             # caller asserts |flow| < NEAR_RADIUS: skip far-path launches
    use_tma: bool = True                  # stage source layout rows / windows with TMA tensor maps when possible
    pass2_records: bool = True            # pass 2 gathers from the tap records pass 1 wrote (all staging by TMA);
                                          # False: it re-derives them from the coordinates (first pass-2 kernel)
    far_packed: bool = True               # far path packs two 32-bit lanes per 64-bit atomic where the far-pixel count of a source-tile row allows
                                          # (False: always one 64-bit accumulator per channel)
    term_mask: int = 0                    # 0 = all terms
    class_weight: Optional[torch.Tensor] = None   # per-class CE weights (K floats on the device)
    ce_norm: str = "torch"                # 'torch' (weighted mean) | 'count' (sum / n_known, src/models/simple.py:56-59)
    want_argmax: bool = False
    debug: bool = False                   # read the device status word after the call (synchronises) and raise on labels
                                          # outside [0,K) (nn.CrossEntropyLoss device-asserts there) / far taps under assume_near


def _require_cuda(*tensors):
    """All tensors on ONE CUDA device (no CPU fallback); returns that device."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise VlgError("video-layout-generation_b200 runs on CUDA tensors only (no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise VlgError(f"all tensors must live on one device (got {dev} and {t.device})")
    return dev


def _expect(t: Optional[torch.Tensor], shape, what: str, dtype=None):
    """torch would raise a shape error where raw pointers would read out of bounds: check before data_ptr()."""
    if t is None:
        return
    if tuple(t.shape) != tuple(shape):
        raise VlgError(f"{what} must have shape {tuple(shape)}, got {tuple(t.shape)}")
    if dtype is not None and t.dtype != dtype:
        raise VlgError(f"{what} must be {dtype}, got {t.dtype}")


def _nhwc_strides(shape):
    N, Cc, H, W = shape
    return (H * W * Cc, 1, W * Cc, Cc)


def to_nhwc(x: torch.Tensor) -> torch.Tensor:
    """Return `x` (NCHW-logical) backed by dense NHWC storage; no copy if it already is."""
    if x.dim() != 4:
        raise VlgError(f"expected a 4-d NCHW-logical tensor, got shape {tuple(x.shape)}")
    want = _nhwc_strides(x.shape)
    ok = all(x.shape[d] == 1 or x.stride(d) == want[d] for d in range(4))
    if ok and x.data_ptr() % 16 == 0:
        return x
    y = torch.empty_strided(x.shape, want, dtype=x.dtype, device=x.device)
    y.copy_(x)
    return y


def empty_nhwc(shape, dtype, device) -> torch.Tensor:
    return torch.empty_strided(tuple(shape), _nhwc_strides(shape), dtype=dtype, device=device)


def _coords(c: torch.Tensor, N, H, W) -> torch.Tensor:
    if c.dtype != torch.float32:
        raise VlgError("flow / grid must be float32 (bf16 cannot address 2048 columns)")
    if tuple(c.shape) != (N, H, W, 2):
        raise VlgError(f"flow / grid must be [N,H,W,2]={N, H, W, 2}, got {tuple(c.shape)}")
    return c.contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


# torch.cuda.current_stream() and the torch.cuda.device() context manager cost 15-20 us of Python each (device-index
# resolution, availability checks); an end-to-end step used a dozen of them -- a fifth of its host time.  The raw
# accessors below are what they end in.
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """The current stream of the current device as a ctypes pointer."""
    if _raw_stream is not None and _raw_device is not None:
        return C.c_void_p(_raw_stream(_raw_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _NoSwitch:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def _on(dev):
    """Context that makes `dev` current -- a no-op object when it already is (the usual case: one process per GPU)."""
    if _raw_device is not None and dev is not None and dev.index is not None and _raw_device() == dev.index:
        return _NO_SWITCH
    return torch.cuda.device(dev)


def _class_weight_ptr(cfg: "WarpLossConfig", K: int):
    w = cfg.class_weight
    if w is None:
        return None
    if not w.is_cuda or w.dtype != torch.float32 or w.numel() != K or not w.is_contiguous():
        raise VlgError(f"class_weight must be a contiguous float32 CUDA tensor of {K} elements")
    return w.data_ptr()


def _problem(N, H, W, K, dtype, cfg: WarpLossConfig) -> Problem:
    if dtype not in _DTYPES:
        raise VlgError(f"unsupported activation dtype {dtype}; use float32 or bfloat16")
    flags = (_cabi.FLAG_NO_FAR_PATH if cfg.assume_near else 0) | (0 if cfg.use_tma else _cabi.FLAG_NO_TMA)
    if not cfg.pass2_records:
        flags |= _cabi.FLAG_PASS2_COORDS
    if not cfg.far_packed:
        flags |= _cabi.FLAG_FAR_WIDE
    return Problem(N=N, H=H, W=W, K=K, dtype=_DTYPES[dtype], padding=_PADDING[cfg.padding_mode],
                   coord_mode=_cabi.COORD_GRID if cfg.coords_are_grid else _cabi.COORD_FLOW, flags=flags,
                   ignore_index=cfg.ignore_index, w_l1=cfg.w_l1, w_gd=cfg.w_gd, w_ssim=cfg.w_ssim,
                   w_ce=cfg.w_ce, w_tv=cfg.w_tv, term_mask=cfg.term_mask,
                   ce_norm=_cabi.CE_NORM_COUNT if cfg.ce_norm == "count" else _cabi.CE_NORM_TORCH,
                   global_N=cfg.global_batch, ce_class_weight=_class_weight_ptr(cfg, K))


# Workspaces are scratch for ONE call (both passes are launched inside it; the gradients live in their own
# tensors), so successive calls on the same stream reuse one buffer: stream order serialises them.  Keyed by
# (device, stream); grown on demand; a handful of streams at most.
_WS_CACHE: dict = {}


def _workspace(prob: Problem, with_src: bool, device, cached: bool = True) -> torch.Tensor:
    lib = _cabi.load()
    n = lib.vlg_workspace_bytes(C.byref(prob), int(with_src))
    if n == 0:
        raise VlgError(lib.vlg_last_error().decode())
    if not cached:
        return torch.empty(n, dtype=torch.uint8, device=device)
    device = torch.device(device)
    if _raw_stream is not None and device.index is not None:
        key = (device.index, _raw_stream(device.index))
    else:
        key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _WS_CACHE.get(key)
    if ws is None or ws.numel() < n:
        if len(_WS_CACHE) >= 8:
            _WS_CACHE.clear()
        ws = torch.empty(n, dtype=torch.uint8, device=device)
        _WS_CACHE[key] = ws
    return ws


def _check_status(ws: torch.Tensor, cfg: "WarpLossConfig"):
    """debug mode: the status word is sticky until the next pass-1 launch on this workspace."""
    st = read_status(ws)
    if st & _cabi.STATUS_BAD_LABEL:
        raise VlgError("a target label lies outside [0, K) and is not ignore_index (nn.CrossEntropyLoss asserts on the device here)")
    if st & _cabi.STATUS_FAR_TAPS:
        raise VlgError(f"assume_near=True but a sampling position lies >= {_cabi.NEAR_RADIUS} px from its pixel: "
                       "source-gradient contributions were dropped")


# --------------------------------------------------------------------------- forward-only warp
@torch.no_grad()
def warp(src_rgb: Optional[torch.Tensor], src_layout: Optional[torch.Tensor], coords: torch.Tensor, *,
         padding_mode: str = "border", coords_are_grid: bool = False, want_layout: bool = True,
         want_argmax: bool = True, debug_indices: bool = False):
    """Validation / rollout warp (src/trainer.py:329-342,460-469).  Returns
    (warped_rgb | None, warped_layout | None, argmax | None[, x0y0 int32])."""
    lib = _cabi.load()
    dev = _require_cuda(src_rgb, src_layout, coords)
    ref = src_rgb if src_rgb is not None else src_layout
    if ref is None:
        raise VlgError("warp needs at least one source tensor")
    if ref.dim() != 4:
        raise VlgError(f"sources must be NCHW-logical 4-d tensors, got shape {tuple(ref.shape)}")
    N, _, H, W = ref.shape
    K = src_layout.shape[1] if src_layout is not None else 20
    _expect(src_rgb, (N, 3, H, W), "src_rgb")
    _expect(src_layout, (N, K, H, W), "src_layout", ref.dtype)
    cfg = WarpLossConfig(padding_mode=padding_mode, coords_are_grid=coords_are_grid)
    prob = _problem(N, H, W, K, ref.dtype, cfg)
    coords = _coords(coords, N, H, W)
    a = to_nhwc(src_rgb) if src_rgb is not None else None
    b = to_nhwc(src_layout) if src_layout is not None else None
    out_rgb = empty_nhwc((N, 3, H, W), ref.dtype, dev) if a is not None else None
    out_lay = empty_nhwc((N, K, H, W), ref.dtype, dev) if (b is not None and want_layout) else None
    out_arg = torch.empty((N, H, W), dtype=torch.int64, device=dev) if (b is not None and want_argmax) else None
    dbg = torch.empty((N, H, W, 2), dtype=torch.int32, device=dev) if debug_indices else None
    with _on(dev):
        check(lib.vlg_warp_fwd(C.byref(prob), _ptr(a), _ptr(b), _ptr(coords), _ptr(out_rgb), _ptr(out_lay),
                               _ptr(out_arg), _ptr(dbg), _stream()))
    res = (out_rgb, out_lay, out_arg)
    return res + (dbg,) if debug_indices else res


@torch.no_grad()
def warp_labels(src_rgb: Optional[torch.Tensor], src_label: torch.Tensor, coords: torch.Tensor, *,
                padding_mode: str = "border", coords_are_grid: bool = False):
    """Rollout warp with an integer label map as the layout source: returns (warped_rgb | None,
    warped_label int64 [N,H,W]) where warped_label == argmax(warp(one_hot(src_label))) bit for bit,
    at 8 B/px of layout traffic instead of 80 (SURVEY section 8f-2)."""
    lib = _cabi.load()
    dev = _require_cuda(src_rgb, src_label, coords)
    if src_label.dtype != torch.int64 or src_label.dim() != 3:
        raise VlgError("src_label must be int64 [N,H,W]")
    N, H, W = src_label.shape
    _expect(src_rgb, (N, 3, H, W), "src_rgb")
    dt = src_rgb.dtype if src_rgb is not None else torch.float32
    prob = _problem(N, H, W, 20, dt, WarpLossConfig(padding_mode=padding_mode, coords_are_grid=coords_are_grid))
    coords = _coords(coords, N, H, W)
    a = to_nhwc(src_rgb) if src_rgb is not None else None
    lab = src_label.contiguous()
    out_rgb = empty_nhwc((N, 3, H, W), dt, lab.device) if a is not None else None
    out_lab = torch.empty_like(lab)
    with _on(dev):
        check(lib.vlg_warp_fwd_labels(C.byref(prob), _ptr(a), _ptr(lab), _ptr(coords), _ptr(out_rgb), _ptr(out_lab), _stream()))
    return out_rgb, out_lab


# Cityscapes train-id palette (19 classes + "None"), the table `vis_seg_mask` indexes at
# src/trainer.py:31-52,416-427
CITYSCAPES_PALETTE = (
    (128, 64, 128), (244, 35, 232), (70, 70, 70), (102, 102, 156), (190, 153, 153), (153, 153, 153),
    (250, 170, 30), (220, 220, 0), (107, 142, 35), (152, 251, 152), (70, 130, 180), (220, 20, 60),
    (255, 0, 0), (0, 0, 142), (0, 0, 70), (0, 60, 100), (0, 80, 100), (0, 0, 230), (119, 11, 32), (0, 0, 0))


@torch.no_grad()
def colorize(seg: torch.Tensor, n_classes: int = 20, argmax: bool = False, palette=CITYSCAPES_PALETTE,
             dtype=torch.float32):
    """`Trainer.vis_seg_mask(seg, n_classes, argmax)` (src/trainer.py:416-427): layout -> RGB in [0,1].
    seg: [N,K,H,W] scores (argmax=True) or int64 [N,H,W] class ids.  Returns [N,3,H,W] (channels_last)."""
    lib = _cabi.load()
    _require_cuda(seg)
    if len(palette) != n_classes:
        raise VlgError("palette length must equal n_classes")
    lut = torch.tensor(palette, dtype=torch.uint8, device=seg.device).contiguous()
    if argmax:
        N, K, H, W = seg.shape
        if K != n_classes:
            raise VlgError("seg has a different number of channels than n_classes")
        lay, lab, dt = to_nhwc(seg), None, seg.dtype
    else:
        if seg.dtype != torch.int64 or seg.dim() != 3:
            raise VlgError("class-id input must be int64 [N,H,W]")
        N, H, W = seg.shape
        lay, lab, dt = None, seg.contiguous(), dtype
    prob = _problem(N, H, W, n_classes, dt, WarpLossConfig())
    out = empty_nhwc((N, 3, H, W), dt, seg.device)
    with _on(seg.device):
        check(lib.vlg_colorize(C.byref(prob), _ptr(lay), _ptr(lab), _ptr(lut), _ptr(out), None, _stream()))
    return out


@torch.no_grad()
def _confusion_into(counts: torch.Tensor, pred: torch.Tensor, target: torch.Tensor, n_classes: int = 20, *,
                   ignore_index: int = -100):
    """Adds the confusion counts of (pred, target) into `counts`, one vlg_confusion launch, no synchronisation and no
    allocation when the inputs need no copy.  `counts` is int64 [K*K + 1] on the device, contiguous: row-major
    [target, prediction] bins, then the pixels skipped for a label outside [0, K).  `pred` is int64 [N,H,W] class ids or
    [N,K,H,W] fp32 / bf16 scores (argmax taken on the device; channels_last and plain-contiguous are read as they are,
    any other stride pattern gets one copy); `target` is int64 [N,H,W]; pixels whose target is `ignore_index` count
    nowhere."""
    lib = _cabi.load()
    dev = _require_cuda(counts, pred, target)
    K = n_classes
    if target.dim() != 3:
        raise VlgError(f"target must be int64 [N,H,W], got shape {tuple(target.shape)}")
    N, H, W = target.shape
    _expect(target, (N, H, W), "target", torch.int64)
    _expect(counts, (K * K + 1,), "counts", torch.int64)
    if not counts.is_contiguous():
        raise VlgError("counts must be contiguous")
    lay = lab = None
    nchw = 0
    if pred.dtype == torch.int64:
        _expect(pred, (N, H, W), "pred (class ids)")
        lab, dt = pred.contiguous(), torch.float32
    else:
        _expect(pred, (N, K, H, W), "pred (scores)")
        dt = pred.dtype
        if all(pred.shape[d] == 1 or pred.stride(d) == _nhwc_strides(pred.shape)[d] for d in range(4)):
            lay = to_nhwc(pred)
        else:
            lay, nchw = pred.contiguous(), 1
    prob = _problem(N, H, W, K, dt, WarpLossConfig(ignore_index=ignore_index))
    tgt = target.contiguous()
    with _on(dev):
        check(lib.vlg_confusion(C.byref(prob), _ptr(lay), nchw, _ptr(lab), _ptr(tgt), _ptr(counts), _stream()))


@torch.no_grad()
def confusion_matrix(pred: torch.Tensor, target: torch.Tensor, n_classes: int = 20, *, ignore_index: int = -100,
                     debug: bool = False) -> torch.Tensor:
    """Confusion matrix of a predicted layout against the target labels: int64 [K, K] on the device, rows = target class,
    columns = predicted class.  `pred` is int64 [N,H,W] class ids or [N,K,H,W] fp32 / bf16 scores, whose argmax (first
    maximal index, as `torch.argmax(seg, 1)` at src/trainer.py:342) is taken on the device; `target` is int64 [N,H,W].
    Pixels whose target is `ignore_index` count nowhere; pixels with a target or prediction outside [0, K) count nowhere
    either -- `debug=True` reads their number (synchronises) and raises if it is not 0."""
    counts = torch.zeros(n_classes * n_classes + 1, dtype=torch.int64, device=target.device)
    _confusion_into(counts, pred, target, n_classes, ignore_index=ignore_index)
    if debug:
        skipped = int(counts[-1])
        if skipped:
            raise VlgError(f"{skipped} pixels have a target or predicted label outside [0, {n_classes}) (and not ignore_index)")
    return counts[:-1].view(n_classes, n_classes)


@torch.no_grad()
def one_hot_layout(seg: torch.Tensor, n_classes: int = 20, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """`transform_seg_one_hot` (src/models/net_utils.py:14-24): class-id map -> one-hot layout.

    `seg` is [N,H,W] or [N,1,H,W], int64 or float32 class ids (the dataset hands float maps,
    src/folder.py:97-99; truncated like `.long()`).  Returns an NCHW-logical [N,K,H,W] tensor in NHWC
    storage, ready to be a `src_layout` -- so a data pipeline uploads 4-8 bytes per pixel instead of 4*K."""
    _require_cuda(seg)
    if seg.dim() == 4:
        if seg.shape[1] != 1:
            raise VlgError("one_hot_layout expects class ids of shape [N,H,W] or [N,1,H,W]")
        seg = seg[:, 0]
    if seg.dtype not in (torch.int64, torch.float32):
        raise VlgError("one_hot_layout expects int64 or float32 class ids")
    seg = seg.contiguous()
    N, H, W = seg.shape
    prob = _problem(N, H, W, n_classes, dtype, WarpLossConfig())
    out = empty_nhwc((N, n_classes, H, W), dtype, seg.device)
    lib = _cabi.load()
    li, lf = (_ptr(seg), None) if seg.dtype == torch.int64 else (None, _ptr(seg))
    with _on(seg.device):
        check(lib.vlg_one_hot(C.byref(prob), li, lf, _ptr(out), None, _stream()))
    return out


# src/trainer.py:120-123
IMG_MEAN, IMG_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)          # img_mean_arr, img_std_arr
OUT_MEAN, OUT_STD = (-0.03, -0.088, -0.188), (0.448, 0.448, 0.450)        # mean_arr, std_arr


@torch.no_grad()
def prepare_frames(frames: torch.Tensor, mean=IMG_MEAN, std=IMG_STD, *, flip: bool = False, denormalize: bool = False,
                   labels: Optional[torch.Tensor] = None, dtype: torch.dtype = torch.float32):
    """Per-channel renormalisation (+ optional horizontal flip and NCHW -> NHWC re-layout) in one pass.

    normalise   `(frames - mean[None,:,None,None]) / std[None,:,None,None]`   src/trainer.py:193-195,212,324
    denormalize `frames * std + mean`                                          src/trainer.py:215
    flip        `torch.flip(frames, [3])`, `torch.flip(labels, [2])`           src/trainer.py:200-206
    `frames` is fp32 [N,3,H,W], plain-contiguous (what the DataLoader hands) or channels_last; the result is an
    NCHW-logical tensor in NHWC storage of `dtype`, bit-identical to the torch expressions above.  With `labels`
    ([N,H,W] int64) returns (frames, labels)."""
    _require_cuda(frames, labels)
    if frames.dim() != 4 or frames.shape[1] != 3 or frames.dtype != torch.float32:
        raise VlgError("prepare_frames expects float32 frames of shape [N,3,H,W]")
    N, _, H, W = frames.shape
    nhwc = all(frames.shape[d] == 1 or frames.stride(d) == _nhwc_strides(frames.shape)[d] for d in range(4))
    if not nhwc:
        frames = frames.contiguous()
    prob = _problem(N, H, W, 20, dtype, WarpLossConfig())
    out = empty_nhwc((N, 3, H, W), dtype, frames.device)
    a3, b3 = (C.c_float * 3)(*[float(v) for v in mean]), (C.c_float * 3)(*[float(v) for v in std])
    lab_out = None
    if labels is not None:
        if labels.dtype != torch.int64 or tuple(labels.shape) != (N, H, W):
            raise VlgError(f"labels must be int64 [N,H,W]={N, H, W}")
        labels = labels.contiguous()
        lab_out = torch.empty_like(labels)
    with _on(frames.device):
        check(_cabi.load().vlg_frame_affine(C.byref(prob), _ptr(frames), int(not nhwc), a3, b3, int(denormalize), int(flip),
                                            _ptr(out), _ptr(labels), _ptr(lab_out), _stream()))
    return out if labels is None else (out, lab_out)


_F3_CACHE: dict = {}


def _float3(v):
    """(C float)[3] of a mean / std triple, cached by value."""
    if v is None:
        return None
    key = tuple(float(x) for x in v)
    arr = _F3_CACHE.get(key)
    if arr is None:
        arr = _F3_CACHE[key] = (C.c_float * 3)(*key)
    return arr


@torch.no_grad()
def ingest(frames_u8: Optional[torch.Tensor] = None, seg_u8: Optional[torch.Tensor] = None, *, mean=IMG_MEAN, std=IMG_STD,
           flip: bool = False, n_classes: int = 20, dtype: torch.dtype = torch.float32, want_label: bool = True,
           want_seg_float: bool = False, want_one_hot: bool = False):
    """What the dataset holds -> what the path consumes, one pass per tensor, bit-identical to the reference's
    torch expressions (so a data pipeline uploads 3 + 1 bytes per pixel instead of 12 + 4 / 8).

    frames_u8 uint8 [N,H,W,3] (cv2 / dataset layout, src/folder.py:122-127): `ToTensor()` (src/data.py:33-35, u8 / 255)
              then `(frame - img_mean_arr) / img_std_arr` (src/trainer.py:193-195; mean=None: ToTensor only), optional
              `torch.flip(frame, [3])` (:200-206) -> NCHW-logical [N,3,H,W] tensor of `dtype` in NHWC storage.
    seg_u8    uint8 [N,H,W] class ids (src/folder.py:95-96): `.long()` labels [N,H,W] (:100), `.float()` class maps
              [N,1,H,W] (:97-99), one-hot layout [N,K,H,W] (`transform_seg_one_hot`, src/models/net_utils.py:14-24), flipped
              along W with the frames.
    Returns a dict with the requested entries among 'frames', 'label', 'seg_float', 'one_hot'."""
    dev = _require_cuda(frames_u8, seg_u8)
    if frames_u8 is None and seg_u8 is None:
        raise VlgError("ingest needs frames_u8 and / or seg_u8")
    ref = frames_u8 if frames_u8 is not None else seg_u8
    N, H, W = ref.shape[0], ref.shape[1], ref.shape[2]
    _expect(frames_u8, (N, H, W, 3), "frames_u8", torch.uint8)
    _expect(seg_u8, (N, H, W), "seg_u8", torch.uint8)
    prob = _problem(N, H, W, n_classes, dtype, WarpLossConfig())
    out = {}
    f_in = frames_u8.contiguous() if frames_u8 is not None else None
    s_in = seg_u8.contiguous() if seg_u8 is not None else None
    if f_in is not None:
        out["frames"] = empty_nhwc((N, 3, H, W), dtype, dev)
    if s_in is not None:
        if want_label:
            out["label"] = torch.empty((N, H, W), dtype=torch.int64, device=dev)
        if want_seg_float:
            out["seg_float"] = torch.empty((N, 1, H, W), dtype=torch.float32, device=dev)
        if want_one_hot:
            out["one_hot"] = empty_nhwc((N, n_classes, H, W), dtype, dev)
        if not (want_label or want_seg_float or want_one_hot):
            raise VlgError("seg_u8 given but no output requested for it")
    m3, s3 = _float3(mean), (_float3(std) if mean is not None else None)
    with _on(dev):
        check(_cabi.load().vlg_ingest(C.byref(prob), _ptr(f_in), m3, s3, int(flip), _ptr(out.get("frames")), _ptr(s_in),
                                      _ptr(out.get("label")), _ptr(out.get("seg_float")), _ptr(out.get("one_hot")), None, _stream()))
    return out


def rollout(img: torch.Tensor, label: torch.Tensor, flow_fn, steps: int = 5, *, padding_mode: str = "border"):
    """Autoregressive rollout (shape of src/trainer.py:453-476, which runs 8 steps and feeds the
    argmax back): step t warps the previous frame and label map with `flow_fn(t, img, label)`
    ([N,H,W,2] pixels) and feeds both back.  Returns (list of frames, list of label maps)."""
    imgs, labels = [img], [label]
    for t in range(steps):
        flow = flow_fn(t, imgs[-1], labels[-1])
        nxt_img, nxt_lab = warp_labels(imgs[-1], labels[-1], flow, padding_mode=padding_mode)
        imgs.append(nxt_img)
        labels.append(nxt_lab)
    return imgs[1:], labels[1:]


def _scale_all(tensors, g_total):
    """g <- g * g_total for every gradient buffer, on the device, in ONE launch (it exits at once when g_total == 1)."""
    ts = [t for t in tensors if t is not None]
    if not ts:
        return
    g = g_total.detach().to(torch.float32).contiguous()
    n = len(ts)
    ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    sizes = (C.c_int64 * n)(*[t.numel() for t in ts])
    dts = (C.c_int32 * n)(*[_DTYPES[t.dtype] for t in ts])
    with _on(g.device):
        check(_cabi.load().vlg_scale_grads_multi(n, ptrs, sizes, dts, _ptr(g), _stream()))


# --------------------------------------------------------------------------- fused warp + loss
class _WarpLossFn(torch.autograd.Function):
    """Fused forward+backward: the gradients are produced by the SAME pass as the losses (for an
    upstream gradient of 1) and rescaled on the device in backward() only if it differs from 1."""

    @staticmethod
    def forward(ctx, src_rgb, src_layout, coords, tgt_rgb, tgt_label, cfg: WarpLossConfig):
        lib = _cabi.load()
        dev = _require_cuda(src_rgb, src_layout, coords, tgt_rgb, tgt_label)
        if src_rgb.dim() != 4 or src_layout.dim() != 4:
            raise VlgError("src_rgb / src_layout must be NCHW-logical 4-d tensors")
        N, _, H, W = src_rgb.shape
        K = src_layout.shape[1]
        dt = src_rgb.dtype
        _expect(src_rgb, (N, 3, H, W), "src_rgb")
        _expect(src_layout, (N, K, H, W), "src_layout", dt)
        _expect(tgt_rgb, (N, 3, H, W), "tgt_rgb", dt)
        _expect(tgt_label, (N, H, W), "tgt_label (src/folder.py:100)", torch.int64)
        prob = _problem(N, H, W, K, dt, cfg)
        need_c, need_a, need_b = ctx.needs_input_grad[2], ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_src = need_a or need_b
        need_any = need_c or need_src
        a, b, t = to_nhwc(src_rgb), to_nhwc(src_layout), to_nhwc(tgt_rgb)
        c = _coords(coords, N, H, W)
        lab = tgt_label.contiguous()
        ws = _workspace(prob, need_src, dev)
        loss = torch.empty(_cabi.LOSS_SLOTS, dtype=torch.float32, device=dev)
        d_c = torch.empty_like(c) if need_any else None
        d_a = empty_nhwc(a.shape, dt, dev) if need_src else None
        d_b = empty_nhwc(b.shape, dt, dev) if need_src else None
        arg = torch.empty((N, H, W), dtype=torch.int64, device=dev) if cfg.want_argmax else None
        with _on(dev):
            check(lib.vlg_warp_loss_fwd_bwd(C.byref(prob), _ptr(a), _ptr(b), _ptr(c), _ptr(t), _ptr(lab), _ptr(loss),
                                            _ptr(d_c), _ptr(d_a), _ptr(d_b), _ptr(arg), _ptr(ws), ws.numel(), _stream()))
            if cfg.debug:
                _check_status(ws, cfg)
        ctx.grads = (d_a if need_a else None, d_b if need_b else None, d_c if need_c else None)
        ctx.consumed = False
        total = loss[_cabi.LOSS_TOTAL].clone()   # own storage: `loss` itself is returned non-differentiable
        ctx.mark_non_differentiable(*([loss] if arg is None else [loss, arg]))  # one call only
        return total, loss, arg

    @staticmethod
    def backward(ctx, g_total, g_loss, g_arg):
        if ctx.consumed:
            raise VlgError("the fused warp-loss gradients were already consumed (retain_graph is unsupported)")
        ctx.consumed = True
        lib = _cabi.load()
        d_a, d_b, d_c = ctx.grads
        ctx.grads = None     # sole owner from here on: autograd adopts the buffers as .grad instead of cloning them (a 100 B/px copy)
        _scale_all((d_a, d_b, d_c), g_total)
        return d_a, d_b, d_c, None, None, None


class _WarpLossLabelsFn(torch.autograd.Function):
    """The fused op with a LABEL layout source (sources are data: the gradient goes to the coordinates only)."""

    @staticmethod
    def forward(ctx, src_rgb, src_label, coords, tgt_rgb, tgt_label, cfg: WarpLossConfig, n_classes: int):
        lib = _cabi.load()
        dev = _require_cuda(src_rgb, src_label, coords, tgt_rgb, tgt_label)
        if src_label.dim() != 3 or src_label.dtype != torch.int64:
            raise VlgError("src_label must be int64 [N,H,W] class ids")
        N, H, W = src_label.shape
        dt = src_rgb.dtype if src_rgb is not None else torch.float32
        _expect(src_rgb, (N, 3, H, W), "src_rgb")
        _expect(tgt_rgb, (N, 3, H, W), "tgt_rgb", dt)
        _expect(tgt_label, (N, H, W), "tgt_label (src/folder.py:100)", torch.int64)
        if (src_rgb is None) != (tgt_rgb is None):
            raise VlgError("src_rgb and tgt_rgb go together")
        prob = _problem(N, H, W, n_classes, dt, cfg)
        need_c = ctx.needs_input_grad[2]
        a = to_nhwc(src_rgb) if src_rgb is not None else None
        t = to_nhwc(tgt_rgb) if tgt_rgb is not None else None
        c = _coords(coords, N, H, W)
        ws = _workspace(prob, False, dev)
        loss = torch.empty(_cabi.LOSS_SLOTS, dtype=torch.float32, device=dev)
        d_c = torch.empty_like(c) if need_c else None
        arg = torch.empty((N, H, W), dtype=torch.int64, device=dev) if cfg.want_argmax else None
        with _on(dev):
            check(lib.vlg_warp_loss_labels_fwd_bwd(C.byref(prob), _ptr(a), _ptr(src_label.contiguous()), _ptr(c), _ptr(t),
                                                   _ptr(tgt_label.contiguous()), _ptr(loss), _ptr(d_c), _ptr(arg), _ptr(ws),
                                                   ws.numel(), _stream()))
            if cfg.debug:
                _check_status(ws, cfg)
        ctx.grad_c = d_c
        ctx.consumed = False
        total = loss[_cabi.LOSS_TOTAL].clone()
        ctx.mark_non_differentiable(*([loss] if arg is None else [loss, arg]))
        return total, loss, arg

    @staticmethod
    def backward(ctx, g_total, g_loss, g_arg):
        if ctx.consumed:
            raise VlgError("the fused warp-loss gradients were already consumed (retain_graph is unsupported)")
        ctx.consumed = True
        d_c, ctx.grad_c = ctx.grad_c, None     # see _WarpLossFn.backward
        if d_c is not None:
            g = g_total.detach().to(torch.float32).contiguous()
            with _on(g.device):
                check(_cabi.load().vlg_scale_grads(_ptr(d_c), d_c.numel(), _cabi.F32, _ptr(g), _stream()))
        return None, None, d_c, None, None, None, None


def warp_loss_labels(src_rgb, src_label, coords, tgt_rgb, tgt_label, cfg: Optional[WarpLossConfig] = None, n_classes: int = 20):
    """`warp_loss` with the layout source given as the int64 class-id map [N,H,W] the reference's dataset holds
    (it stands for one_hot(src_label), src/models/net_utils.py:14-24): same losses, argmax bit-exact with the dense
    path, 8 B/px of layout traffic instead of 80, differentiable w.r.t. coords only (the sources are data).
    Returns (total, loss_vector[LOSS_SLOTS], argmax | None)."""
    return _WarpLossLabelsFn.apply(src_rgb, src_label, coords, tgt_rgb, tgt_label, cfg or WarpLossConfig(), n_classes)


def warp_loss(src_rgb, src_layout, coords, tgt_rgb, tgt_label, cfg: Optional[WarpLossConfig] = None):
    """Returns (total, loss_vector[LOSS_SLOTS], argmax | None).  `total` is differentiable w.r.t.
    coords (flow / grid), src_rgb and src_layout.  An int64 [N,H,W] `src_layout` is a label source
    (see warp_loss_labels)."""
    if src_layout is not None and src_layout.dim() == 3 and src_layout.dtype == torch.int64:
        return warp_loss_labels(src_rgb, src_layout, coords, tgt_rgb, tgt_label, cfg)
    return _WarpLossFn.apply(src_rgb, src_layout, coords, tgt_rgb, tgt_label, cfg or WarpLossConfig())


# --------------------------------------------------------------------------- reference call sites
class _PixelLossFn(torch.autograd.Function):
    """The reference's own criteria (no warp): L1 / GradientLoss / SsimLoss on (output, target),
    cross-entropy on (input, target) -- src/trainer.py:248-250, src/loss.py:16-25,64-91."""

    @staticmethod
    def forward(ctx, out_rgb, tgt_rgb, logits, tgt_label, cfg: WarpLossConfig):
        lib = _cabi.load()
        dev = _require_cuda(out_rgb, tgt_rgb, logits, tgt_label)
        ref = out_rgb if out_rgb is not None else logits
        if ref is None or ref.dim() != 4:
            raise VlgError("expected NCHW-logical 4-d tensors")
        N, _, H, W = ref.shape
        K = logits.shape[1] if logits is not None else 20
        dt = ref.dtype
        _expect(out_rgb, (N, 3, H, W), "output rgb")
        _expect(tgt_rgb, (N, 3, H, W), "target rgb")
        _expect(logits, (N, K, H, W), "logits", dt)
        if (out_rgb is None) != (tgt_rgb is None) or (logits is None) != (tgt_label is None):
            raise VlgError("(output, target) go together")
        prob = _problem(N, H, W, K, dt, cfg)
        need_a = out_rgb is not None and ctx.needs_input_grad[0]
        need_z = logits is not None and ctx.needs_input_grad[2]
        a = to_nhwc(out_rgb) if out_rgb is not None else None
        t = to_nhwc(tgt_rgb.to(dt)) if tgt_rgb is not None else None
        z = to_nhwc(logits) if logits is not None else None
        lab = tgt_label.contiguous() if tgt_label is not None else None
        if lab is not None and (lab.dtype != torch.int64 or tuple(lab.shape) != (N, H, W)):
            raise VlgError("target labels must be int64 [N,H,W]")
        ws = _workspace(prob, False, dev)
        loss = torch.empty(_cabi.LOSS_SLOTS, dtype=torch.float32, device=dev)
        d_a = empty_nhwc(a.shape, dt, dev) if need_a else None
        d_z = empty_nhwc(z.shape, dt, dev) if need_z else None
        arg = torch.empty((N, H, W), dtype=torch.int64, device=dev) if (cfg.want_argmax and z is not None) else None
        with _on(dev):
            check(lib.vlg_pixel_loss_fwd_bwd(C.byref(prob), _ptr(a), _ptr(t), _ptr(z), _ptr(lab), _ptr(loss), _ptr(d_a),
                                             _ptr(d_z), _ptr(arg), _ptr(ws), ws.numel(), _stream()))
            if cfg.debug:
                _check_status(ws, cfg)
        ctx.grads = (d_a, d_z)
        ctx.consumed = False
        ctx.mark_non_differentiable(*([loss] if arg is None else [loss, arg]))  # one call only
        return loss[_cabi.LOSS_TOTAL].clone(), loss, arg

    @staticmethod
    def backward(ctx, g_total, g_loss, g_arg):
        if ctx.consumed:
            raise VlgError("the fused pixel-loss gradients were already consumed (retain_graph is unsupported)")
        ctx.consumed = True
        lib = _cabi.load()
        d_a, d_z = ctx.grads
        ctx.grads = None     # see _WarpLossFn.backward
        _scale_all((d_a, d_z), g_total)
        return d_a, None, d_z, None, None


def pixel_losses(out_rgb, tgt_rgb, logits, tgt_label, cfg: Optional[WarpLossConfig] = None):
    """Returns (total, loss_vector, argmax | None) for the reference's un-warped loss call sites."""
    return _PixelLossFn.apply(out_rgb, tgt_rgb, logits, tgt_label, cfg or WarpLossConfig())


def read_status(workspace: torch.Tensor) -> int:
    """Synchronising debug helper: VLG_STATUS_* bits left by the last pass on this workspace."""
    st = C.c_uint32(0)
    with _on(workspace.device):
        check(_cabi.load().vlg_read_status(_ptr(workspace), workspace.numel(), C.byref(st), _stream()))
    return st.value
