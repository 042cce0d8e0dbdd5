"""GPU tests of the rows either side of the hot path (SURVEY.md section 8f), through the C ABI:
 * `vlg_ingest`                    uint8 dataset arrays -> normalised frames / labels / one-hot, bit-identical to
                                   the reference's torch expressions (src/data.py:33-35, src/trainer.py:193-206,
                                   src/folder.py:97-100, src/models/net_utils.py:14-24)
 * `vlg_warp_loss_labels_fwd_bwd`  the fused op with a label layout source: argmax bit-exact with the dense path,
                                   losses / d_flow at the fp32 parity bar against the oracle on one_hot(label)
 * argument validation and the debug status check of the Python surface."""
import numpy as np
import pytest
import torch

import vlg_b200
from vlg_b200 import _cabi
from conftest import assert_grad_parity, assert_terms_parity
from oracle import torch_oracle as TO
from test_gpu_parity import _cl, _make_case, TERMS

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5


# ------------------------------------------------------------------ ingest
@pytest.mark.parametrize("shape", [(2, 64, 96), (1, 37, 53), (3, 8, 4)])
@pytest.mark.parametrize("flip", [False, True])
def test_ingest_matches_reference_expressions_bit_for_bit(shape, flip):
    N, H, W = shape
    K = 20
    g = torch.Generator().manual_seed(7 + H)
    frames = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, generator=g)       # cv2 hands HWC uint8 (src/folder.py:122-127)
    seg = torch.randint(0, K, (N, H, W), dtype=torch.uint8, generator=g)
    # the reference, on the CPU exactly as its DataLoader workers and trainer do it
    t = frames.permute(0, 3, 1, 2).contiguous().to(torch.float32).div(255)               # transforms.ToTensor(), src/data.py:33-35
    mean = torch.tensor(TO.IMG_MEAN)[None, :, None, None]
    std = torch.tensor(TO.IMG_STD)[None, :, None, None]
    want = (t - mean) / std                                                              # src/trainer.py:193-195
    lab = seg.long()                                                                     # src/folder.py:100
    segf = seg.float().unsqueeze(1)                                                      # src/folder.py:97-99
    if flip:
        want, t = torch.flip(want, [3]), torch.flip(t, [3])                              # src/trainer.py:200-206
        lab, segf = torch.flip(lab, [2]), torch.flip(segf, [3])
    onehot = torch.eye(K)[lab].permute(0, 3, 1, 2)                                       # src/models/net_utils.py:23

    out = vlg_b200.ingest(frames.to(DEV), seg.to(DEV), flip=flip, want_label=True, want_seg_float=True, want_one_hot=True)
    assert torch.equal(out["frames"].cpu(), want)
    assert out["frames"].is_contiguous(memory_format=torch.channels_last) or W == 1
    assert torch.equal(out["label"].cpu(), lab) and out["label"].dtype == torch.int64
    assert torch.equal(out["seg_float"].cpu(), segf)
    assert torch.equal(out["one_hot"].cpu(), onehot)
    # ToTensor only, and bf16 outputs (rounded once from the fp32 value)
    raw = vlg_b200.ingest(frames.to(DEV), None, mean=None, flip=flip)["frames"]
    assert torch.equal(raw.cpu(), t)
    b16 = vlg_b200.ingest(frames.to(DEV), seg.to(DEV), flip=flip, dtype=torch.bfloat16, want_label=False, want_one_hot=True)
    assert torch.equal(b16["frames"].cpu(), want.to(torch.bfloat16))
    assert torch.equal(b16["one_hot"].cpu(), onehot.to(torch.bfloat16))
    # the same tensors through the older fp32 entry points
    assert torch.equal(vlg_b200.prepare_frames(t.to(DEV) if not flip else torch.flip(t, [3]).to(DEV), flip=flip).cpu(), want)
    assert torch.equal(vlg_b200.one_hot_layout(out["label"], K), out["one_hot"])


def test_ingest_feeds_the_fused_op():
    """End to end as bench.py's e2e leg does it: uint8 frames + class maps -> ingest -> fused op; equals the op on the
    tensors the reference would have built on the host."""
    N, H, W, K = 2, 48, 80, 20
    g = torch.Generator().manual_seed(3)
    f2 = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, generator=g)
    f3 = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, generator=g)
    s2 = torch.randint(0, K, (N, H // 8, W // 8), dtype=torch.uint8, generator=g).repeat_interleave(8, 1).repeat_interleave(8, 2)
    s3 = torch.randint(0, K, (N, H // 8, W // 8), dtype=torch.uint8, generator=g).repeat_interleave(8, 1).repeat_interleave(8, 2)
    flow = (torch.randn(N, H, W, 2, generator=g) * 1.5).to(DEV)
    a = vlg_b200.ingest(f2.to(DEV), s2.to(DEV), want_label=True, want_one_hot=True)
    b = vlg_b200.ingest(f3.to(DEV), s3.to(DEV), want_label=True)
    cfg = vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True)
    t1, v1, arg1 = vlg_b200.warp_loss(a["frames"], a["one_hot"], flow, b["frames"], b["label"], cfg)
    norm = lambda u8: (u8.permute(0, 3, 1, 2).float().div(255) - torch.tensor(TO.IMG_MEAN)[None, :, None, None]) / torch.tensor(TO.IMG_STD)[None, :, None, None]
    ref = TO.warp_loss(norm(f2), TO.one_hot_layout(s2.long(), K), flow.cpu(), norm(f3), s3.long(), w_tv=0.5)
    assert_terms_parity(v1.cpu().numpy()[:5], np.array([ref["terms"][k].item() for k in TERMS]), None, RTOL)
    assert torch.equal(arg1.cpu(), ref["argmax"])
    # label source == dense one-hot source
    t2, v2, arg2 = vlg_b200.warp_loss(a["frames"], a["label"], flow, b["frames"], b["label"], cfg)
    assert torch.equal(arg2, arg1)
    np.testing.assert_allclose(v2.cpu().numpy()[:6], v1.cpu().numpy()[:6], rtol=5e-6)


# ------------------------------------------------------------------ label-source fused op
F32, BF16 = torch.float32, torch.bfloat16
LAB_CASES = [
    # N, H, W, K, sigma, far_frac, w_tv, padding, half-pixel flow, rgb dtype
    (2, 128, 256, 20, 4.0, 0.0, 0.5, "border", False, F32),       # BASELINE config 1
    (2, 61, 93, 20, 3.0, 0.0, 0.3, "zeros", True, F32),           # ragged, zeros padding, exact ties between classes
    (1, 375, 1242, 20, 48.0, 0.05, 0.1, "border", False, F32),    # KITTI-shaped, large displacement
    (1, 40, 72, 19, 2.0, 0.0, 1.0, "border", False, F32),         # odd K: nothing in this kernel depends on K % 4
    (1, 33, 35, 5, 2.0, 0.0, 0.0, "zeros", False, F32),
    # bf16 rgb (rgb_strip_kernel<bf16>); the dense comparison then takes lay_tile_kernel (even W) / pass1_kernel (odd W)
    (2, 128, 256, 20, 4.0, 0.0, 0.5, "border", False, BF16),
    (2, 61, 93, 20, 3.0, 0.0, 0.3, "zeros", True, BF16),
    (1, 375, 1242, 20, 48.0, 0.05, 0.1, "border", False, BF16),
    (1, 33, 35, 5, 2.0, 0.0, 0.0, "zeros", False, BF16),
]


@pytest.mark.parametrize("case", LAB_CASES, ids=[f"{c[0]}x{c[1]}x{c[2]}k{c[3]}s{c[4]}{c[7]}" + ("" if c[9] == F32 else "-bf16")
                                                 for c in LAB_CASES])
def test_label_source_op_vs_oracle_and_dense_path(case):
    N, H, W, K, sigma, far, w_tv, padding, half, dt = case
    d = _make_case(N, H, W, K, sigma, seed=1024, layout="onehot", far_frac=far)
    # bf16 rgb: the oracle sees the same bf16-rounded values, in fp32; the one-hot layout is exact in bf16
    d = dict(d, **{k: d[k].to(dt).float() for k in ("src_rgb", "src_layout", "tgt_rgb")})
    flow = torch.round(d["flow"] * 2) / 2 if half else d["flow"]
    lab_src = d["src_layout"].argmax(1)
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], flow, d["tgt_rgb"], d["tgt_label"], w_tv=w_tv, padding_mode=padding)
    ref64 = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], flow, d["tgt_rgb"], d["tgt_label"], w_tv=w_tv, padding_mode=padding,
                                 dtype=torch.float64)
    cfg = vlg_b200.WarpLossConfig(w_tv=w_tv, padding_mode=padding, want_argmax=True)
    f = flow.to(DEV).requires_grad_(True)
    total, vec, arg = vlg_b200.warp_loss_labels(_cl(d["src_rgb"].to(dt)), lab_src.to(DEV), f, _cl(d["tgt_rgb"].to(dt)), d["tgt_label"].to(DEV), cfg,
                                                n_classes=K)
    total.backward()
    assert torch.equal(arg.cpu(), ref["argmax"])                                  # bit-exact layouts
    want = np.array([ref["terms"][k].item() for k in TERMS])
    want64 = np.array([ref64["terms"][k].item() for k in TERMS])
    assert_terms_parity(vec.cpu().numpy()[:5], want, want64, RTOL)
    np.testing.assert_allclose(vec[_cabi.LOSS_TOTAL].item(), ref["total"].item(), rtol=RTOL)
    assert_grad_parity(f.grad, ref["d_flow"], ref64["d_flow"], RTOL, "d_flow")
    # against the dense path of the product on the one-hot layout: same argmax, loss vector and d_flow to fp32 rounding
    if K % 4 == 0:
        f2 = flow.to(DEV).requires_grad_(True)
        t2, v2, a2 = vlg_b200.warp_loss(_cl(d["src_rgb"].to(dt)), _cl(d["src_layout"].to(dt)), f2, _cl(d["tgt_rgb"].to(dt)),
                                        d["tgt_label"].to(DEV), cfg)
        t2.backward()
        assert torch.equal(a2, arg)
        np.testing.assert_allclose(vec.cpu().numpy()[:6], v2.cpu().numpy()[:6], rtol=5e-6, atol=1e-7)
        assert_grad_parity(f.grad, f2.grad, None, 5e-6, "d_flow label source vs dense source")
    # validation mode (no gradient) and two runs bitwise identical
    with torch.no_grad():
        t3, v3, a3 = vlg_b200.warp_loss_labels(_cl(d["src_rgb"].to(dt)), lab_src.to(DEV), flow.to(DEV), _cl(d["tgt_rgb"].to(dt)),
                                               d["tgt_label"].to(DEV), cfg, n_classes=K)
    assert torch.equal(v3[:6], vec[:6]) and torch.equal(a3, arg)


def test_label_source_op_ignore_index_weights_and_full_size():
    """ignore_index, class weights (both normalisations) and BASELINE config 2 at full size against the oracle
    evaluated by torch CUDA."""
    N, H, W, K = 16, 256, 512, 20
    d = _make_case(N, H, W, K, 4.0, seed=1024)
    lab_src = d["src_layout"].argmax(1).to(DEV)
    lab = d["tgt_label"].clone()
    lab[:, :16] = -100
    w = torch.linspace(0.5, 2.0, K)
    ra, rb, rf = d["src_rgb"].to(DEV), d["src_layout"].to(DEV), d["flow"].to(DEV).requires_grad_(True)
    wl = TO.warp(rb, TO.flow_to_grid(rf))
    ce_mean = torch.nn.functional.cross_entropy(wl, lab.to(DEV), weight=w.to(DEV))
    ce_cnt = torch.nn.functional.cross_entropy(wl, lab.to(DEV), weight=w.to(DEV), reduction="sum") / (lab != -100).sum()
    g_mean, = torch.autograd.grad(ce_mean, rf, retain_graph=True)
    for norm, want, in (("torch", ce_mean), ("count", ce_cnt)):
        f = d["flow"].to(DEV).requires_grad_(True)
        cfg = vlg_b200.WarpLossConfig(w_l1=0, w_gd=0, w_ssim=0, w_ce=1.0, term_mask=_cabi.TERM_CE, class_weight=w.to(DEV), ce_norm=norm,
                                      want_argmax=True)
        total, vec, arg = vlg_b200.warp_loss_labels(None, lab_src, f, None, lab.to(DEV), cfg)
        total.backward()
        np.testing.assert_allclose(vec[_cabi.LOSS_CE].item(), want.item(), rtol=RTOL)
        assert vec[_cabi.LOSS_NVALID].item() == (lab != -100).sum().item()
        assert torch.equal(arg, torch.argmax(wl, 1))
        if norm == "torch":
            assert_grad_parity(f.grad, g_mean, None, RTOL, "d_flow (class-weighted CE)")


# ------------------------------------------------------------------ the Python surface refuses what raw pointers cannot check
def test_shape_and_device_validation():
    N, H, W, K = 1, 16, 24, 20
    rgb = torch.zeros(N, 3, H, W, device=DEV)
    lay = torch.zeros(N, K, H, W, device=DEV)
    flow = torch.zeros(N, H, W, 2, device=DEV)
    lab = torch.zeros(N, H, W, dtype=torch.int64, device=DEV)
    bad = [
        lambda: vlg_b200.warp_loss(rgb, lay, flow, torch.zeros(N, 3, H // 2, W // 2, device=DEV), lab),      # target at another pyramid scale
        lambda: vlg_b200.warp_loss(torch.zeros(N, 1, H, W, device=DEV), lay, flow, rgb, lab),                # 1-channel image
        lambda: vlg_b200.warp_loss(rgb, torch.zeros(N, K, H, W + 1, device=DEV), flow, rgb, lab),
        lambda: vlg_b200.warp_loss(rgb, lay, flow, rgb, lab[:, :-1]),
        lambda: vlg_b200.warp_loss(rgb, lay, flow.cpu(), rgb, lab),
        lambda: vlg_b200.warp(rgb, torch.zeros(N, K, H + 1, W, device=DEV), flow),
        lambda: vlg_b200.warp_labels(torch.zeros(N, 3, H, W + 2, device=DEV), lab, flow),
        lambda: vlg_b200.PixelLosses()(rgb, rgb[:, :, :-1], lay, lab),
        lambda: vlg_b200.ingest(torch.zeros(N, H, W, 4, dtype=torch.uint8, device=DEV)),
    ]
    for fn in bad:
        with pytest.raises(vlg_b200.VlgError):
            fn()
    torch.cuda.synchronize()          # nothing was launched with a bad pointer


def test_debug_mode_raises_on_bad_labels_and_far_taps():
    """nn.CrossEntropyLoss device-asserts on a label outside [0,K); the product sets a status bit and, with
    debug=True, raises (the default path never synchronises)."""
    d = _make_case(1, 32, 64, 20, 1.0, seed=5, layout="soft")
    lab = d["tgt_label"].clone()
    lab[0, 3, 5] = 25
    args = (_cl(d["src_rgb"]), _cl(d["src_layout"]), d["flow"].to(DEV), _cl(d["tgt_rgb"]))
    vlg_b200.warp_loss(*args, lab.to(DEV))                                                  # silent by default
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        vlg_b200.warp_loss(*args, lab.to(DEV), vlg_b200.WarpLossConfig(debug=True))
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        vlg_b200.WarpLoss(debug=True)(*args, lab.to(DEV))
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        vlg_b200.warp_loss_labels(args[0], d["src_layout"].argmax(1).to(DEV), args[2], args[3], lab.to(DEV), vlg_b200.WarpLossConfig(debug=True))
    vlg_b200.warp_loss(*args, d["tgt_label"].to(DEV), vlg_b200.WarpLossConfig(debug=True))   # clean labels pass
    far = d["flow"].clone()
    far[0, 10, 10] = 9.0
    a = args[0].clone().requires_grad_(True)
    with pytest.raises(vlg_b200.VlgError, match="assume_near"):
        vlg_b200.warp_loss(a, args[1], far.to(DEV), args[3], d["tgt_label"].to(DEV), vlg_b200.WarpLossConfig(debug=True, assume_near=True))
