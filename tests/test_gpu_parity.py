"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against
 (1) the committed golden fixtures (real reference loss modules + torch 2.11 CPU grid_sample),
 (2) the oracle (oracle/torch_oracle.py, oracle/warp_oracle.c) on seeded inputs,
 (3) size-independent properties at BASELINE.json's full sizes.

Bars (BASELINE.json north_star): sampling indices and argmax bit-exact; losses and gradients
within 1e-5 relative in fp32.  bf16 runs compute in fp32 and round once at the store: their fp32 outputs (losses,
d_flow) meet the fp32 bar and their bf16 outputs are the fp32 result rounded once (bf16_bars).  No test in this file
asserts a wider bar.  For gradient
tensors "relative" is evaluated normwise-max AND RMS-relative (conftest.assert_grad_parity; element-wise
relative error is meaningless where terms cancel), against the fp32 oracle or -- where torch's own
atomic-ordered fp32 scatter drifts -- the fp64 evaluation of the same oracle (SURVEY Appendix A.10).
"""
import numpy as np
import pytest
import torch

import vlg_b200
from vlg_b200 import _cabi
from conftest import assert_grad_parity, assert_terms_parity, golden_names, load_golden
from bf16_bars import assert_bf16_rounded_once
from oracle import c_oracle as CO
from oracle import torch_oracle as TO

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
TERMS = ["l1", "gd", "ssim", "ce", "tv"]


def _cl(x):  # NCHW numpy/tensor -> channels_last CUDA tensor
    t = torch.as_tensor(x).to(DEV)
    return t.contiguous(memory_format=torch.channels_last)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def _nchw(t):
    return t.detach().float().cpu().contiguous().numpy()


def _assert_close_norm(got, ref, rtol, what):
    """Normwise-max AND RMS-relative error of a gradient tensor against one oracle evaluation."""
    assert_grad_parity(got, ref, None, rtol, what)


def _assert_close_either(got, ref32, ref64, rtol, what):
    """SURVEY Appendix A.10: torch's own fp32 accumulation drifts by ~1e-5 where thousands of
    contributions meet (border pixels under large displacement); an fp64 evaluation of the same
    oracle is the tie-breaker.  Pass if within rtol of EITHER (normwise-max and RMS-relative)."""
    assert_grad_parity(got, ref32, ref64, rtol, what)


def _gpu_oracle(d, dtype, w_tv=0.5, padding="border", flow=None, label=None):
    """The oracle (oracle/torch_oracle.py) evaluated by torch CUDA in `dtype` on the case `d`: returns the dict of
    TO.warp_loss_fwd_bwd (terms, argmax, warped_*, d_flow, d_src_rgb, d_src_layout), tensors on the device."""
    dev = lambda t: t.to(DEV)
    return TO.warp_loss_fwd_bwd(dev(d["src_rgb"]), dev(d["src_layout"]), dev(d["flow"] if flow is None else flow), dev(d["tgt_rgb"]),
                                dev(d["tgt_label"] if label is None else label), w_tv=w_tv, padding_mode=padding, dtype=dtype)


def _terms(ref):
    return np.array([ref["terms"][k].item() for k in TERMS])


def _cfg(g, **kw):
    return vlg_b200.WarpLossConfig(w_tv=g["w_tv"], padding_mode=g["padding"], **kw)


# ------------------------------------------------------------------ goldens: forward warp
@pytest.mark.parametrize("name", golden_names())
def test_warp_forward_bit_exact_vs_golden(name):
    g = load_golden(name)
    flow = torch.as_tensor(g["flow"]).to(DEV)
    out_rgb, out_lay, arg, dbg = vlg_b200.warp(_cl(g["src_rgb"]), _cl(g["src_layout"]), flow,
                                               padding_mode=g["padding"], debug_indices=True)
    assert (_bits(_nchw(out_rgb)) == _bits(g["warped_rgb"])).all()
    assert (_bits(_nchw(out_lay)) == _bits(g["warped_layout"])).all()
    assert (arg.cpu().numpy() == g["argmax"]).all()
    # sampling indices against the strict-fp32 C restatement
    _, x0y0, _ = CO.sample_coords(g["grid"], g["padding"])
    inr = (np.abs(x0y0) < 2 ** 20).all(-1)
    assert (dbg.cpu().numpy()[inr] == x0y0[inr]).all()
    # grid mode consumes the same fp32 grid tensor and must agree bit for bit as well
    o2, l2, a2 = vlg_b200.warp(_cl(g["src_rgb"]), _cl(g["src_layout"]), torch.as_tensor(g["grid"]).to(DEV),
                               padding_mode=g["padding"], coords_are_grid=True)
    assert torch.equal(o2, out_rgb) and torch.equal(l2, out_lay) and torch.equal(a2, arg)


# ------------------------------------------------------------------ goldens: fused loss + grads
@pytest.mark.parametrize("name", golden_names())
def test_warp_loss_fwd_bwd_vs_golden(name):
    g = load_golden(name)
    a = _cl(g["src_rgb"]).requires_grad_(True)
    b = _cl(g["src_layout"]).requires_grad_(True)
    f = torch.as_tensor(g["flow"]).to(DEV).requires_grad_(True)
    total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(g["tgt_rgb"]), torch.as_tensor(g["tgt_label"]).to(DEV),
                                         _cfg(g, want_argmax=True))
    total.backward()
    vec = vec.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(vec[:5], g["terms"], rtol=RTOL, atol=1e-7)
    np.testing.assert_allclose(vec[_cabi.LOSS_TOTAL], g["total"], rtol=RTOL)
    assert (arg.cpu().numpy() == g["argmax"]).all()
    _assert_close_norm(_nchw(f.grad), g["d_flow"], RTOL, "d_flow")
    _assert_close_norm(_nchw(a.grad), g["d_src_rgb"], RTOL, "d_src_rgb")
    _assert_close_norm(_nchw(b.grad), g["d_src_layout"], RTOL, "d_src_layout")


def test_flow_grad_only_matches_full(golden):
    g = golden
    f = torch.as_tensor(g["flow"]).to(DEV).requires_grad_(True)
    total, vec, _ = vlg_b200.warp_loss(_cl(g["src_rgb"]), _cl(g["src_layout"]), f, _cl(g["tgt_rgb"]),
                                       torch.as_tensor(g["tgt_label"]).to(DEV), _cfg(g))
    total.backward()
    _assert_close_norm(_nchw(f.grad), g["d_flow"], RTOL, "d_flow")
    # validation mode: no gradient requested at all
    with torch.no_grad():
        t2, v2, _ = vlg_b200.warp_loss(_cl(g["src_rgb"]), _cl(g["src_layout"]), f.detach(), _cl(g["tgt_rgb"]),
                                       torch.as_tensor(g["tgt_label"]).to(DEV), _cfg(g))
    assert torch.equal(v2[:6], vec[:6])


# ------------------------------------------------------------------ reference call sites (no warp)
@pytest.mark.parametrize("name", golden_names())
def test_reference_criteria_modules(name):
    g = load_golden(name)
    img = _cl(g["warped_rgb"]).requires_grad_(True)
    seg = _cl(g["warped_layout"]).requires_grad_(True)
    frame3 = _cl(g["tgt_rgb"])
    seg3 = torch.as_tensor(g["tgt_label"]).to(DEV)
    # same three lines as src/trainer.py:248-250
    loss_G_L1 = vlg_b200.L1Loss()(img, frame3) * 40
    style_loss = vlg_b200.CombinedLoss()(output=img, target=frame3) * 20
    seg_loss = vlg_b200.CrossEntropyLoss()(input=seg, target=seg3) * 10
    loss_G = loss_G_L1 + style_loss + seg_loss
    loss_G.backward()
    t = g["terms"]
    np.testing.assert_allclose(loss_G_L1.item(), 40 * t[0], rtol=RTOL)
    np.testing.assert_allclose(style_loss.item(), 20 * (t[1] + t[2]), rtol=RTOL)
    np.testing.assert_allclose(seg_loss.item(), 10 * t[3], rtol=RTOL)
    # gradients against torch autograd on the oracle composition
    a = torch.as_tensor(g["warped_rgb"]).clone().requires_grad_(True)
    z = torch.as_tensor(g["warped_layout"]).clone().requires_grad_(True)
    ref = (40 * TO.l1_loss(a, torch.as_tensor(g["tgt_rgb"]))
           + 20 * (TO.gradient_loss(a, torch.as_tensor(g["tgt_rgb"])) + TO.ssim_loss(a, torch.as_tensor(g["tgt_rgb"])))
           + 10 * TO.cross_entropy(z, torch.as_tensor(g["tgt_label"])))
    ref.backward()
    _assert_close_norm(_nchw(img.grad), a.grad.numpy(), RTOL, "d_img")
    _assert_close_norm(_nchw(seg.grad), z.grad.numpy(), RTOL, "d_seg")
    # the fused single-launch composition agrees with the three separate criteria
    img2 = _cl(g["warped_rgb"]).requires_grad_(True)
    seg2 = _cl(g["warped_layout"]).requires_grad_(True)
    fused = vlg_b200.PixelLosses()(img2, frame3, seg2, seg3)
    fused.backward()
    np.testing.assert_allclose(fused.item(), loss_G.item(), rtol=RTOL)
    _assert_close_norm(_nchw(img2.grad), _nchw(img.grad), RTOL, "fused d_img")
    _assert_close_norm(_nchw(seg2.grad), _nchw(seg.grad), RTOL, "fused d_seg")
    # single criteria
    for mod, fn in ((vlg_b200.GradientLoss(), TO.gradient_loss), (vlg_b200.SsimLoss(), TO.ssim_loss)):
        got = mod(_cl(g["warped_rgb"]), frame3).item()
        np.testing.assert_allclose(got, fn(torch.as_tensor(g["warped_rgb"]), torch.as_tensor(g["tgt_rgb"])).item(), rtol=RTOL)


def test_nchw_contiguous_inputs_are_accepted(golden):
    """Plain NCHW-contiguous tensors (the reference's layout) get one permute-copy and the same result."""
    g = golden
    f = torch.as_tensor(g["flow"]).to(DEV)
    lab = torch.as_tensor(g["tgt_label"]).to(DEV)
    t1, v1, _ = vlg_b200.warp_loss(_cl(g["src_rgb"]), _cl(g["src_layout"]), f, _cl(g["tgt_rgb"]), lab, _cfg(g))
    nchw = lambda k: torch.as_tensor(g[k]).to(DEV).contiguous()
    t2, v2, _ = vlg_b200.warp_loss(nchw("src_rgb"), nchw("src_layout"), f, nchw("tgt_rgb"), lab, _cfg(g))
    assert torch.equal(v1, v2)


# ------------------------------------------------------------------ seeded cases vs the oracle
def _make_case(N, H, W, K, sigma, seed, layout="onehot", far_frac=0.0, device=DEV):
    g = torch.Generator(device="cpu").manual_seed(seed)
    mean = torch.tensor([0.485, 0.456, 0.406])[None, :, None, None]
    std = torch.tensor([0.229, 0.224, 0.225])[None, :, None, None]
    src_rgb = (torch.rand(N, 3, H, W, generator=g) - mean) / std
    tgt_rgb = (torch.rand(N, 3, H, W, generator=g) - mean) / std
    blk = 32
    def labels():
        l = torch.randint(0, K, (N, (H + blk - 1) // blk, (W + blk - 1) // blk), generator=g)
        return l.repeat_interleave(blk, 1).repeat_interleave(blk, 2)[:, :H, :W].contiguous()
    lab_src, lab_tgt = labels(), labels()
    src_layout = TO.one_hot_layout(lab_src, K).contiguous() if layout == "onehot" else torch.randn(N, K, H, W, generator=g)
    flow = torch.randn(N, 2, H, W, generator=g) * sigma
    flow = torch.nn.functional.avg_pool2d(torch.nn.functional.pad(flow, (4, 4, 4, 4), mode="replicate"), 9, 1)
    if far_frac > 0:
        m = torch.rand(N, 1, H, W, generator=g) < far_frac
        far = (torch.rand(N, 2, H, W, generator=g) - 0.5) * 2 * max(H, W)
        flow = torch.where(m, far, flow)
    flow = flow.permute(0, 2, 3, 1).contiguous()
    return dict(src_rgb=src_rgb, src_layout=src_layout, flow=flow, tgt_rgb=tgt_rgb, tgt_label=lab_tgt)


def _squeeze_flow(H, W):
    """Compressive near flow: inside every 8-pixel tooth x -> 0.3 x (|displacement| < 3 px), so that source cells
    receive three to four output pixels each (twelve and more contributions per source pixel in pass 2's gather)."""
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    return torch.stack((-0.7 * ((xx % 8) - 3.5), -0.6 * ((yy % 8) - 3.5)), -1)[None]


CASES = [
    # N, H, W, K, sigma, layout, far_frac, w_tv, padding
    (2, 128, 256, 20, 4.0, "onehot", 0.0, 0.5, "border"),      # BASELINE config 1
    (1, 375, 1242, 20, 48.0, "soft", 0.05, 0.1, "border"),     # KITTI-shaped, large displacement + outliers
    (2, 67, 129, 20, 12.0, "soft", 0.0, 1.0, "zeros"),         # ragged tiles, zeros padding
    (1, 33, 35, 5, 2.0, "soft", 0.0, 0.0, "border"),           # small K
    (1, 41, 70, 19, 3.0, "soft", 0.02, 0.3, "border"),         # 19 train ids, odd K (scalar channel path)
    (1, 41, 70, 30, 3.0, "onehot", 0.02, 0.3, "zeros"),        # 29+1 classes of src/models/simple.py
]


@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}x{c[1]}x{c[2]}k{c[3]}s{c[4]}{c[8]}" for c in CASES])
def test_seeded_case_vs_oracle(case):
    N, H, W, K, sigma, layout, far, w_tv, padding = case
    d = _make_case(N, H, W, K, sigma, seed=1024, layout=layout, far_frac=far)
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"],
                               w_tv=w_tv, padding_mode=padding)
    a = _cl(d["src_rgb"]).requires_grad_(True)
    b = _cl(d["src_layout"]).requires_grad_(True)
    f = d["flow"].to(DEV).requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(w_tv=w_tv, padding_mode=padding, want_argmax=True)
    total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV), cfg)
    total.backward()
    # forward pieces bit-exact through the forward-only entry point
    o_rgb, o_lay, o_arg = vlg_b200.warp(a.detach(), b.detach(), f.detach(), padding_mode=padding)
    assert (_bits(_nchw(o_rgb)) == _bits(ref["warped_rgb"].detach().numpy())).all()
    assert (_bits(_nchw(o_lay)) == _bits(ref["warped_layout"].detach().numpy())).all()
    assert torch.equal(o_arg.cpu(), ref["argmax"]) and torch.equal(arg.cpu(), ref["argmax"])
    got = vec.cpu().numpy().astype(np.float64)
    want = np.array([ref["terms"][k].item() for k in TERMS])
    np.testing.assert_allclose(got[:5], want, rtol=RTOL, atol=1e-7)
    np.testing.assert_allclose(got[_cabi.LOSS_TOTAL], ref["total"].item(), rtol=RTOL)
    ref64 = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"],
                                 w_tv=w_tv, padding_mode=padding, dtype=torch.float64)
    _assert_close_norm(_nchw(f.grad), ref["d_flow"].numpy(), RTOL, "d_flow")
    _assert_close_either(_nchw(a.grad), ref["d_src_rgb"].numpy(), ref64["d_src_rgb"].numpy(), RTOL, "d_src_rgb")
    _assert_close_either(_nchw(b.grad), ref["d_src_layout"].numpy(), ref64["d_src_layout"].numpy(), RTOL, "d_src_layout")
    # C restatement as second witness of the loss terms
    np.testing.assert_allclose(got[0], CO.l1(_nchw(o_rgb), d["tgt_rgb"].numpy()), rtol=RTOL)
    np.testing.assert_allclose(got[2], CO.ssim(_nchw(o_rgb), d["tgt_rgb"].numpy()), rtol=RTOL)


def test_gradients_are_deterministic_and_far_path_runs():
    """Bitwise-identical gradients over repeated runs, with and without far (fixed-point) pixels."""
    for far in (0.0, 0.05, "squeeze"):
        d = _make_case(2, 96, 160, 20, 2.0, seed=7, layout="soft", far_frac=0.0 if far == "squeeze" else far)
        if far == "squeeze":   # source cells with three to four contributors
            d["flow"] = d["flow"] * 0.1 + _squeeze_flow(96, 160)
        outs = []
        for _ in range(5):
            a = _cl(d["src_rgb"]).requires_grad_(True)
            b = _cl(d["src_layout"]).requires_grad_(True)
            f = d["flow"].to(DEV).requires_grad_(True)
            total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV),
                                               vlg_b200.WarpLossConfig(w_tv=0.3))
            total.backward()
            outs.append((vec.clone(), a.grad.clone(), b.grad.clone(), f.grad.clone()))
        for o in outs[1:]:
            for x, y in zip(o, outs[0]):
                assert torch.equal(x, y)
        md = outs[0][0][_cabi.LOSS_MAXDISP].item()
        assert (md >= _cabi.NEAR_RADIUS) == (far == 0.05)


@pytest.mark.parametrize("padding", ["border", "zeros"])
def test_compressive_flow_source_gradient_vs_oracle(padding):
    """Flow that maps three to four output pixels into one source cell (every candidate row of pass 2's scan then
    holds several hits of the same source pixel).  Source gradients against the oracle at the parity bar, on a ragged
    shape."""
    H, W = 61, 150
    d = _make_case(2, H, W, 20, 0.3, seed=31, layout="soft")
    d["flow"] = d["flow"] + _squeeze_flow(H, W)
    kw = dict(w_tv=0.2, padding_mode=padding)
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"], **kw)
    ref64 = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"], dtype=torch.float64, **kw)
    a = _cl(d["src_rgb"]).requires_grad_(True)
    b = _cl(d["src_layout"]).requires_grad_(True)
    f = d["flow"].to(DEV).requires_grad_(True)
    total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV), vlg_b200.WarpLossConfig(**kw))
    total.backward()
    assert vec[_cabi.LOSS_MAXDISP].item() < _cabi.NEAR_RADIUS      # everything travels through the near path
    np.testing.assert_allclose(vec[_cabi.LOSS_TOTAL].item(), ref["total"].item(), rtol=RTOL)
    _assert_close_norm(_nchw(f.grad), ref["d_flow"].numpy(), RTOL, "d_flow")
    _assert_close_either(_nchw(a.grad), ref["d_src_rgb"].numpy(), ref64["d_src_rgb"].numpy(), RTOL, "d_src_rgb")
    _assert_close_either(_nchw(b.grad), ref["d_src_layout"].numpy(), ref64["d_src_layout"].numpy(), RTOL, "d_src_layout")


@pytest.mark.parametrize("packed", [True, False])
@pytest.mark.parametrize("padding", ["border", "zeros"])
def test_far_path_many_pixels_into_one_source_tile(padding, packed):
    """The far path packs two 32-bit lanes into one 64-bit atomic in every source-tile row that receives at most 512 far
    pixels and keeps one 64-bit accumulator per channel elsewhere (vlg_pass2.cuh).  Here every pixel of a 64x96 image
    samples around the same few source pixels (6 000 far pixels into two tile rows: those rows run wide, the rest of
    the image packed or empty) -- against the oracle at the parity bar (fp64 tie-breaker: thousands of contributions
    meet in a handful of source pixels), bitwise reproducible, with and without VLG_FLAG_FAR_WIDE."""
    N, H, W, K = 2, 64, 96, 20
    d = _make_case(N, H, W, K, 0.3, seed=41, layout="soft")
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    tgt_x, tgt_y = 70.3, 11.6                                    # everybody looks at (70.3, 11.6) +- 1.5 px
    d["flow"] = d["flow"] * 3.0 + torch.stack((tgt_x - xx, tgt_y - yy), -1)[None]
    kw = dict(w_tv=0.2, padding_mode=padding)
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"], **kw)
    ref64 = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"], dtype=torch.float64, **kw)
    outs = []
    for _ in range(2):
        a = _cl(d["src_rgb"]).requires_grad_(True)
        b = _cl(d["src_layout"]).requires_grad_(True)
        f = d["flow"].to(DEV).requires_grad_(True)
        total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV),
                                           vlg_b200.WarpLossConfig(far_packed=packed, **kw))
        total.backward()
        outs.append((a.grad.clone(), b.grad.clone(), f.grad.clone()))
    assert vec[_cabi.LOSS_MAXDISP].item() >= _cabi.NEAR_RADIUS
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    _assert_close_norm(_nchw(outs[0][2]), ref["d_flow"].numpy(), RTOL, "d_flow")
    _assert_close_either(_nchw(outs[0][0]), ref["d_src_rgb"].numpy(), ref64["d_src_rgb"].numpy(), RTOL, "d_src_rgb")
    _assert_close_either(_nchw(outs[0][1]), ref["d_src_layout"].numpy(), ref64["d_src_layout"].numpy(), RTOL, "d_src_layout")


@pytest.mark.parametrize("padding", ["border", "zeros"])
@pytest.mark.parametrize("sigma", [48.0, 150.0])
def test_far_path_packed_lanes_agree_with_wide_accumulators(padding, sigma):
    """Rough flow (most pixels far, a few per source-tile row): the packed 32-bit lanes round every contribution at
    2^-(30-h) of its group's largest gradient (h = bits of the row's far-pixel count), the wide mode at ~2^-40.
    Their results agree to 1e-6 of the largest gradient (a tenth of the parity bar) for the rgb AND the layout
    group, whose gradients differ by orders of magnitude (separate scales); ragged shape, both paddings."""
    N, H, W, K = 2, 61, 131, 20
    d = _make_case(N, H, W, K, sigma, seed=43, layout="soft", far_frac=0.05)
    kw = dict(w_tv=0.7, padding_mode=padding)
    res = {}
    for packed in (True, False):
        a = _cl(d["src_rgb"]).requires_grad_(True)
        b = _cl(d["src_layout"]).requires_grad_(True)
        f = d["flow"].to(DEV).requires_grad_(True)
        total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV),
                                           vlg_b200.WarpLossConfig(far_packed=packed, **kw))
        total.backward()
        res[packed] = (a.grad.clone(), b.grad.clone(), f.grad.clone(), vec.clone())
    assert res[True][3][_cabi.LOSS_MAXDISP].item() >= _cabi.NEAR_RADIUS
    assert torch.equal(res[True][2], res[False][2]) and torch.equal(res[True][3], res[False][3])
    for i, name in ((0, "d_src_rgb"), (1, "d_src_layout")):
        mx = res[False][i].abs().max().item()
        err = (res[True][i] - res[False][i]).abs().max().item()
        assert err <= 1e-6 * mx, f"{name}: packed vs wide {err / mx:.2e}"


def test_upstream_gradient_scaling():
    d = _make_case(1, 40, 72, 20, 2.0, seed=3)
    grads = []
    for scale in (1.0, 0.125):
        a = _cl(d["src_rgb"]).requires_grad_(True)
        b = _cl(d["src_layout"]).requires_grad_(True)
        f = d["flow"].to(DEV).requires_grad_(True)
        total, _, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV))
        (total * scale).backward()
        grads.append((a.grad.clone(), b.grad.clone(), f.grad.clone()))     # one vlg_scale_grads_multi launch for the three
    for g1, g2 in zip(*grads):
        assert torch.equal(g1 * 0.125, g2)   # power-of-two scale is exact


def test_ignore_index_and_bad_label_status():
    d = _make_case(1, 32, 64, 20, 1.0, seed=5, layout="soft")
    lab = d["tgt_label"].clone()
    lab[0, :8] = -100
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], lab)
    b = _cl(d["src_layout"]).requires_grad_(True)
    total, vec, _ = vlg_b200.warp_loss(_cl(d["src_rgb"]), b, d["flow"].to(DEV), _cl(d["tgt_rgb"]), lab.to(DEV))
    total.backward()
    np.testing.assert_allclose(vec[_cabi.LOSS_CE].item(), ref["terms"]["ce"].item(), rtol=RTOL)
    assert vec[_cabi.LOSS_NVALID].item() == (lab != -100).sum().item()
    _assert_close_norm(_nchw(b.grad), ref["d_src_layout"].numpy(), RTOL, "d_src_layout")


def test_assume_near_matches_default_path():
    d = _make_case(2, 64, 96, 20, 3.0, seed=11)
    res = []
    for near in (False, True):
        b = _cl(d["src_layout"]).requires_grad_(True)
        total, vec, _ = vlg_b200.warp_loss(_cl(d["src_rgb"]), b, d["flow"].to(DEV), _cl(d["tgt_rgb"]),
                                           d["tgt_label"].to(DEV), vlg_b200.WarpLossConfig(assume_near=near))
        total.backward()
        res.append((vec.clone(), b.grad.clone()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


# ------------------------------------------------------------------ full-size properties (BASELINE config 2)
def test_full_size_properties_config2():
    """16x256x512, K=20 (BASELINE.json configs[1]) against the oracle evaluated by torch CUDA on the same
    GPU in fp32 AND fp64: warp / argmax bit-exact, losses and all three gradients at 1e-5 (normwise-max and
    RMS-relative), plus size-independent properties."""
    N, H, W, K = 16, 256, 512, 20
    d = _make_case(N, H, W, K, 4.0, seed=1024)
    a = _cl(d["src_rgb"]).requires_grad_(True)
    b = _cl(d["src_layout"]).requires_grad_(True)
    f = d["flow"].to(DEV).requires_grad_(True)
    tgt, lab = _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV)
    total, vec, arg = vlg_b200.warp_loss(a, b, f, tgt, lab, vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True))
    total.backward()
    ref = _gpu_oracle(d, torch.float32)
    ref64 = _gpu_oracle(d, torch.float64)
    assert_terms_parity(vec.cpu().numpy()[:5], _terms(ref), _terms(ref64), RTOL)
    o_rgb, o_lay, o_arg = vlg_b200.warp(a.detach(), b.detach(), f.detach())
    assert torch.equal(o_arg, ref["argmax"]) and torch.equal(arg, ref["argmax"])
    assert torch.equal(o_lay.contiguous(), ref["warped_layout"].detach().contiguous())   # bit-exact vs torch CUDA
    assert torch.equal(o_rgb.contiguous(), ref["warped_rgb"].detach().contiguous())
    assert_grad_parity(f.grad, ref["d_flow"], ref64["d_flow"], RTOL, "d_flow")
    assert_grad_parity(a.grad, ref["d_src_rgb"], ref64["d_src_rgb"], RTOL, "d_src_rgb")
    assert_grad_parity(b.grad, ref["d_src_layout"], ref64["d_src_layout"], RTOL, "d_src_layout")
    # properties: one-hot sources warp to a partition of unity; gradient mass is conserved by the
    # transpose (sum of d_src == sum of weights * d_out == d/d(eps) of loss under src += eps)
    s = o_lay.float().sum(1)
    assert (s - 1).abs().max().item() < 1e-5
    assert arg.min().item() >= 0 and arg.max().item() < K


def test_linearity_of_source_gradient_transpose():
    """<warp(src), g> == <src, warp^T(g)> : the deterministic pass 2 is the exact adjoint of the
    forward gather (checked through CE-free L1-only losses with random targets)."""
    d = _make_case(1, 48, 80, 20, 5.0, seed=21, layout="soft")
    f = d["flow"].to(DEV)
    b = _cl(d["src_layout"]).requires_grad_(True)
    a = _cl(d["src_rgb"]).requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(w_l1=1.0, w_gd=0.0, w_ssim=0.0, w_ce=0.0, term_mask=_cabi.TERM_L1 | _cabi.TERM_CE)
    total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV), cfg)
    total.backward()
    # L1 gradient wrt warped = sign(a-b)/numel ; so <d_src, src> must equal <sign/numel, warp(src)>
    o_rgb, _, _ = vlg_b200.warp(a.detach(), None, f)
    gout = torch.sign(o_rgb.float() - _cl(d["tgt_rgb"])) / o_rgb.numel()
    lhs = (a.grad.double() * a.detach().double()).sum().item()
    rhs = (gout.double() * o_rgb.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-5 * abs(rhs)
    assert b.grad.abs().max().item() == 0.0   # w_ce = 0 -> no layout gradient


# ------------------------------------------------------------------ bf16 activations (BASELINE config 3)
def test_bf16_io_rounded_once_vs_oracle():
    """bf16 inputs/outputs, fp32 flow and accumulation, against the oracle evaluated in fp32 and fp64 on the SAME
    bf16-rounded inputs: the loss vector and d_flow (fp32 outputs) at the fp32 bar, d_src_rgb / d_src_layout the fp32
    result rounded once to bf16, the forward warp the fp32 oracle value rounded once, bit for bit."""
    d = _make_case(2, 64, 96, 20, 2.0, seed=9, layout="soft")
    bf = lambda t: t.to(torch.bfloat16)
    src_rgb, src_lay, tgt = bf(d["src_rgb"]), bf(d["src_layout"]), bf(d["tgt_rgb"])
    ref = TO.warp_loss_fwd_bwd(src_rgb.float(), src_lay.float(), d["flow"], tgt.float(), d["tgt_label"], w_tv=0.5)
    ref64 = TO.warp_loss_fwd_bwd(src_rgb.float(), src_lay.float(), d["flow"], tgt.float(), d["tgt_label"], w_tv=0.5,
                                 dtype=torch.float64)
    a = _cl(src_rgb).requires_grad_(True)
    b = _cl(src_lay).requires_grad_(True)
    f = d["flow"].to(DEV).requires_grad_(True)
    total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(tgt), d["tgt_label"].to(DEV),
                                         vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True))
    total.backward()
    assert_terms_parity(vec.cpu().numpy()[:5], _terms(ref), _terms(ref64), RTOL)
    assert_terms_parity([vec[_cabi.LOSS_TOTAL].item()], [ref["total"].item()], [ref64["total"].item()], RTOL)
    assert torch.equal(arg.cpu(), ref["argmax"])
    assert a.grad.dtype == torch.bfloat16 and b.grad.dtype == torch.bfloat16 and f.grad.dtype == torch.float32
    assert_grad_parity(f.grad, ref["d_flow"], ref64["d_flow"], RTOL, "d_flow")
    assert_bf16_rounded_once(a.grad.cpu(), ref["d_src_rgb"], ref64["d_src_rgb"], "d_src_rgb")
    assert_bf16_rounded_once(b.grad.cpu(), ref["d_src_layout"], ref64["d_src_layout"], "d_src_layout")
    # forward warp in bf16: same taps, values rounded once at the store
    o_rgb, o_lay, o_arg = vlg_b200.warp(a.detach(), b.detach(), f.detach())
    assert o_lay.dtype == torch.bfloat16
    want_lay = ref["warped_layout"].detach().to(torch.bfloat16)
    assert torch.equal(o_lay.cpu().contiguous(), want_lay.contiguous())
    assert torch.equal(o_rgb.cpu().contiguous(), ref["warped_rgb"].detach().to(torch.bfloat16).contiguous())


def test_full_res_forward_config3_properties():
    """8x1024x2048 is too large for the CPU oracle; check the forward-only path against torch CUDA
    grid_sample on one full-resolution image (src/val.py:172-176 shape) in fp32, bit for bit."""
    N, H, W, K = 1, 1024, 2048, 20
    d = _make_case(N, H, W, K, 4.0, seed=31)
    a, b, f = _cl(d["src_rgb"]), _cl(d["src_layout"]), d["flow"].to(DEV)
    o_rgb, o_lay, o_arg = vlg_b200.warp(a, b, f)
    grid = TO.flow_to_grid(f)
    r_lay = TO.warp(d["src_layout"].to(DEV), grid)
    assert torch.equal(o_lay.contiguous(), r_lay.contiguous())
    assert torch.equal(o_arg, torch.argmax(r_lay, 1))
    assert tuple(o_arg.shape) == (N, 1024, 2048)


# ------------------------------------------------------------------ rollout with label sources (SURVEY 8f-2)
@pytest.mark.parametrize("padding", ["border", "zeros"])
def test_label_source_warp_matches_dense_one_hot(padding):
    """warp_labels(label) == argmax(warp(one_hot(label))) bit for bit, including half-pixel ties."""
    K = 20
    for seed, sigma, half in ((3, 2.0, False), (4, 3.0, True), (5, 30.0, False)):
        d = _make_case(2, 61, 93, K, sigma, seed=seed)
        flow = d["flow"]
        if half:
            flow = torch.round(flow * 2) / 2          # exact ties between classes
        lab = d["src_layout"].argmax(1)
        f = flow.to(DEV)
        o_rgb, _, o_arg = vlg_b200.warp(_cl(d["src_rgb"]), _cl(d["src_layout"]), f, padding_mode=padding)
        l_rgb, l_lab = vlg_b200.warp_labels(_cl(d["src_rgb"]), lab.to(DEV), f, padding_mode=padding)
        assert torch.equal(l_lab, o_arg)
        assert torch.equal(l_rgb, o_rgb)
        ref = TO.warp(d["src_layout"], TO.flow_to_grid(flow), padding)
        assert torch.equal(l_lab.cpu(), TO.argmax_layout(ref))


def test_rollout_five_steps_matches_dense_feedback():
    """5-step autoregressive rollout (BASELINE config 4 shape, reduced): label feedback equals the
    dense argmax -> one-hot -> warp loop of src/trainer.py:460-469 at every step."""
    K, steps = 20, 5
    d = _make_case(2, 64, 128, K, 3.0, seed=17)
    flows = [(_make_case(2, 64, 128, K, 3.0, seed=100 + t)["flow"]).to(DEV) for t in range(steps)]
    img0, lab0 = _cl(d["src_rgb"]), d["src_layout"].argmax(1).to(DEV)
    imgs, labs = vlg_b200.rollout(img0, lab0, lambda t, i, l: flows[t], steps=steps)
    img, lay = img0, _cl(d["src_layout"])
    for t in range(steps):
        img, _, arg = vlg_b200.warp(img, lay, flows[t])
        lay = torch.zeros_like(lay).scatter_(1, arg[:, None], 1.0)     # argmax -> one-hot feedback
        assert torch.equal(labs[t], arg), t
        assert torch.equal(imgs[t], img), t


def test_rollout_config4_real_shape_matches_dense_feedback():
    """BASELINE.json configs[3] at the per-GPU shape of the dp8 run (32x512x1024 over 8 GPUs = 4x512x1024 per rank),
    5 autoregressive steps: label feedback equals the dense argmax -> one-hot -> warp loop of
    src/trainer.py:460-469 at every step, frames and label maps bit for bit."""
    K, steps, N, H, W = 20, 5, 4, 512, 1024
    d = _make_case(N, H, W, K, 4.0, seed=41)
    flows = [(_make_case(N, H, W, K, 4.0, seed=200 + t)["flow"]).to(DEV) for t in range(steps)]
    img0, lab0 = _cl(d["src_rgb"]), d["src_layout"].argmax(1).to(DEV)
    imgs, labs = vlg_b200.rollout(img0, lab0, lambda t, i, l: flows[t], steps=steps)
    img, lay = img0, _cl(d["src_layout"])
    for t in range(steps):
        img, _, arg = vlg_b200.warp(img, lay, flows[t])
        # the dense loop of the reference, evaluated by torch CUDA on the same inputs
        r_lay = TO.warp(lay.contiguous(), TO.flow_to_grid(flows[t]))
        assert torch.equal(torch.argmax(r_lay, 1), arg), t
        lay = torch.zeros_like(lay).scatter_(1, arg[:, None], 1.0)     # argmax -> one-hot feedback
        assert torch.equal(labs[t], arg), t
        assert torch.equal(imgs[t], img), t
    assert len(labs) == steps and tuple(labs[-1].shape) == (N, H, W)


def test_colorize_matches_vis_seg_mask():
    """src/trainer.py:416-427: rgb = color_map[argmax(seg)] / 255, as NCHW float."""
    K = 20
    g = torch.Generator().manual_seed(5)
    seg = torch.randn(2, K, 33, 47, generator=g)
    seg[0, 3, 0, 0] = seg[0, 7, 0, 0] = 9.0            # tie -> first index
    pal = torch.tensor(vlg_b200.CITYSCAPES_PALETTE)
    want = pal[torch.argmax(seg, 1)].permute(0, 3, 1, 2).contiguous().float() / 255
    got = vlg_b200.colorize(_cl(seg), K, argmax=True)
    assert torch.equal(got.cpu().contiguous(), want)
    ids = torch.argmax(seg, 1)
    got2 = vlg_b200.colorize(ids.to(DEV), K)
    assert torch.equal(got2.cpu().contiguous(), want)


# ------------------------------------------------------------------ loss variants (SURVEY 8f-4)
def test_class_weighted_cross_entropy_variants():
    """nn.CrossEntropyLoss(weight=w) (weighted mean) and the reference's class-weighted variant
    F.cross_entropy(weight=w, reduction='sum') / n_known (src/models/simple.py:56-59), with ignored
    labels; loss, gradient and bitwise run-to-run reproducibility of the weighted divisor."""
    K = 20
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(2, K, 45, 67, generator=g)
    label = torch.randint(0, K, (2, 45, 67), generator=g)
    label[0, :5] = -100
    w = torch.rand(K, generator=g) + 0.25
    for reduction in ("mean", "sum_over_known"):
        z = logits.clone().requires_grad_(True)
        if reduction == "mean":
            ref = torch.nn.functional.cross_entropy(z, label, weight=w, reduction="mean")
        else:
            ref = torch.nn.functional.cross_entropy(z, label, weight=w, reduction="sum") / (label != -100).sum()
        ref.backward()
        outs = []
        for _ in range(3):
            zz = _cl(logits).requires_grad_(True)
            crit = vlg_b200.CrossEntropyLoss(weight=w, reduction=reduction).to(DEV)
            loss = crit(input=zz, target=label.to(DEV))
            loss.backward()
            outs.append((loss.detach().clone(), zz.grad.clone()))
        np.testing.assert_allclose(outs[0][0].item(), ref.item(), rtol=RTOL)
        _assert_close_norm(_nchw(outs[0][1]), z.grad.numpy(), RTOL, "d_logits " + reduction)
        for o in outs[1:]:
            assert torch.equal(o[0], outs[0][0]) and torch.equal(o[1], outs[0][1])
    # the fused warp op takes the same weights
    d = _make_case(1, 40, 64, K, 1.5, seed=2, layout="soft")
    b = _cl(d["src_layout"]).requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(class_weight=w.to(DEV))
    total, vec, _ = vlg_b200.warp_loss(_cl(d["src_rgb"]), b, d["flow"].to(DEV), _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV), cfg)
    total.backward()
    rb = d["src_layout"].clone().requires_grad_(True)
    wl = TO.warp(rb, TO.flow_to_grid(d["flow"]))
    ce = torch.nn.functional.cross_entropy(wl, d["tgt_label"], weight=w)
    np.testing.assert_allclose(vec[_cabi.LOSS_CE].item(), ce.item(), rtol=RTOL)


def test_kernel_organisations_agree():
    """The layout terms of a warped step run in two organisations of the same arithmetic: the persistent
    double-buffered tile kernel (lay_tile_kernel: TMA-staged windows, read-once taps, online softmax) and the
    first tile kernel (pass1_kernel: cp.async staging; here selected by use_tma=False).  Argmax layouts are
    bit-identical (same FMA chain); losses and gradients, whose sums are associated differently, agree well
    inside the parity bar."""
    variants = (dict(), dict(use_tma=False))
    for sigma, padding, shape in ((0.6, "border", (2, 77, 141)), (5.0, "zeros", (2, 77, 141)), (2.0, "border", (1, 19, 33)),
                                  (9.0, "border", (3, 64, 200))):
        d = _make_case(*shape, 20, sigma, seed=17, layout="soft")
        res = []
        for kw in variants:
            a = _cl(d["src_rgb"]).requires_grad_(True)
            b = _cl(d["src_layout"]).requires_grad_(True)
            f = d["flow"].to(DEV).requires_grad_(True)
            cfg = vlg_b200.WarpLossConfig(w_tv=0.4, padding_mode=padding, want_argmax=True, **kw)
            total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV), cfg)
            total.backward()
            res.append((vec.clone(), arg.clone(), a.grad.clone(), b.grad.clone(), f.grad.clone()))
        v1, arg1, ga1, gb1, gf1 = res[-1]
        for (v0, arg0, ga0, gb0, gf0), kw in zip(res[:-1], variants):
            assert torch.equal(arg0, arg1), kw
            np.testing.assert_allclose(v0[:6].cpu().numpy(), v1[:6].cpu().numpy(), rtol=2e-6)
            for name, x, y in (("d_src_rgb", ga0, ga1), ("d_src_layout", gb0, gb1), ("d_flow", gf0, gf1)):
                err = (x - y).abs().max().item()
                assert err <= 1e-5 * y.abs().max().item(), (kw, name, err)   # the parity bar; typical 3e-6


def test_pass2_from_records_matches_pass2_from_coords_bitwise():
    """Pass 2 exists twice: pass2_rec_kernel gathers from the tap records pass 1 wrote (TMA-staged windows of
    d_out, cell codes and fractional weights), pass2_kernel re-derives them from the coordinates.  Same
    candidate order, same weights: d_src_rgb / d_src_layout must be bit-identical -- for odd widths (pitched
    rows), both paddings, far pixels (fixed-point path), compressive flow (three to four hits per source cell),
    bf16 and both pass-1 organisations (lay_tile_kernel writes the records itself; pass1_kernel, which takes
    bf16 K = 20 rows of odd width, goes through tap_records_kernel)."""
    cases = ((0.6, "border", (2, 77, 141)), (5.0, "zeros", (2, 77, 141)), (2.0, "border", (1, 19, 33)),
             (30.0, "border", (2, 64, 200)), (2.5, "zeros", (1, 40, 251)), (2.5, "border", (1, 40, 251)),
             (1.5, "border", (2, 375 // 5, 1242 // 6)), ("squeeze", "border", (2, 64, 160)), ("squeeze", "zeros", (1, 33, 97)))
    for sigma, padding, shape in cases:
        if sigma == "squeeze":   # sawtooth x -> 0.3 x per 8-pixel tooth: three to four output pixels per source cell, all near
            d = _make_case(*shape, 20, 0.3, seed=23, layout="soft")
            d["flow"] = d["flow"] * 0.2 + _squeeze_flow(shape[1], shape[2])
        else:
            d = _make_case(*shape, 20, sigma, seed=23, layout="soft")
        for dt in (torch.float32, torch.bfloat16):
            res = []
            for rec in (True, False):
                a = _cl(d["src_rgb"].to(dt)).requires_grad_(True)
                b = _cl(d["src_layout"].to(dt)).requires_grad_(True)
                f = d["flow"].to(DEV).requires_grad_(True)
                cfg = vlg_b200.WarpLossConfig(w_tv=0.4, padding_mode=padding, pass2_records=rec)
                total, vec, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"].to(dt)), d["tgt_label"].to(DEV), cfg)
                total.backward()
                res.append((vec.clone(), a.grad.clone(), b.grad.clone(), f.grad.clone()))
            for x, y in zip(*res):
                assert torch.equal(x, y), (sigma, padding, shape, dt)
            assert res[0][2].abs().max().item() > 0


def test_one_hot_layout_matches_reference_encoding():
    """`transform_seg_one_hot` (src/models/net_utils.py:14-24) on the device: int64 and float32 class-id
    maps (the dataset hands float maps, src/folder.py:97-99), fp32 and bf16 layouts, K in {20, 19, 5}."""
    g = torch.Generator().manual_seed(3)
    for K in (20, 19, 5):
        lab = torch.randint(0, K, (2, 37, 53), generator=g)
        want = TO.one_hot_layout(lab, K)
        for dt in (torch.float32, torch.bfloat16):
            for src in (lab, lab.float(), lab.float()[:, None]):
                got = vlg_b200.one_hot_layout(src.to(DEV), K, dt)
                assert got.shape == (2, K, 37, 53) and got.dtype == dt
                assert got.is_contiguous(memory_format=torch.channels_last)
                assert torch.equal(got.float().cpu(), want)
    # the encoded layout is a valid source of the fused op
    d = _make_case(1, 40, 64, 20, 1.0, seed=4, layout="onehot")
    lay = vlg_b200.one_hot_layout(d["src_layout"].argmax(1).to(DEV), 20)
    assert torch.equal(lay.cpu(), d["src_layout"])


def test_prepare_frames_matches_reference_renorm_and_flip():
    """Per-channel renorm `(x - mean) / std` (src/trainer.py:193-195,212,324), its inverse (:215) and the flip
    augmentation (:200-206) fused with the NCHW -> NHWC re-layout: bit-identical to the torch expressions,
    for plain-contiguous and channels_last inputs, vectorised (W % 4 == 0) and scalar widths."""
    g = torch.Generator().manual_seed(5)
    for (N, H, W) in ((2, 16, 32), (1, 13, 37), (3, 8, 1242 // 6)):
        frames = torch.rand(N, 3, H, W, generator=g)
        labels = torch.randint(0, 20, (N, H, W), generator=g)
        for flip in (False, True):
            for denorm in (False, True):
                want, want_lab = TO.renorm_frames(frames, flip=flip, denormalize=denorm, labels=labels)
                for src in (frames.to(DEV), _cl(frames)):
                    got, got_lab = vlg_b200.prepare_frames(src, flip=flip, denormalize=denorm, labels=labels.to(DEV))
                    assert got.is_contiguous(memory_format=torch.channels_last) and got.shape == want.shape
                    assert torch.equal(got.cpu(), want), (N, H, W, flip, denorm)
                    assert torch.equal(got_lab.cpu(), want_lab)
        # generator-output normalisation constants (src/trainer.py:120-121,212) and bf16 output
        want = TO.renorm_frames(frames, vlg_b200.ops.OUT_MEAN, vlg_b200.ops.OUT_STD)
        got = vlg_b200.prepare_frames(frames.to(DEV), vlg_b200.ops.OUT_MEAN, vlg_b200.ops.OUT_STD)
        assert torch.equal(got.cpu(), want)
        got16 = vlg_b200.prepare_frames(frames.to(DEV), dtype=torch.bfloat16)
        assert torch.equal(got16.cpu(), TO.renorm_frames(frames).to(torch.bfloat16))


def test_forward_warp_matches_oracle_bitwise_all_modes():
    """vlg_warp_fwd against the oracle (fp32 evaluation of the same inputs, rounded once at the store): warped
    layout, warped rgb and argmax bit for bit -- both paddings, ragged widths, out-of-image flows, fp32 and
    bf16, K = 20, 19, 30 and 5.  warp_fwd_kernel sends whole 32-pixel runs as bulk copies when a pixel is a multiple
    of 8 bytes and the tail of P % 32 pixels a multiple of 16 (launch_fwd): bulk for fp32 K = 20 (every P), bf16
    K = 20 and fp32 K = 30 (P % 32 even, zero included); scalar stores for an odd P % 32 there, and for K = 19, K = 5 and
    bf16 K = 30 always.  The shapes give P % 32 = 0, odd and even non-zero for each K.  warp_labels on argmax(layout)
    returns the same warped rgb, bit for bit, and argmax(warp(one_hot(labels)))."""
    for (shape, K, sigma, padding) in (((2, 37, 70), 20, 2.0, "border"), ((1, 19, 33), 20, 40.0, "zeros"),
                                       ((2, 64, 200), 20, 9.0, "zeros"), ((1, 24, 1242 // 6), 20, 3.0, "border"),
                                       ((1, 30, 45), 19, 3.0, "zeros"), ((1, 16, 64), 19, 2.0, "border"),
                                       ((1, 19, 33), 19, 9.0, "border"),
                                       ((1, 16, 64), 30, 2.0, "zeros"), ((1, 19, 33), 30, 9.0, "border"),
                                       ((2, 17, 57), 30, 3.0, "zeros"),
                                       ((1, 32, 48), 5, 3.0, "border"), ((1, 21, 35), 5, 40.0, "zeros"),
                                       ((2, 13, 30), 5, 2.0, "zeros")):
        d = _make_case(*shape, K, sigma, seed=41, layout="soft")
        for dt in (torch.float32, torch.bfloat16):
            a, b, f = _cl(d["src_rgb"].to(dt)), _cl(d["src_layout"].to(dt)), d["flow"].to(DEV)
            o_rgb, o_lay, o_arg = vlg_b200.warp(a, b, f, padding_mode=padding)
            grid = TO.flow_to_grid(d["flow"])
            want = TO.warp(d["src_layout"].to(dt).float(), grid, padding_mode=padding).to(dt)
            assert torch.equal(o_lay.cpu().contiguous(), want.contiguous()), (shape, K, padding, dt)
            assert torch.equal(o_arg.cpu(), torch.argmax(want.float(), 1)), (shape, K, padding, dt)
            want_rgb = TO.warp(d["src_rgb"].to(dt).float(), grid, padding_mode=padding).to(dt)
            assert torch.equal(o_rgb.cpu().contiguous(), want_rgb.contiguous()), (shape, K, padding, dt)
            if K == 20:
                lab = d["src_layout"].argmax(1)
                l_rgb, l_lab = vlg_b200.warp_labels(a, lab.to(DEV), f, padding_mode=padding)
                assert l_rgb.dtype == dt and torch.equal(l_rgb, o_rgb), (shape, padding, dt)
                want_lab = torch.argmax(TO.warp(TO.one_hot_layout(lab, K), grid, padding_mode=padding), 1)
                assert torch.equal(l_lab.cpu(), want_lab), (shape, padding, dt)


def test_full_res_bf16_fwd_bwd_config3_vs_gpu_oracle():
    """BASELINE.json configs[2] at its REAL size (8x1024x2048, bf16 I/O, fp32 flow) against the oracle evaluated by
    torch CUDA in fp32 and fp64 on the SAME bf16-rounded inputs: the loss vector and d_flow (fp32 outputs) at the fp32
    bar, d_src_rgb / d_src_layout the fp32 result rounded once to bf16 (bf16_bars); two runs are bitwise identical
    (no float atomics anywhere).  Argmax: the product takes it on the fp32-accumulated warp of the bf16 layouts, the
    oracle on ITS fp32 warp of the same inputs -- identical arithmetic (Appendix A.6), so the maps must be equal
    everywhere, not only where the margin is clear."""
    N, H, W, K = 8, 1024, 2048, 20
    d = _make_case(N, H, W, K, 4.0, seed=33, layout="soft")
    bf = lambda t: t.to(torch.bfloat16)
    src_rgb, src_lay, tgt = bf(d["src_rgb"]), bf(d["src_layout"]), bf(d["tgt_rgb"])
    lab = d["tgt_label"].to(DEV)
    runs = []
    for _ in range(2):
        a = _cl(src_rgb).requires_grad_(True)
        b = _cl(src_lay).requires_grad_(True)
        f = d["flow"].to(DEV).requires_grad_(True)
        total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(tgt), lab, vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True))
        total.backward()
        runs.append((vec.clone(), arg.clone(), a.grad.clone(), b.grad.clone(), f.grad.clone()))
        del a, b, f, total
    for x, y in zip(*runs):
        assert torch.equal(x, y)
    vec, arg, ga, gb, gf = runs[0]
    del runs
    d32 = dict(d, src_rgb=src_rgb.float(), src_layout=src_lay.float(), tgt_rgb=tgt.float())
    ref = _gpu_oracle(d32, torch.float32)
    assert torch.equal(arg, ref["argmax"])
    t32 = _terms(ref)
    g32 = {k: ref[k].detach().clone() for k in ("d_flow", "d_src_rgb", "d_src_layout")}
    del ref
    torch.cuda.empty_cache()
    ref64 = _gpu_oracle(d32, torch.float64)
    assert_terms_parity(vec.cpu().numpy()[:5], t32, _terms(ref64), RTOL)
    assert_grad_parity(gf, g32["d_flow"], ref64["d_flow"], RTOL, "d_flow")
    assert_bf16_rounded_once(ga, g32["d_src_rgb"], ref64["d_src_rgb"], "d_src_rgb")
    assert_bf16_rounded_once(gb, g32["d_src_layout"], ref64["d_src_layout"], "d_src_layout")


@pytest.mark.parametrize("B", [1, 2, 64])
def test_kitti_shape_large_displacement_config5_vs_gpu_oracle(B):
    """BASELINE.json configs[4] (375x1242: ragged tiles, rows that need the pitched workspace arrays; batch sweep
    ends 1 and 64 plus B=2) with large-displacement flow (sigma = 48 px smoothed, 5 % of the pixels uniform over the
    image): most pixels leave the 3-pixel near path.  Against the oracle evaluated by torch CUDA in fp32 and
    fp64: warp and argmax bit-exact, losses and all gradients at 1e-5 (normwise-max and RMS-relative); two runs
    bitwise identical."""
    N, H, W, K = B, 375, 1242, 20
    d = _make_case(N, H, W, K, 48.0, seed=55, layout="soft", far_frac=0.05)
    flow = d["flow"]
    lab = d["tgt_label"].to(DEV)
    runs = []
    for _ in range(2):
        a = _cl(d["src_rgb"]).requires_grad_(True)
        b = _cl(d["src_layout"]).requires_grad_(True)
        f = flow.to(DEV).requires_grad_(True)
        total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), lab, vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True))
        total.backward()
        runs.append((vec.clone(), arg.clone(), a.grad.clone(), b.grad.clone(), f.grad.clone()))
        if len(runs) == 2:
            o_rgb, o_lay, _ = vlg_b200.warp(a.detach(), b.detach(), f.detach())
        del a, b, f, total
    for x, y in zip(*runs):
        assert torch.equal(x, y)
    vec, arg, ga, gb, gf = runs[0]
    del runs
    assert vec[_cabi.LOSS_MAXDISP].item() > 100.0          # the large-displacement machinery really ran

    ref = _gpu_oracle(d, torch.float32)
    assert torch.equal(arg, ref["argmax"])
    assert torch.equal(o_lay.contiguous(), ref["warped_layout"].detach().contiguous())
    assert torch.equal(o_rgb.contiguous(), ref["warped_rgb"].detach().contiguous())
    del o_lay, o_rgb
    t32 = _terms(ref)
    g32 = {k: ref[k].detach().clone() for k in ("d_flow", "d_src_rgb", "d_src_layout")}
    del ref
    torch.cuda.empty_cache()
    ref64 = _gpu_oracle(d, torch.float64)
    assert_terms_parity(vec.cpu().numpy()[:5], t32, _terms(ref64), RTOL)
    # border pixels collect thousands of clamped contributions: torch's own fp32 atomic scatter drifts there
    # (SURVEY Appendix A.10) -- the fp64 evaluation of the same oracle settles those
    assert_grad_parity(gf, g32["d_flow"], ref64["d_flow"], RTOL, "d_flow")
    assert_grad_parity(ga, g32["d_src_rgb"], ref64["d_src_rgb"], RTOL, "d_src_rgb")
    assert_grad_parity(gb, g32["d_src_layout"], ref64["d_src_layout"], RTOL, "d_src_layout")


def test_split_entry_points_equal_the_fused_call():
    """`vlg_warp_loss_pass1` (pass 1 with the fused loss reduction) followed by `vlg_warp_bwd_src` is what a
    data-parallel caller uses to put its loss all-reduce between the passes; it must give exactly the fused
    `vlg_warp_loss_fwd_bwd` result: loss vector and all three gradients bit for bit."""
    import ctypes as C
    from vlg_b200 import ops as vops
    lib = _cabi.load()
    N, H, W, K = 2, 61, 93, 20
    d = _make_case(N, H, W, K, 3.0, seed=77, layout="soft", far_frac=0.01)
    a, b, f = _cl(d["src_rgb"]), _cl(d["src_layout"]), d["flow"].to(DEV)
    t, lab = _cl(d["tgt_rgb"]), d["tgt_label"].to(DEV)
    prob = vops._problem(N, H, W, K, torch.float32, vlg_b200.WarpLossConfig(w_tv=0.5))
    ptr = vops._ptr
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = []
    for split in (False, True):
        ws = vops._workspace(prob, True, a.device)
        loss = torch.zeros(_cabi.LOSS_SLOTS, dtype=torch.float32, device=DEV)
        d_c = torch.empty(N, H, W, 2, dtype=torch.float32, device=DEV)
        d_a = vops.empty_nhwc((N, 3, H, W), torch.float32, a.device)
        d_b = vops.empty_nhwc((N, K, H, W), torch.float32, a.device)
        if split:
            vops.check(lib.vlg_warp_loss_pass1(C.byref(prob), ptr(a), ptr(b), ptr(f), ptr(t), ptr(lab), ptr(loss), ptr(d_c), None, 1,
                                               ptr(ws), ws.numel(), sp))
            vops.check(lib.vlg_warp_bwd_src(C.byref(prob), ptr(f), ptr(d_a), ptr(d_b), ptr(ws), ws.numel(), sp))
        else:
            vops.check(lib.vlg_warp_loss_fwd_bwd(C.byref(prob), ptr(a), ptr(b), ptr(f), ptr(t), ptr(lab), ptr(loss), ptr(d_c), ptr(d_a),
                                                 ptr(d_b), None, ptr(ws), ws.numel(), sp))
        torch.cuda.synchronize()
        res.append((loss.clone(), d_c.clone(), d_a.clone(), d_b.clone()))
    for x, y in zip(*res):
        assert torch.equal(x, y)
    assert res[0][0][_cabi.LOSS_TOTAL].item() > 0 and res[0][3].abs().max().item() > 0


def test_one_thread_alternating_devices_repeats_each_devices_result():
    """The library keeps its launch state (kernel attributes, resident grid sizes, the side stream of the label count)
    per device ordinal.  One thread that alternates the fused op between two GPUs gets, on each, the result of its
    first call there bit for bit: losses, argmax and every gradient."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    d = _make_case(2, 77, 141, 20, 2.0, seed=29, layout="soft", device="cpu")
    cfg = vlg_b200.WarpLossConfig(w_tv=0.4, want_argmax=True)
    first = {}
    for it in range(6):
        dev = torch.device("cuda", it % 2)
        a = torch.as_tensor(d["src_rgb"]).to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        b = torch.as_tensor(d["src_layout"]).to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
        f = torch.as_tensor(d["flow"]).to(dev).requires_grad_(True)
        t = torch.as_tensor(d["tgt_rgb"]).to(dev).contiguous(memory_format=torch.channels_last)
        total, vec, arg = vlg_b200.warp_loss(a, b, f, t, torch.as_tensor(d["tgt_label"]).to(dev), cfg)
        total.backward()
        out = tuple(x.detach().cpu() for x in (vec, arg, a.grad, b.grad, f.grad))
        if dev.index not in first:
            first[dev.index] = out
            continue
        for x, y in zip(first[dev.index], out):
            assert torch.equal(x, y), (it, dev)
