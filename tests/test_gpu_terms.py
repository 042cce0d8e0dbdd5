"""Each loss term on its own, and the un-warped criteria, against the oracle (run on a GPU).

The parity tests elsewhere compare the five-term composite 40*L1 + 20*(GD+SSIM) + 10*CE + w_tv*TV: their bars are
relative to the composite, so a term with a small share of a gradient tensor (TV in d_flow, GD in d_src_rgb) could be
wrong by many times the bar unnoticed.  Here every term runs alone -- `term_mask` set to its VLG_TERM_* bit, the other
weights left at their defaults, since a masked term must vanish whatever its weight -- and is compared with the oracle
gradient of that single weighted term:
  * the fused op in every pass-1 organisation, K = 20 / 19 (19 takes pass1_kernel: lay_tile_kernel needs K % 4 == 0),
    5 and 30, near, compressive and far flow (far: one fixed-point group of pass 2 is zero or small), both paddings,
    shapes whose stencil pairs and 3x3 SSIM windows straddle every seam of the 32x8 tile, the 28-column rgb strip, the
    40x12 layout window and the 36x10 / 40x12 pass-1 stage;
  * the label-source op (lab_pix_kernel);
  * the reference's un-warped criteria (pass1_kernel without a warp) in fp32 and bf16, down to the 2xN and 3x3
    minimum sizes, with ignore_index 255, argmax maps and the data-parallel batch divisor.

Bars: 1e-5 in fp32 (normwise-max and RMS-relative for gradient tensors, against the fp32 or the fp64 evaluation of the
oracle on the same fp32 sampling positions), 1e-2 in bf16, exact where the arithmetic is exact.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import vlg_b200
from vlg_b200 import _cabi
from conftest import assert_grad_parity, assert_terms_parity
from oracle import torch_oracle as TO

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
RTOL_BF16 = 1e-2
RTOL_LINEAR = 2e-6      # five single-term runs against one all-terms run: same arithmetic, other association
W_TV = 0.7

TERMS = ("l1", "gd", "ssim", "ce", "tv")
BIT = dict(zip(TERMS, (_cabi.TERM_L1, _cabi.TERM_GD, _cabi.TERM_SSIM, _cabi.TERM_CE, _cabi.TERM_TV)))
SLOT = dict(zip(TERMS, (_cabi.LOSS_L1, _cabi.LOSS_GD, _cabi.LOSS_SSIM, _cabi.LOSS_CE, _cabi.LOSS_TV)))
_DEFAULTS = vlg_b200.WarpLossConfig(w_tv=W_TV)
WEIGHT = {t: getattr(_DEFAULTS, "w_" + t) for t in TERMS}
# which gradients a term reaches: (d_flow, d_src_rgb, d_src_layout)
REACH = {"l1": (True, True, False), "gd": (True, True, False), "ssim": (True, True, False),
         "ce": (True, False, True), "tv": (True, False, False)}

ORGS = {
    "default": {},                               # rgb_strip_kernel + lay_tile_kernel (K % 4 == 0)
    "tile": dict(layout_kernel="tile"),          # rgb_strip_kernel + pass1_kernel for the layout
    "tile_kernels": dict(tile_kernels=True),     # everything in pass1_kernel
    "no_tma": dict(use_tma=False),               # cp.async staging of the layout window
    "no_records": dict(pass2_records=False),     # pass 2 re-derives its taps from the coordinates
}


def _cl(t):
    return t.to(DEV).contiguous(memory_format=torch.channels_last)


def _zero(t):
    return t is not None and torch.count_nonzero(t).item() == 0


def _squeeze_flow(H, W):
    """Compressive near flow: x -> 0.3 x inside every 8-pixel tooth, so that source cells receive three to four output
    pixels each (|displacement| < 3 px)."""
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    return torch.stack((-0.7 * ((xx % 8) - 3.5), -0.6 * ((yy % 8) - 3.5)), -1)[None]


def _flow(N, H, W, kind, g):
    """[N,H,W,2] pixel flow.  near: smoothed sigma 2; squeeze: compressive sawtooth plus a little noise;
    far: smoothed sigma 48 with 5 % of the pixels uniform over the image (most pixels leave the near path)."""
    sigma = 48.0 if kind == "far" else 2.0
    flow = torch.randn(N, 2, H, W, generator=g) * sigma
    flow = F.avg_pool2d(F.pad(flow, (4, 4, 4, 4), mode="replicate"), 9, 1)
    if kind == "far":
        m = torch.rand(N, 1, H, W, generator=g) < 0.05
        flow = torch.where(m, (torch.rand(N, 2, H, W, generator=g) - 0.5) * 2 * max(H, W), flow)
    flow = flow.permute(0, 2, 3, 1).contiguous()
    if kind == "squeeze":
        flow = flow * 0.1 + _squeeze_flow(H, W)
    return flow


def _case(N, H, W, K, flow_kind, seed, ignore=-100):
    """Seeded inputs on the device: soft layout, per-pixel labels with ~5 % `ignore`."""
    g = torch.Generator().manual_seed(seed)
    mean = torch.tensor([0.485, 0.456, 0.406])[None, :, None, None]
    std = torch.tensor([0.229, 0.224, 0.225])[None, :, None, None]
    d = dict(src_rgb=(torch.rand(N, 3, H, W, generator=g) - mean) / std,
             tgt_rgb=(torch.rand(N, 3, H, W, generator=g) - mean) / std,
             src_layout=torch.randn(N, K, H, W, generator=g) * 2.0,
             src_label=torch.randint(0, K, (N, H, W), generator=g))
    lab = torch.randint(0, K, (N, H, W), generator=g)
    lab[torch.rand(N, H, W, generator=g) < 0.05] = ignore
    lab.view(-1)[0] = 0                     # at least one valid label
    d["tgt_label"] = lab
    d["flow"] = _flow(N, H, W, flow_kind, g)
    return {k: v.to(DEV) for k, v in d.items()}


def _warp_oracle(d, padding, dt, layout=None):
    """{term: (value, grads of WEIGHT[term] * term w.r.t. (flow, src_rgb, src_layout), None where unreached)} and the
    warped layout, by torch on the device in `dt`; fp64 samples at the fp32 positions (TO.high_precision_grid)."""
    layout = d["src_layout"] if layout is None else layout
    a, b, c = (t.to(dt).clone().requires_grad_(True) for t in (d["src_rgb"], layout, d["flow"]))
    N, H, W, _ = c.shape
    if dt == torch.float32:
        grid = TO.flow_to_grid(c)
    else:
        grid = TO.high_precision_grid(TO.flow_to_grid(d["flow"]), c, TO.flow_scale(H, W, torch.float32).to(dt).to(DEV))
    w_rgb, w_lay = TO.warp(a, grid, padding), TO.warp(b, grid, padding)
    tgt = d["tgt_rgb"].to(dt)
    vals = {"l1": TO.l1_loss(w_rgb, tgt), "gd": TO.gradient_loss(w_rgb, tgt), "ssim": TO.ssim_loss(w_rgb, tgt),
            "ce": TO.cross_entropy(w_lay, d["tgt_label"]), "tv": TO.flow_tv(c)}
    out = {}
    for t, v in vals.items():
        gr = torch.autograd.grad(WEIGHT[t] * v, (c, a, b), retain_graph=True, allow_unused=True)
        out[t] = (v.item(),) + tuple(gr)
    return out, w_lay.detach()


def _check_vec(vec, term, want32, want64, rtol, what, slots=TERMS):
    """The chosen slot against the oracle, every other term slot exactly 0, the total exactly the weighted slot
    (the total is summed in fp64 and rounded once: fp32 rounding of w * slot apart)."""
    for t in slots:
        if t != term:
            assert vec[SLOT[t]] == 0.0, f"{what}: slot {t} = {vec[SLOT[t]]!r} with only {term} evaluated"
    assert_terms_parity(vec[SLOT[term]:SLOT[term] + 1], [want32], None if want64 is None else [want64], rtol)
    w_slot = WEIGHT[term] * float(vec[SLOT[term]])
    assert abs(float(vec[_cabi.LOSS_TOTAL]) - w_slot) <= 2.4e-7 * abs(w_slot), (what, vec[_cabi.LOSS_TOTAL], w_slot)


# ------------------------------------------------------------------ 1. each term alone through the fused op
FUSED = [
    # organisation, K, flow, padding, (N, H, W)
    ("default", 20, "near", "border", (2, 17, 57)),
    ("default", 19, "squeeze", "zeros", (1, 9, 33)),
    ("default", 20, "far", "zeros", (2, 67, 129)),
    ("default", 20, "far_wide", "border", (3, 24, 84)),
    ("tile", 20, "squeeze", "zeros", (3, 24, 84)),
    ("tile", 19, "far", "border", (2, 17, 57)),
    ("tile_kernels", 20, "far", "border", (2, 67, 129)),
    ("tile_kernels", 19, "near", "zeros", (1, 9, 33)),
    ("no_tma", 20, "near", "zeros", (2, 67, 129)),
    ("no_tma", 19, "far_wide", "border", (3, 24, 84)),
    ("no_records", 20, "far_wide", "zeros", (1, 9, 33)),
    ("no_records", 19, "squeeze", "border", (2, 67, 129)),
    ("default", 5, "near", "zeros", (2, 17, 57)),
    ("default", 30, "far", "border", (1, 9, 33)),
    ("default", 20, "far", "border", (1, 375, 1242)),
]


@pytest.mark.parametrize("case", FUSED, ids=[f"{o}-k{k}-{fl}-{p}-{'x'.join(map(str, s))}" for o, k, fl, p, s in FUSED])
def test_each_term_alone_through_fused_op(case):
    org, K, flow_kind, padding, (N, H, W) = case
    d = _case(N, H, W, K, "far" if flow_kind == "far_wide" else flow_kind, seed=1000 + H * 7 + K)
    ref32, w_lay = _warp_oracle(d, padding, torch.float32)
    ref64, _ = _warp_oracle(d, padding, torch.float64)
    want_arg = torch.argmax(w_lay, 1)
    kw = dict(ORGS[org], far_packed=flow_kind != "far_wide", padding_mode=padding, want_argmax=True)

    def run(mask):
        a, b = _cl(d["src_rgb"]).requires_grad_(True), _cl(d["src_layout"]).requires_grad_(True)
        f = d["flow"].clone().requires_grad_(True)
        cfg = vlg_b200.WarpLossConfig(w_tv=W_TV, term_mask=mask, **kw)
        total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"]), d["tgt_label"], cfg)
        total.backward()
        return vec.cpu().double().numpy(), arg, (f.grad, a.grad, b.grad)

    sums = None
    for term in TERMS:
        vec, arg, grads = run(BIT[term])
        what = f"{term} alone {case}"
        _check_vec(vec, term, ref32[term][0], ref64[term][0], RTOL, what)
        assert torch.equal(arg, want_arg), what + ": argmax"
        if flow_kind != "near":
            assert (vec[_cabi.LOSS_MAXDISP] >= _cabi.NEAR_RADIUS) == flow_kind.startswith("far"), what
        for i, name in enumerate(("d_flow", "d_src_rgb", "d_src_layout")):
            if REACH[term][i]:
                assert_grad_parity(grads[i], ref32[term][1 + i], ref64[term][1 + i], RTOL, f"{what}: {name}")
            else:
                assert _zero(grads[i]), f"{what}: {name} must be exactly 0, max |g| = {grads[i].abs().max().item():.3e}"
        sums = [vec[_cabi.LOSS_TOTAL]] + list(grads) if sums is None else \
            [sums[0] + vec[_cabi.LOSS_TOTAL]] + [s + g for s, g in zip(sums[1:], grads)]

    # linearity: the five single-term runs add up to the all-terms run
    vec, arg, grads = run(0)
    assert torch.equal(arg, want_arg)
    assert abs(sums[0] - vec[_cabi.LOSS_TOTAL]) <= RTOL_LINEAR * abs(vec[_cabi.LOSS_TOTAL]), (sums[0], vec[_cabi.LOSS_TOTAL])
    for name, s, g in zip(("d_flow", "d_src_rgb", "d_src_layout"), sums[1:], grads):
        err = (s - g).abs().max().item()
        assert err <= RTOL_LINEAR * g.abs().max().item(), f"sum of single-term {name} vs all terms: {err:.3e} {case}"


# ------------------------------------------------------------------ 2. each term alone through the label-source op
LABELS = [
    # K, flow, padding, (N, H, W)
    (20, "near", "border", (2, 17, 57)),
    (19, "far", "zeros", (2, 67, 129)),
    (20, "far", "border", (1, 24, 84)),
]


@pytest.mark.parametrize("case", LABELS, ids=[f"k{k}-{fl}-{p}-{'x'.join(map(str, s))}" for k, fl, p, s in LABELS])
def test_each_term_alone_through_label_source_op(case):
    K, flow_kind, padding, (N, H, W) = case
    d = _case(N, H, W, K, flow_kind, seed=2000 + H + K)
    onehot = TO.one_hot_layout(d["src_label"].cpu(), K).to(DEV).contiguous()
    ref32, w_lay = _warp_oracle(d, padding, torch.float32, layout=onehot)
    ref64, _ = _warp_oracle(d, padding, torch.float64, layout=onehot)
    want_arg = torch.argmax(w_lay, 1)
    sum_total, sum_flow = 0.0, None
    for mask in [BIT[t] for t in TERMS] + [0]:
        f = d["flow"].clone().requires_grad_(True)
        cfg = vlg_b200.WarpLossConfig(w_tv=W_TV, term_mask=mask, padding_mode=padding, want_argmax=True)
        total, vec, arg = vlg_b200.warp_loss_labels(_cl(d["src_rgb"]), d["src_label"], f, _cl(d["tgt_rgb"]), d["tgt_label"],
                                                    cfg, n_classes=K)
        total.backward()
        vec = vec.cpu().double().numpy()
        assert torch.equal(arg, want_arg), (mask, case)
        if mask == 0:
            assert abs(sum_total - vec[_cabi.LOSS_TOTAL]) <= RTOL_LINEAR * abs(vec[_cabi.LOSS_TOTAL])
            err = (sum_flow - f.grad).abs().max().item()
            assert err <= RTOL_LINEAR * f.grad.abs().max().item(), f"sum of single-term d_flow vs all terms: {err:.3e}"
            continue
        term = TERMS[[BIT[t] for t in TERMS].index(mask)]
        what = f"{term} alone, label source {case}"
        _check_vec(vec, term, ref32[term][0], ref64[term][0], RTOL, what)
        assert_grad_parity(f.grad, ref32[term][1], ref64[term][1], RTOL, f"{what}: d_flow")
        sum_total += vec[_cabi.LOSS_TOTAL]
        sum_flow = f.grad.clone() if sum_flow is None else sum_flow + f.grad


# ------------------------------------------------------------------ 3. the un-warped criteria (src/loss.py, src/trainer.py:124,130)
def _pixel_inputs(N, H, W, K, dt, seed, ignore=-100, frac=0.05):
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(N, 3, H, W, generator=g)
    frame3 = torch.randn(N, 3, H, W, generator=g)
    seg = torch.randn(N, K, H, W, generator=g) * 3.0
    seg3 = torch.randint(0, K, (N, H, W), generator=g)
    seg3[torch.rand(N, H, W, generator=g) < frac] = ignore
    seg3.view(-1)[0] = 0
    # bf16: the oracle sees the same bf16-rounded values, in fp32
    img, frame3, seg = (t.to(dt).to(DEV) for t in (img, frame3, seg))
    return img, frame3, seg, seg3.to(DEV)


def _pixel_oracle(img, frame3, seg, seg3, dt, ignore_index=-100):
    """Oracle terms on the un-warped inputs in `dt`, with their gradients w.r.t. the rgb output and the logits.
    SSIM is 0 below 3x3 (the reference raises there; the product documents 0)."""
    a = img.to(dt).clone().requires_grad_(True)
    z = seg.to(dt).clone().requires_grad_(True)
    t = frame3.to(dt)
    H, W = a.shape[2], a.shape[3]
    vals = {"l1": TO.l1_loss(a, t), "gd": TO.gradient_loss(a, t),
            "ssim": TO.ssim_loss(a, t) if (H >= 3 and W >= 3) else (a * 0).sum(),
            "ce": F.cross_entropy(z, seg3, ignore_index=ignore_index)}
    out = {}
    for k, v in vals.items():
        ga, gz = torch.autograd.grad(v, (a, z), retain_graph=True, allow_unused=True)
        out[k] = (v.item(), ga, gz)
    return out


def _combine(ref, weights):
    """Value and gradients of sum_k weights[k] * term_k from the per-term oracle."""
    val = sum(w * ref[k][0] for k, w in weights.items())
    grads = []
    for i in (1, 2):
        gs = [w * ref[k][i] for k, w in weights.items() if ref[k][i] is not None]
        grads.append(sum(gs) if gs else None)
    return val, grads[0], grads[1]


PIXEL = [
    # (N, H, W), K, dtype
    ((1, 2, 5), 20, torch.float32),
    ((1, 5, 2), 5, torch.float32),
    ((1, 3, 3), 19, torch.float32),
    ((2, 17, 57), 30, torch.float32),
    ((1, 9, 33), 20, torch.float32),
    ((3, 24, 84), 19, torch.float32),
    ((2, 67, 129), 5, torch.float32),
    ((1, 375, 1242), 20, torch.float32),
    ((1, 2, 5), 19, torch.bfloat16),
    ((1, 3, 3), 20, torch.bfloat16),
    ((2, 17, 57), 19, torch.bfloat16),
    ((2, 67, 129), 30, torch.bfloat16),
    ((1, 375, 1242), 20, torch.bfloat16),
]
_DT = {torch.float32: "f32", torch.bfloat16: "bf16"}
_PIXEL_IDS = [f"{'x'.join(map(str, s))}-k{k}-{_DT[dt]}" for s, k, dt in PIXEL]


@pytest.mark.parametrize("shape,K,dt", PIXEL, ids=_PIXEL_IDS)
def test_reference_criteria_against_oracle(shape, K, dt):
    """L1Loss, GradientLoss, SsimLoss, CombinedLoss, CrossEntropyLoss and PixelLosses: value and input gradient."""
    N, H, W = shape
    img, frame3, seg, seg3 = _pixel_inputs(N, H, W, K, dt, seed=H * 131 + W + K)
    ref32 = _pixel_oracle(img, frame3, seg, seg3, torch.float32)
    ref64 = _pixel_oracle(img, frame3, seg, seg3, torch.float64) if dt == torch.float32 else None
    rtol = RTOL if dt == torch.float32 else RTOL_BF16
    has_ssim = H >= 3 and W >= 3
    rgb_criteria = ((vlg_b200.L1Loss(), {"l1": 1.0}), (vlg_b200.GradientLoss(), {"gd": 1.0}),
                    (vlg_b200.SsimLoss(), {"ssim": 1.0}), (vlg_b200.CombinedLoss(), {"gd": 1.0, "ssim": 1.0}))
    for mod, weights in rgb_criteria + ((vlg_b200.CrossEntropyLoss(), {"ce": 1.0}),):
        what = f"{type(mod).__name__} {shape} K={K} {dt}"
        x = (seg if "ce" in weights else img).clone().requires_grad_(True)
        out = mod(x, seg3) if "ce" in weights else mod(x, frame3)
        out.backward()
        assert x.grad.dtype == dt, what
        v32, ga32, gz32 = _combine(ref32, weights)
        g32 = gz32 if "ce" in weights else ga32
        if ref64 is not None:
            v64, ga64, gz64 = _combine(ref64, weights)
            g64 = gz64 if "ce" in weights else ga64
        else:
            v64, g64 = None, None
        if weights == {"ssim": 1.0} and not has_ssim:
            assert out.item() == 0.0 and _zero(x.grad), what
            continue
        assert_terms_parity([out.item()], [v32], None if v64 is None else [v64], rtol)
        assert_grad_parity(x.grad.float(), g32, g64, rtol, what)

    # the whole src/trainer.py:248-251 composition in one launch
    a, z = img.clone().requires_grad_(True), seg.clone().requires_grad_(True)
    crit = vlg_b200.PixelLosses()
    total = crit(a, frame3, z, seg3)
    total.backward()
    assert a.grad.dtype == dt and z.grad.dtype == dt
    weights = {"l1": 40.0, "gd": 20.0, "ssim": 20.0, "ce": 10.0}
    v32, ga32, gz32 = _combine(ref32, weights)
    v64, ga64, gz64 = _combine(ref64, weights) if ref64 is not None else (None, None, None)
    vec = crit.last_terms.cpu().double().numpy()
    assert_terms_parity(vec[:4], [ref32[k][0] for k in TERMS[:4]], None if ref64 is None else [ref64[k][0] for k in TERMS[:4]], rtol)
    assert vec[_cabi.LOSS_TV] == 0.0 and (has_ssim or vec[_cabi.LOSS_SSIM] == 0.0)
    assert vec[_cabi.LOSS_NVALID] == (seg3 != -100).sum().item()
    assert_terms_parity([total.item()], [v32], None if v64 is None else [v64], rtol)
    assert_grad_parity(a.grad.float(), ga32, ga64, rtol, f"PixelLosses d_img {shape} K={K} {dt}")
    assert_grad_parity(z.grad.float(), gz32, gz64, rtol, f"PixelLosses d_seg {shape} K={K} {dt}")


@pytest.mark.parametrize("shape,K,dt", [((2, 17, 57), 20, torch.float32), ((1, 9, 33), 19, torch.float32),
                                        ((1, 5, 2), 30, torch.float32), ((3, 24, 84), 5, torch.bfloat16)],
                         ids=["2x17x57-k20-f32", "1x9x33-k19-f32", "1x5x2-k30-f32", "3x24x84-k5-bf16"])
def test_each_term_alone_through_pixel_losses(shape, K, dt):
    """The un-warped pass with one VLG_TERM_* bit and the default weights: the other slots read 0, the other
    gradient is exactly 0, the chosen term matches the oracle (TV has no meaning without a flow: everything is 0)."""
    N, H, W = shape
    img, frame3, seg, seg3 = _pixel_inputs(N, H, W, K, dt, seed=77 + H + K)
    ref32 = _pixel_oracle(img, frame3, seg, seg3, torch.float32)
    ref64 = _pixel_oracle(img, frame3, seg, seg3, torch.float64) if dt == torch.float32 else None
    rtol = RTOL if dt == torch.float32 else RTOL_BF16
    for term in TERMS:
        a, z = img.clone().requires_grad_(True), seg.clone().requires_grad_(True)
        cfg = vlg_b200.WarpLossConfig(w_tv=W_TV, term_mask=BIT[term], want_argmax=True)
        total, vec, arg = vlg_b200.pixel_losses(a, frame3, z, seg3, cfg)
        total.backward()
        vec = vec.cpu().double().numpy()
        what = f"{term} alone, un-warped {shape} K={K} {dt}"
        assert torch.equal(arg, torch.argmax(seg, 1)), what
        if term == "tv" or (term == "ssim" and not (H >= 3 and W >= 3)):
            assert (vec[:_cabi.LOSS_TOTAL + 1] == 0.0).all() and _zero(a.grad) and _zero(z.grad), what
            continue
        _check_vec(vec, term, ref32[term][0], None if ref64 is None else ref64[term][0], rtol, what)
        w = WEIGHT[term]
        if term == "ce":
            assert _zero(a.grad), what + ": d_img must be exactly 0"
            assert_grad_parity(z.grad.float(), w * ref32[term][2], None if ref64 is None else w * ref64[term][2], rtol, what)
        else:
            assert _zero(z.grad), what + ": d_seg must be exactly 0"
            assert_grad_parity(a.grad.float(), w * ref32[term][1], None if ref64 is None else w * ref64[term][1], rtol, what)


@pytest.mark.parametrize("K", [19, 20])
def test_ignore_index_255(K):
    """Cityscapes marks unlabelled pixels 255 (>= K): they are skipped, not reported as bad labels."""
    N, H, W = 2, 67, 129
    img, frame3, seg, seg3 = _pixel_inputs(N, H, W, K, torch.float32, seed=255 + K, ignore=255, frac=0.2)
    seg3[0, :3] = 255                               # whole rows, across several tiles
    z_ref = seg.clone().requires_grad_(True)
    ref = F.cross_entropy(z_ref, seg3, ignore_index=255)
    ref.backward()
    z = seg.clone().requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(w_l1=0.0, w_gd=0.0, w_ssim=0.0, w_ce=1.0, term_mask=_cabi.TERM_CE, ignore_index=255,
                                  debug=True)
    total, vec, _ = vlg_b200.pixel_losses(None, None, z, seg3, cfg)     # debug: raises on STATUS_BAD_LABEL
    total.backward()
    np.testing.assert_allclose(vec[_cabi.LOSS_CE].item(), ref.item(), rtol=RTOL)
    assert vec[_cabi.LOSS_NVALID].item() == (seg3 != 255).sum().item()
    assert_grad_parity(z.grad, z_ref.grad, None, RTOL, f"d_logits ignore_index=255 K={K}")
    out = vlg_b200.CrossEntropyLoss(ignore_index=255)(seg, seg3)
    np.testing.assert_allclose(out.item(), ref.item(), rtol=RTOL)

    # the fused op (lay_tile_kernel for K = 20, pass1_kernel for K = 19) with the same labels
    d = _case(N, H, W, K, "near", seed=256 + K, ignore=255)
    d["tgt_label"] = seg3
    ref32, _ = _warp_oracle(dict(d, tgt_label=torch.where(seg3 == 255, -100, seg3)), "border", torch.float32)
    b = _cl(d["src_layout"]).requires_grad_(True)
    f = d["flow"].clone().requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(term_mask=_cabi.TERM_CE, ignore_index=255, debug=True)
    total, vec, _ = vlg_b200.warp_loss(_cl(d["src_rgb"]), b, f, _cl(d["tgt_rgb"]), seg3, cfg)
    total.backward()
    np.testing.assert_allclose(vec[_cabi.LOSS_CE].item(), ref32["ce"][0], rtol=RTOL)
    assert vec[_cabi.LOSS_NVALID].item() == (seg3 != 255).sum().item()
    assert_grad_parity(f.grad, ref32["ce"][1], None, RTOL, f"d_flow ignore_index=255 K={K}")
    assert_grad_parity(b.grad, ref32["ce"][3], None, RTOL, f"d_src_layout ignore_index=255 K={K}")


@pytest.mark.parametrize("K", [5, 19, 20, 30])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_pixel_losses_argmax_bit_exact(K, dt):
    """PixelLosses(want_argmax=True) writes torch.argmax(seg, 1) bit for bit, ties to the first maximal index."""
    img, frame3, seg, seg3 = _pixel_inputs(2, 37, 70, K, dt, seed=K)
    g = torch.Generator().manual_seed(K + 1)
    tie = (torch.rand(2, 37, 70, generator=g) < 0.3).to(DEV)
    c0, c1 = K // 3, K - 1                                   # equal maxima in two channels
    seg = seg.clone()
    seg[:, c0] = torch.where(tie, torch.full_like(seg[:, c0], 20.0), seg[:, c0])
    seg[:, c1] = torch.where(tie, torch.full_like(seg[:, c1], 20.0), seg[:, c1])
    crit = vlg_b200.PixelLosses(want_argmax=True)
    crit(img, frame3, seg, seg3)
    want = torch.argmax(seg, 1)
    assert (want[tie] == c0).all()
    assert torch.equal(crit.last_argmax, want)


@pytest.mark.parametrize("shape,K,dt", [((2, 17, 57), 19, torch.float32), ((1, 9, 33), 20, torch.float32),
                                        ((2, 67, 129), 20, torch.bfloat16)],
                         ids=["2x17x57-k19-f32", "1x9x33-k20-f32", "2x67x129-k20-bf16"])
def test_global_batch_halves_everything(shape, K, dt):
    """Data-parallel divisor: with global_batch = 2N every loss slot and every gradient is exactly half of the
    global_batch = 0 result (all scales involved are powers of two); the valid-label count is unchanged."""
    N, H, W = shape
    img, frame3, seg, seg3 = _pixel_inputs(N, H, W, K, dt, seed=H + K)
    res = []
    for gb in (0, 2 * N):
        a, z = img.clone().requires_grad_(True), seg.clone().requires_grad_(True)
        cfg = vlg_b200.WarpLossConfig(global_batch=gb, term_mask=_cabi.TERM_L1 | _cabi.TERM_GD | _cabi.TERM_SSIM | _cabi.TERM_CE)
        total, vec, _ = vlg_b200.pixel_losses(a, frame3, z, seg3, cfg)
        total.backward()
        res.append((vec.clone(), a.grad.clone(), z.grad.clone()))
    (v0, a0, z0), (v1, a1, z1) = res
    assert torch.equal(v1[:_cabi.LOSS_TOTAL + 1], v0[:_cabi.LOSS_TOTAL + 1] * 0.5), (v0, v1)
    assert v1[_cabi.LOSS_NVALID] == v0[_cabi.LOSS_NVALID]
    assert torch.equal(a1, a0 * 0.5) and torch.equal(z1, z0 * 0.5)
    assert v0[_cabi.LOSS_TOTAL].item() > 0 and a0.abs().max().item() > 0 and z0.abs().max().item() > 0
