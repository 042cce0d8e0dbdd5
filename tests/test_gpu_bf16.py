"""bf16 is storage only: what the oracle-parametrised tests cannot take as one more parameter (run on a GPU).

The kernels widen bf16 to fp32 on load, compute and stage d_out in fp32, and round once when they store an output
(bf16_bars).  So the same bf16-valued inputs given as fp32 tensors and as bf16 tensors must give the same step:
  * for every organisation of a bf16 step (the table below), with near and far flow;
  * in validation (no gradient) and flow-only calls;
  * under an upstream gradient scale (scale_multi_kernel);
  * with the coordinates given as a sampling grid.

Organisations (selection: run_pass1 / launch_pass2 / pass2_from_records in csrc/vlg_api.cu).  `lay_tile` says whether
the layout terms run in lay_tile_kernel (else pass1_kernel) -- the tests read it back from the kernel timeline.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import vlg_b200
from vlg_b200 import _cabi
from conftest import assert_grad_parity, assert_terms_parity
from bf16_bars import assert_bf16_rounded_once
from oracle import torch_oracle as TO
from test_gpu_parity import _cl, _make_case

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5
RTOL_ASSOC = 2e-6       # loss slots: same arithmetic, partial sums associated by a grid sized per instantiation
F32, BF16 = torch.float32, torch.bfloat16

ORGS = [
    # id, K, (N, H, W), config, lay_tile for fp32, lay_tile for bf16
    # K = 20, even W: lay_tile_kernel<bf16,20,PX8> + pass2_rec_kernel, as fp32 (lay_tile_kernel<float,20>)
    ("k20-even", 20, (2, 33, 70), {}, True, True),
    # K = 20, odd W: a bf16 row is not a 16-byte multiple (make_window_map), so bf16 takes pass1_kernel +
    # tap_records_kernel; fp32 stays on lay_tile_kernel.  Both gather pass 2 from the records.
    ("k20-odd", 20, (2, 33, 69), {}, True, False),
    # use_tma=False: pass1_kernel + pass2_kernel with cp.async staging, both dtypes
    ("k20-no_tma", 20, (2, 33, 70), dict(use_tma=False), False, False),
    # pass2_records=False: lay_tile_kernel + pass2_kernel with the TMA d_out map, both dtypes
    ("k20-no_records", 20, (2, 33, 70), dict(pass2_records=False), True, True),
    # K % 4 != 0: pass1_kernel + pass2_kernel (cp.async), both dtypes
    ("k19", 19, (2, 33, 69), {}, False, False),
    ("k30", 30, (1, 40, 70), {}, False, False),
    ("k5", 5, (2, 33, 69), {}, False, False),
]
_ORG_IDS = [o[0] for o in ORGS]
FLOWS = {"near": (2.0, 0.0), "far": (48.0, 0.05)}     # sigma, fraction of pixels uniform over the image


def _inputs(K, shape, flow_kind, seed):
    """A seeded case whose activations are bf16 values, held in fp32."""
    sigma, far = FLOWS[flow_kind]
    d = _make_case(*shape, K, sigma, seed=seed, layout="soft", far_frac=far)
    return dict(d, **{k: d[k].to(BF16).float() for k in ("src_rgb", "src_layout", "tgt_rgb")})


def _step(d, dt, cfg, grads=(True, True, True), timeline=False):
    """The fused op on `d` with activations in `dt`.  grads: which of (flow, src_rgb, src_layout) require a gradient;
    none -> a call under torch.no_grad().  Returns (vec, argmax, d_flow, d_src_rgb, d_src_layout, lay_tile ran)."""
    a = _cl(d["src_rgb"].to(dt)).requires_grad_(grads[1])
    b = _cl(d["src_layout"].to(dt)).requires_grad_(grads[2])
    f = d["flow"].to(DEV).requires_grad_(grads[0])
    lib = _cabi.load()
    if timeline:
        _cabi.check(lib.vlg_timeline_arm(1))
    if any(grads):
        total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"].to(dt)), d["tgt_label"].to(DEV), cfg)
        total.backward()
    else:
        with torch.no_grad():
            total, vec, arg = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"].to(dt)), d["tgt_label"].to(DEV), cfg)
    lay_tile = None
    if timeline:
        _cabi.check(lib.vlg_timeline_arm(0))
        ms4 = (C.c_float * 4)()
        _cabi.check(lib.vlg_timeline_read(ms4))
        lay_tile = ms4[1] >= 0.0            # -1: lay_tile_kernel did not run
    return vec.clone(), arg.clone(), f.grad, a.grad, b.grad, lay_tile


@pytest.mark.parametrize("flow_kind", list(FLOWS))
@pytest.mark.parametrize("org", ORGS, ids=_ORG_IDS)
def test_bf16_is_storage_only(org, flow_kind):
    """The same bf16-valued inputs as fp32 tensors and as bf16 tensors.  Same organisation in both dtypes: pass 1
    stages d_out in fp32 in both and pass 2 accumulates in the same order, so d_flow is bitwise equal and the bf16
    source gradients are the fp32 ones rounded once, bitwise; argmax is bitwise equal.  Organisations that differ
    (K = 20, odd W) are held to the bars of test_kernel_organisations_agree, the bf16 gradients rounded once."""
    name, K, shape, kw, tile32, tile16 = org
    d = _inputs(K, shape, flow_kind, seed=K * 7 + shape[2])
    cfg = vlg_b200.WarpLossConfig(w_tv=0.4, want_argmax=True, **kw)
    v32, arg32, gf32, ga32, gb32, lt32 = _step(d, F32, cfg, timeline=True)
    v16, arg16, gf16, ga16, gb16, lt16 = _step(d, BF16, cfg, timeline=True)
    assert (lt32, lt16) == (tile32, tile16), f"{name}: lay_tile_kernel ran (fp32, bf16) = {(lt32, lt16)}"
    if flow_kind == "far":
        assert v16[_cabi.LOSS_MAXDISP].item() >= _cabi.NEAR_RADIUS
    assert ga16.dtype == BF16 and gb16.dtype == BF16 and gf16.dtype == F32
    assert torch.equal(arg16, arg32), name
    assert ga32.abs().max().item() > 0 and gb32.abs().max().item() > 0
    np.testing.assert_allclose(v16[:6].cpu().numpy(), v32[:6].cpu().numpy(), rtol=RTOL_ASSOC)
    assert torch.equal(v16[_cabi.LOSS_NVALID:], v32[_cabi.LOSS_NVALID:])
    if tile32 == tile16:
        assert torch.equal(gf16, gf32), f"{name} {flow_kind}: d_flow"
        assert torch.equal(ga16, ga32.to(BF16)), f"{name} {flow_kind}: d_src_rgb"
        assert torch.equal(gb16, gb32.to(BF16)), f"{name} {flow_kind}: d_src_layout"
    else:
        err = (gf16 - gf32).abs().max().item()
        assert err <= RTOL * gf32.abs().max().item(), (name, flow_kind, "d_flow", err)
        assert_bf16_rounded_once(ga16, ga32, None, f"{name} {flow_kind}: d_src_rgb vs the fp32 organisation")
        assert_bf16_rounded_once(gb16, gb32, None, f"{name} {flow_kind}: d_src_layout vs the fp32 organisation")


@pytest.mark.parametrize("org", ORGS, ids=_ORG_IDS)
def test_bf16_validation_and_flow_only_calls(org):
    """A bf16 step without gradients (torch.no_grad()) and with the flow gradient only (sources without
    requires_grad): the loss vector and argmax bitwise equal to the training call, and the flow-only d_flow too."""
    name, K, shape, kw, _, _ = org
    d = _inputs(K, shape, "far", seed=K * 11 + shape[1])
    cfg = vlg_b200.WarpLossConfig(w_tv=0.4, want_argmax=True, **kw)
    vec, arg, gf, _, _, _ = _step(d, BF16, cfg)
    for grads in ((False, False, False), (True, False, False)):
        v, a, g, ga, gb, _ = _step(d, BF16, cfg, grads=grads)
        what = f"{name}, gradients {grads}"
        assert torch.equal(v, vec), what + ": loss vector"
        assert torch.equal(a, arg), what + ": argmax"
        assert ga is None and gb is None
        if grads[0]:
            assert torch.equal(g, gf), what + ": d_flow"


@pytest.mark.parametrize("K,shape", [(20, (1, 9, 33)), (19, (1, 9, 34))], ids=["k20-1x9x33", "k19-1x9x34"])
def test_bf16_upstream_gradient_scale(K, shape):
    """(0.3 * total).backward(): scale_multi_kernel widens each bf16 gradient, multiplies by the fp32 scale and rounds
    once more, so the result is round(round(g) * s) -- a double rounding, the intended semantics (the unit-scale
    gradient is produced by the step itself; a scale != 1 is a separate pass over the stored tensors).  That is bit for
    bit (g1.float() * torch.tensor(0.3)).bfloat16(); d_flow (fp32) is g1 * 0.3f.  Element counts are not multiples
    of 8 (N*3*H*W = 891 / 918, N*K*H*W = 5940 / 5814), so the tails of the vectorised loop are reached."""
    d = _inputs(K, shape, "near", seed=5 + K)
    res = []
    for scale in (1.0, 0.3):
        a = _cl(d["src_rgb"].to(BF16)).requires_grad_(True)
        b = _cl(d["src_layout"].to(BF16)).requires_grad_(True)
        f = d["flow"].to(DEV).requires_grad_(True)
        total, _, _ = vlg_b200.warp_loss(a, b, f, _cl(d["tgt_rgb"].to(BF16)), d["tgt_label"].to(DEV),
                                         vlg_b200.WarpLossConfig(w_tv=0.4))
        (total * scale).backward()
        res.append((a.grad, b.grad, f.grad))
    s = torch.tensor(0.3, device=DEV)
    (ga1, gb1, gf1), (ga, gb, gf) = res
    assert torch.equal(ga, (ga1.float() * s).to(BF16)) and torch.equal(gb, (gb1.float() * s).to(BF16))
    assert torch.equal(gf, gf1 * s)
    assert ga.dtype == BF16 and ga1.abs().max().item() > 0 and gb1.abs().max().item() > 0


@pytest.mark.parametrize("org", [o for o in ORGS if o[0] in ("k20-even", "k20-odd", "k20-no_tma", "k19")],
                         ids=["k20-even", "k20-odd", "k20-no_tma", "k19"])
@pytest.mark.parametrize("padding", ["border", "zeros"])
def test_bf16_coordinates_as_grid(org, padding):
    """coords_are_grid=True in bf16, once per pass-1 organisation (lay_tile_kernel PX8, pass1_kernel by width, by
    request and by K), against the oracle in fp32 and fp64 on the same bf16 values: losses and d_grid at the fp32 bar,
    the source gradients rounded once, argmax bit for bit."""
    name, K, shape, kw, _, tile16 = org
    d = _inputs(K, shape, "far", seed=K + shape[2])
    grid = TO.flow_to_grid(d["flow"])
    ref = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], grid, d["tgt_rgb"], d["tgt_label"], padding_mode=padding,
                               is_grid=True)
    ref64 = TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], grid, d["tgt_rgb"], d["tgt_label"], padding_mode=padding,
                                 is_grid=True, dtype=torch.float64)
    cfg = vlg_b200.WarpLossConfig(padding_mode=padding, coords_are_grid=True, want_argmax=True, **kw)
    vec, arg, gg, ga, gb, lt = _step(dict(d, flow=grid), BF16, cfg, timeline=True)
    what = f"{name} {padding} grid"
    assert lt == tile16, what
    terms = lambda r: np.array([r["terms"][k].item() for k in ("l1", "gd", "ssim", "ce", "tv")])
    assert_terms_parity(vec.cpu().numpy()[:5], terms(ref), terms(ref64), RTOL)
    assert torch.equal(arg.cpu(), ref["argmax"]), what
    assert_grad_parity(gg, ref["d_flow"], ref64["d_flow"], RTOL, what + ": d_grid")
    assert_bf16_rounded_once(ga.cpu(), ref["d_src_rgb"], ref64["d_src_rgb"], what + ": d_src_rgb")
    assert_bf16_rounded_once(gb.cpu(), ref["d_src_layout"], ref64["d_src_layout"], what + ": d_src_layout")
