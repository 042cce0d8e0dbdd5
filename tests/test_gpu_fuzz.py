"""Property / fuzz tests on the GPU (hypothesis): random small shapes -- ragged tiles, 2-pixel images,
both paddings, flow and grid coordinates, ignored labels, K in {5, 19, 20, 30}, fp32 and bf16 activations (odd
widths take bf16 K = 20 to pass1_kernel) -- against the torch oracle."""
import os

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings, strategies as st

import vlg_b200
from vlg_b200 import _cabi
from oracle import torch_oracle as TO
from conftest import assert_grad_parity, assert_terms_parity
from bf16_bars import assert_bf16_rounded_once

pytestmark = pytest.mark.gpu
DEV = "cuda"
RTOL = 1e-5   # BASELINE.json north_star: losses and gradients within 1e-5 relative in fp32


def _cl(t):
    return t.to(DEV).contiguous(memory_format=torch.channels_last)


# VLG_FUZZ_EXAMPLES=N: a longer, non-derandomised campaign (run by hand on a GPU box; the default stays fast and reproducible)
_N_EX = int(os.environ.get("VLG_FUZZ_EXAMPLES", "30"))


@settings(max_examples=_N_EX, deadline=None, suppress_health_check=list(HealthCheck), derandomize=(_N_EX == 30))
@given(N=st.integers(1, 2), H=st.integers(2, 37), W=st.integers(2, 70), K=st.sampled_from([5, 19, 20, 30]),
       padding=st.sampled_from(["border", "zeros"]), as_grid=st.booleans(),
       sigma=st.sampled_from([0.0, 0.4, 2.0, 9.0]), seed=st.integers(0, 2 ** 16), ignore=st.booleans(),
       dtype=st.sampled_from([torch.float32, torch.bfloat16]))
def test_fuzz_warp_loss_against_oracle(N, H, W, K, padding, as_grid, sigma, seed, ignore, dtype):
    g = torch.Generator().manual_seed(seed)
    # activations rounded to `dtype` (kept in fp32 for the oracle): the oracle sees the values the product sees
    rnd = lambda t: t.to(dtype).float()
    src_rgb = rnd(torch.randn(N, 3, H, W, generator=g))
    src_lay = rnd(torch.randn(N, K, H, W, generator=g))
    tgt_rgb = rnd(torch.randn(N, 3, H, W, generator=g))
    label = torch.randint(0, K, (N, H, W), generator=g)
    if ignore:
        label[torch.rand(N, H, W, generator=g) < 0.2] = -100
        if (label != -100).sum() == 0:
            label[0, 0, 0] = 0
    flow = torch.randn(N, H, W, 2, generator=g) * sigma
    coords = TO.flow_to_grid(flow) if as_grid else flow
    w_tv = 0.0 if as_grid else 0.7
    has_ssim = H >= 3 and W >= 3

    # oracle (SSIM is undefined below 3x3: the product reports 0 for it, the reference would raise), evaluated in
    # fp32 and -- as the tie-breaker of SURVEY Appendix A.10 -- in fp64 on the SAME fp32 sampling grid
    def oracle(dt):
        a, b, c = (t.to(dt).clone().requires_grad_(True) for t in (src_rgb, src_lay, coords))
        if dt == torch.float32:
            grid = c if as_grid else TO.flow_to_grid(c)
        else:   # same fp32 sampling positions (the spec), fp64 accumulation: TO.high_precision_grid
            g32 = coords if as_grid else TO.flow_to_grid(coords)
            grid = TO.high_precision_grid(g32, c, 1.0 if as_grid else TO.flow_scale(H, W, torch.float32).to(dt))
        w_rgb, w_lay = TO.warp(a, grid, padding), TO.warp(b, grid, padding)
        terms = [TO.l1_loss(w_rgb, tgt_rgb.to(dt)), TO.gradient_loss(w_rgb, tgt_rgb.to(dt)),
                 TO.ssim_loss(w_rgb, tgt_rgb.to(dt)) if has_ssim else torch.zeros(()), TO.cross_entropy(w_lay, label),
                 TO.flow_tv(c) if (not as_grid and H > 1 and W > 1) else torch.zeros(())]
        total = 40 * terms[0] + 20 * (terms[1] + terms[2]) + 10 * terms[3] + w_tv * terms[4]
        total.backward()
        return np.array([t.item() for t in terms]), w_lay.detach(), (c.grad, a.grad, b.grad)

    want32, w_lay, g32_ = oracle(torch.float32)
    want64, _, g64_ = oracle(torch.float64)

    ga, gb = _cl(src_rgb.to(dtype)).requires_grad_(True), _cl(src_lay.to(dtype)).requires_grad_(True)
    gc = coords.to(DEV).requires_grad_(True)
    cfg = vlg_b200.WarpLossConfig(w_tv=w_tv, padding_mode=padding, coords_are_grid=as_grid, want_argmax=True)
    tot, vec, arg = vlg_b200.warp_loss(ga, gb, gc, _cl(tgt_rgb.to(dtype)), label.to(DEV), cfg)
    tot.backward()

    case = (N, H, W, K, padding, as_grid, sigma, seed, dtype)
    # the loss vector and d_coords are fp32 outputs in both dtypes; a bf16 source gradient is the fp32 one rounded once
    assert_terms_parity(vec.cpu().numpy()[:5], want32, want64, RTOL)
    assert torch.equal(arg.cpu(), torch.argmax(w_lay, 1)), case
    assert_grad_parity(gc.grad.detach().cpu().contiguous(), g32_[0], g64_[0], RTOL, f"d_coords {case}")
    for name, x, r32, r64 in (("d_src_rgb", ga.grad, g32_[1], g64_[1]), ("d_src_layout", gb.grad, g32_[2], g64_[2])):
        x = x.detach().cpu().contiguous()
        assert x.dtype == dtype, f"{name} {case}"
        if dtype == torch.bfloat16:
            assert_bf16_rounded_once(x, r32, r64, f"{name} {case}")
        else:
            assert_grad_parity(x, r32, r64, RTOL, f"{name} {case}")
