"""The bar a bf16 output of the product is held to.

The kernels widen bf16 operands to fp32 on load (exact), compute and stage every intermediate in fp32, and round
to bf16 once, when they store an output activation or gradient (`from_f` / `store_px`, round to nearest even).
So on bf16-valued inputs a bf16 output is the fp32 result rounded once:

  * the fp32 result g32 meets the fp32 parity bar against the oracle evaluated on the same bf16 values:
    |g32 - ref| <= 1e-5 max|ref| (normwise, conftest.assert_grad_parity);
  * bf16 keeps an 8-bit significand (7 stored bits and the implicit one), so round-to-nearest errs by at most half
    a unit in the last place: |bf16(x) - x| <= 2^-8 |x|.

Together, element by element, |g - ref| <= 2^-8 |ref| + 1e-5 max|ref| (the cross term 2^-8 * 1e-5 max|ref| is
below what the fp32 bar itself measures).  A truncating store (error up to 2^-7 |x|), a second rounding of an
intermediate to bf16, or one wrong small element all break it, where a bar relative to the largest element does not.
"""
import torch

U_BF16 = 2.0 ** -8      # unit roundoff of bf16 (round to nearest)
RTOL_F32 = 1e-5         # the fp32 parity bar (BASELINE.json north_star)


def assert_bf16_rounded_once(got, ref32, ref64, what, rtol=RTOL_F32):
    """`got` (bf16) is the oracle value rounded once to bf16, element by element:
         |got - ref| <= 2^-8 |ref| + rtol * max|ref|
    against the fp32 OR the fp64 evaluation of the oracle (`ref64` may be None), per element -- the tie-breaker of
    conftest.assert_grad_parity, where torch's fp32 scatter drifts.  Also RMS-relative:
         ||got - ref||_2 <= (rtol + 2^-8) ||ref||_2   against either.
    The failure message names the worst element: index, got, ref."""
    g = torch.as_tensor(got).detach()
    assert g.dtype == torch.bfloat16, f"{what}: expected a bf16 tensor, got {g.dtype}"
    g = g.double()
    refs = [torch.as_tensor(r).detach().to(g.device).double() for r in (ref32, ref64) if r is not None]
    ok = torch.zeros(g.shape, dtype=torch.bool, device=g.device)
    excess = None           # per element: error over the bar, the smaller of the two oracles
    rms = []
    for r in refs:
        assert r.shape == g.shape, f"{what}: shape {tuple(g.shape)} vs oracle {tuple(r.shape)}"
        err = (g - r).abs()
        bar = U_BF16 * r.abs() + rtol * r.abs().max()
        ok |= err <= bar
        e = err - bar
        excess = e if excess is None else torch.minimum(excess, e)
        rms.append((g - r).square().sum().sqrt().item() / max(r.square().sum().sqrt().item(), 1e-300))
    if not bool(ok.all()):
        flat = int(torch.argmax(excess).item())
        idx = tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), g.shape))
        refs_at = ", ".join(f"{r[idx].item():.9g}" for r in refs)
        raise AssertionError(
            f"{what}: {int((~ok).sum().item())} of {g.numel()} elements beyond 2^-8 |ref| + {rtol:g} max|ref|; worst at "
            f"{idx}: got {g[idx].item():.9g}, ref (fp32, fp64) {refs_at}, max|ref| {refs[0].abs().max().item():.6g}")
    assert min(rms) <= rtol + U_BF16, (
        f"{what}: RMS-relative {[f'{x:.3e}' for x in rms]} (vs fp32 oracle, vs fp64 oracle), bar {rtol + U_BF16:.3e}")
