"""vlg_confusion on the B200: every count is compared by exact integer equality with
torch.bincount((t*K + p)[t != ignore], minlength=K*K) evaluated on the CPU."""
import pytest
import torch

import vlg_b200

pytestmark = pytest.mark.gpu

DEV = "cuda"


def oracle(pred, target, K, ignore=-100):
    """K*K + 1 counts: bincount of the in-range pixels, then the non-ignored pixels with a label outside [0, K)."""
    p, t = pred.cpu(), target.cpu()
    keep = t != ignore
    inr = keep & (t >= 0) & (t < K) & (p >= 0) & (p < K)
    out = torch.zeros(K * K + 1, dtype=torch.int64)
    out[:K * K] = torch.bincount((t * K + p)[inr], minlength=K * K)
    out[K * K] = int((keep & ~inr).sum())
    return out


def counts_of(pred, target, K, ignore=-100):
    counts = torch.zeros(K * K + 1, dtype=torch.int64, device=target.device)
    vlg_b200.ops._confusion_into(counts, pred, target, K, ignore_index=ignore)
    return counts.cpu()


def make_labels(kind, N, H, W, K, g):
    if kind == "random":
        return torch.randint(0, K, (N, H, W), generator=g)
    if kind == "blocks":   # Cityscapes-like piecewise-constant 32x32 blocks
        b = torch.randint(0, K, (N, (H + 31) // 32, (W + 31) // 32), generator=g)
        return b.repeat_interleave(32, 1).repeat_interleave(32, 2)[:, :H, :W].contiguous()
    return torch.full((N, H, W), K - 1, dtype=torch.int64)   # "one": every pixel in one bin


def sprinkle_ignore(t, ignore, g, frac=0.1):
    t = t.clone()
    t[torch.rand(t.shape, generator=g) < frac] = ignore
    return t


def offset_by_one(x):
    """The same values one element past a 16-byte boundary: forces the scalar label path."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    buf[1:].copy_(x.reshape(-1))
    return buf[1:].view(x.shape)


# ---------------------------------------------------------------- label mode
SHAPES = [(1, 2, 2), (3, 5, 7), (16, 256, 512), (8, 1024, 2048)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("K", [20, 19, 30, 5])
@pytest.mark.parametrize("ignore", [-100, 255])
@pytest.mark.parametrize("kind", ["random", "blocks", "one"])
def test_label_mode_matches_bincount(shape, K, ignore, kind):
    N, H, W = shape
    g = torch.Generator().manual_seed(N * 7919 + H * 31 + W + K)
    t = make_labels(kind, N, H, W, K, g)
    if kind != "one":
        t = sprinkle_ignore(t, ignore, g)
    p = make_labels(kind if kind != "blocks" else "random", N, H, W, K, g) if kind != "one" else t.clone()
    if kind == "blocks":   # mostly right, like a trained model: the prediction is the target with some blocks changed
        p = torch.where(make_labels("blocks", N, H, W, 2, g) == 0, t.clamp(0, K - 1), p)
    want = oracle(p, t, K, ignore)
    assert int(want[K * K]) == 0
    pd, td = p.to(DEV), t.to(DEV)
    assert torch.equal(counts_of(pd, td, K, ignore), want)
    assert torch.equal(counts_of(offset_by_one(pd), offset_by_one(td), K, ignore), want)        # scalar path
    assert torch.equal(counts_of(pd, offset_by_one(td), K, ignore), want)
    cm = vlg_b200.confusion_matrix(pd, td, K, ignore_index=ignore)
    assert cm.shape == (K, K) and cm.dtype == torch.int64 and torch.equal(cm.cpu().reshape(-1), want[:K * K])


# ---------------------------------------------------------------- layout mode
def as_layout(x, nchw):
    return x.contiguous() if nchw else x.contiguous(memory_format=torch.channels_last)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("nchw", [False, True], ids=["nhwc", "nchw"])
@pytest.mark.parametrize("K", [20, 19, 30, 5])
@pytest.mark.parametrize("shape", [(2, 3, 5), (4, 64, 96)], ids=lambda s: "x".join(map(str, s)))
def test_layout_mode_matches_torch_argmax(dtype, nchw, K, shape):
    N, H, W = shape
    g = torch.Generator().manual_seed(K * 101 + H)
    scores = torch.randn(N, K, H, W, generator=g).to(dtype)
    if dtype == torch.bfloat16:   # coarse scores: many exact ties between channels
        scores = (scores * 2).round().to(dtype)
    t = sprinkle_ignore(torch.randint(0, K, (N, H, W), generator=g), -100, g)
    want = oracle(torch.argmax(scores.float(), 1), t, K)
    lay, td = as_layout(scores.to(DEV), nchw), t.to(DEV)
    assert torch.equal(counts_of(lay, td, K), want)
    # ties resolve to the first maximal channel, as torch.argmax on the device does
    assert torch.equal(counts_of(torch.argmax(lay, 1), td, K), want)


def test_other_stride_patterns_get_one_copy():
    g = torch.Generator().manual_seed(3)
    K = 20
    scores = torch.randn(2, 8, 8, K, generator=g).to(DEV).permute(0, 3, 2, 1)   # [N,K,W,H] storage, viewed [N,K,H,W]
    t = torch.randint(0, K, (2, 8, 8), generator=g)
    assert torch.equal(counts_of(scores, t.to(DEV), K), oracle(torch.argmax(scores.cpu(), 1), t, K))


def _onehot_at_half_pixel(K, dtype, N=2, H=48, W=80, seed=5):
    """One-hot layouts warped by exactly half a pixel: every pixel on a class border is an exact 0.5 / 0.5 tie."""
    g = torch.Generator().manual_seed(seed)
    lab = torch.randint(0, K, (N, H // 4, W // 4), generator=g).repeat_interleave(4, 1).repeat_interleave(4, 2)
    onehot = torch.zeros(N, K, H, W).scatter_(1, lab[:, None], 1.0).to(dtype)
    flow = torch.zeros(N, H, W, 2)
    flow[..., 0] = 0.5
    rgb = torch.randn(N, 3, H, W, generator=g).to(dtype)
    tgt = sprinkle_ignore(torch.randint(0, K, (N, H, W), generator=g), -100, g)
    cl = lambda x: x.to(DEV).contiguous(memory_format=torch.channels_last)
    return cl(rgb), cl(onehot), flow.to(DEV), cl(torch.randn(N, 3, H, W, generator=g).to(dtype)), tgt.to(DEV)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("K", [20, 19])
def test_ties_agree_with_warp_and_the_fused_ops_argmax(dtype, K):
    rgb, onehot, flow, tgt_rgb, tgt = _onehot_at_half_pixel(K, dtype)
    _, warped, arg_warp = vlg_b200.warp(rgb, onehot, flow)
    ties = (warped.float() == warped.float().amax(1, keepdim=True)).sum(1) > 1
    assert int(ties.sum()) > 100, "the fixture must contain exact ties"
    _, _, arg_fused = vlg_b200.warp_loss(rgb, onehot, flow, tgt_rgb, tgt, vlg_b200.WarpLossConfig(want_argmax=True))
    want = oracle(torch.argmax(warped.cpu().float(), 1), tgt, K)
    for nchw in (False, True):
        assert torch.equal(counts_of(as_layout(warped, nchw), tgt, K), want)
    assert torch.equal(counts_of(arg_warp, tgt, K), want)
    # the fused op takes its argmax on the fp32 warped values; warp() on the values as stored, and rounding to bf16 turns
    # near-ties (a sampling position a few ulp off the half pixel) into exact ones -- only fp32 stores what it compares
    want_fused = want if dtype == torch.float32 else oracle(arg_fused, tgt, K)
    assert torch.equal(counts_of(arg_fused, tgt, K), want_fused)


# ---------------------------------------------------------------- accumulation, rollout, skipped pixels, capture
def test_two_updates_equal_the_sum():
    g = torch.Generator().manual_seed(11)
    K = 20
    a, b = (torch.randint(0, K, (3, 40, 64), generator=g).to(DEV) for _ in range(2))
    t1, t2 = (sprinkle_ignore(torch.randint(0, K, (3, 40, 64), generator=g), -100, g).to(DEV) for _ in range(2))
    m = vlg_b200.LayoutIoU(n_classes=K)
    m.update(a, t1)
    m.update(b, t2)
    assert torch.equal(m.counts[0].cpu(), oracle(a, t1, K) + oracle(b, t2, K))
    m.reset()
    assert int(m.counts.abs().sum()) == 0


def test_rollout_rows_are_independent():
    K, steps, N, H, W = 20, 5, 2, 64, 96
    g = torch.Generator().manual_seed(13)
    img = torch.randn(N, 3, H, W, generator=g).to(DEV).contiguous(memory_format=torch.channels_last)
    lab = torch.randint(0, K, (N, H // 8, W // 8), generator=g).repeat_interleave(8, 1).repeat_interleave(8, 2).to(DEV)
    flows = [(torch.randn(N, H, W, 2, generator=g) * 2).to(DEV) for _ in range(steps)]
    gt = [sprinkle_ignore(torch.randint(0, K, (N, H, W), generator=g), -100, g).to(DEV) for _ in range(steps)]
    _, labels = vlg_b200.rollout(img, lab, lambda t, i, l: flows[t], steps=steps)
    m = vlg_b200.LayoutIoU(n_classes=K, steps=steps)
    for t, pred in enumerate(labels):
        m.update(pred, gt[t], step=t)
    for t in range(steps):
        sep = vlg_b200.confusion_matrix(labels[t], gt[t], K).cpu().reshape(-1)
        assert torch.equal(m.counts[t, :K * K].cpu(), sep)
        assert torch.equal(m.counts[t].cpu(), oracle(labels[t], gt[t], K))
    r = m.compute()
    assert r.miou.shape == (steps,) and bool(torch.isfinite(r.pixel_acc).all())


@pytest.mark.parametrize("ignore", [-100, 255])
def test_out_of_range_labels_land_in_the_skipped_slot_only(ignore):
    K = 19
    g = torch.Generator().manual_seed(17)
    t = sprinkle_ignore(torch.randint(0, K, (2, 33, 47), generator=g), ignore, g)
    p = torch.randint(0, K, (2, 33, 47), generator=g)
    bad_t = torch.rand(t.shape, generator=g) < 0.03
    bad_p = torch.rand(t.shape, generator=g) < 0.03
    t[bad_t] = torch.tensor([K, -1, 1000, -101])[torch.randint(0, 4, (int(bad_t.sum()),), generator=g)]
    p[bad_p] = torch.tensor([K, -1, 2 ** 40])[torch.randint(0, 3, (int(bad_p.sum()),), generator=g)]
    want = oracle(p, t, K, ignore)
    assert int(want[K * K]) > 0
    pd, td = p.to(DEV), t.to(DEV)
    assert torch.equal(counts_of(pd, td, K, ignore), want)
    assert torch.equal(counts_of(offset_by_one(pd), offset_by_one(td), K, ignore), want)
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        vlg_b200.confusion_matrix(pd, td, K, ignore_index=ignore, debug=True)
    m = vlg_b200.LayoutIoU(n_classes=K, ignore_index=ignore)
    m.update(pd, td)
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        m.compute()


def test_debug_passes_on_clean_input():
    K = 5
    t = torch.randint(0, K, (2, 8, 8)).to(DEV)
    cm = vlg_b200.confusion_matrix(t, t, K, debug=True)
    assert torch.equal(cm.cpu(), torch.diag(torch.bincount(t.cpu().reshape(-1), minlength=K)))


def test_shape_and_dtype_checks():
    K = 20
    t = torch.zeros(2, 8, 8, dtype=torch.int64, device=DEV)
    with pytest.raises(vlg_b200.VlgError, match="shape"):
        vlg_b200.confusion_matrix(torch.zeros(2, 8, 9, dtype=torch.int64, device=DEV), t, K)
    with pytest.raises(vlg_b200.VlgError, match="shape"):
        vlg_b200.confusion_matrix(torch.zeros(2, 19, 8, 8, device=DEV), t, K)
    with pytest.raises(vlg_b200.VlgError, match="int64"):
        vlg_b200.confusion_matrix(t, t.int(), K)
    with pytest.raises(vlg_b200.VlgError, match="dtype"):
        vlg_b200.confusion_matrix(torch.zeros(2, K, 8, 8, dtype=torch.float16, device=DEV), t, K)


@pytest.mark.parametrize("scores", [False, True], ids=["labels", "scores_nchw"])
def test_update_inside_captured_step(scores):
    K, reps = 20, 4
    g = torch.Generator().manual_seed(19)
    t = sprinkle_ignore(torch.randint(0, K, (4, 64, 128), generator=g), -100, g).to(DEV)
    pred = torch.randn(4, K, 64, 128, generator=g).to(DEV) if scores else torch.randint(0, K, (4, 64, 128), generator=g).to(DEV)
    eager = vlg_b200.confusion_matrix(pred, t, K).cpu()
    m = vlg_b200.LayoutIoU(n_classes=K)
    step = vlg_b200.CapturedStep(lambda: m.update(pred, t))
    m.reset()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    assert torch.equal(m.counts[0, :K * K].cpu().view(K, K), eager * reps)
    assert int(m.counts[0, K * K]) == 0
