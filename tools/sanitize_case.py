"""Small end-to-end case for compute-sanitizer (one tool per gpurun call):
    compute-sanitizer --tool memcheck python tools/sanitize_case.py
Covers pass 1 (staged + global fallback), pass 2 near + far paths, pixel-loss mode, forward warps."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vlg_b200

dev = "cuda"
torch.manual_seed(0)
for (N, H, W, sigma, far) in ((1, 37, 70, 1.5, 0.0), (2, 24, 45, 6.0, 0.05)):
    K = 20
    cl = lambda t: t.to(dev).contiguous(memory_format=torch.channels_last)
    a = cl(torch.randn(N, 3, H, W)).requires_grad_(True)
    b = cl(torch.randn(N, K, H, W)).requires_grad_(True)
    f = torch.randn(N, H, W, 2) * sigma
    if far:
        m = torch.rand(N, H, W, 1) < far
        f = torch.where(m, (torch.rand(N, H, W, 2) - 0.5) * 2 * W, f)
    f = f.to(dev).requires_grad_(True)
    t = cl(torch.randn(N, 3, H, W))
    lab = torch.randint(0, K, (N, H, W), device=dev)
    for pad in ("border", "zeros"):
        total, vec, arg = vlg_b200.warp_loss(a, b, f, t, lab, vlg_b200.WarpLossConfig(w_tv=0.5, padding_mode=pad, want_argmax=True))
        total.backward()
        vlg_b200.warp(a.detach(), b.detach(), f.detach(), padding_mode=pad)
        vlg_b200.warp_labels(a.detach(), lab, f.detach(), padding_mode=pad)
    img = cl(torch.randn(N, 3, H, W)).requires_grad_(True)
    seg = cl(torch.randn(N, K, H, W)).requires_grad_(True)
    vlg_b200.PixelLosses()(img, t, seg, lab).backward()
    fr = torch.rand(N, 3, H, W, device=dev)
    vlg_b200.prepare_frames(fr, flip=True, labels=lab)
    vlg_b200.prepare_frames(cl(fr.cpu()), denormalize=True, dtype=torch.bfloat16)
    # bf16 layouts (8-byte-unit TMA map when W is even; pass1_kernel + tap_records_kernel for W = 45), pass 2 from
    # coordinates, the layout terms in pass1_kernel (cp.async staging)
    a16, b16 = a.detach().to(torch.bfloat16).requires_grad_(True), b.detach().to(torch.bfloat16).requires_grad_(True)
    total, _, _ = vlg_b200.warp_loss(a16, b16, f, t.to(torch.bfloat16), lab, vlg_b200.WarpLossConfig(w_tv=0.5))
    total.backward()
    for kw in (dict(pass2_records=False), dict(use_tma=False)):
        total, _, _ = vlg_b200.warp_loss(a, b, f, t, lab, vlg_b200.WarpLossConfig(w_tv=0.5, **kw))
        total.backward()
    # label-source op and uint8 ingest
    total, _, _ = vlg_b200.warp_loss(a.detach(), lab, f, t, lab, vlg_b200.WarpLossConfig(w_tv=0.5, want_argmax=True))
    total.backward()
    u8 = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, device=dev)
    s8 = torch.randint(0, K, (N, H, W), dtype=torch.uint8, device=dev)
    vlg_b200.ingest(u8, s8, flip=True, n_classes=K, want_label=True, want_seg_float=True, want_one_hot=True)
    vlg_b200.ingest(u8, s8, n_classes=K, dtype=torch.bfloat16, want_one_hot=True)
torch.cuda.synchronize()
print("sanitize case done", float(total))
