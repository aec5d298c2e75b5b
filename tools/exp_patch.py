"""Runs the bottleneck conv2 shapes through sm_conv2d (exact mode) on the resident-patch kernel.  Used under ncu for
the source-level stall picture."""
import sys, torch
sys.path.insert(0, '.')
import siammask_b200 as smb
dev = 'cuda'
for (B, C, H) in [(64, 64, 63), (64, 128, 31)]:
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, C, H, H, generator=g).to(dev)
    w = (torch.randn(C, C, 3, 3, generator=g) * (2.0 / (C * 9)) ** 0.5)
    sc, sh = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    for _ in range(3):
        out = smb.conv2d(x, w, sc, sh, 1, 1, 1, relu=True)
    torch.cuda.synchronize()
    print(f"B={B} C={C} H={H} ok {tuple(out.shape)}", flush=True)
