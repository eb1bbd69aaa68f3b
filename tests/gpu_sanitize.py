"""Small workloads for compute-sanitizer (memcheck / racecheck / synccheck), not a pytest file:

    compute-sanitizer --tool memcheck  python tests/gpu_sanitize.py
    compute-sanitizer --tool racecheck python tests/gpu_sanitize.py
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402
from oracle import focal_stack_oracle as orc  # noqa: E402

lens = aadff_b200.PSFNet(kernel_size=11, device="cuda")
lens.load_net(os.path.join(ROOT, "tests/golden/rf50mm_PSFNet480x640_ks11.pkl"))
img, dm = orc.synthetic_rgbd(1, 24, 40, seed=1)
foc = -orc.synthetic_focus(dm, 2).cuda() * 1e3
img, dep = img.cuda(), -dm.cuda() * 1e3
for mode in ("parity", "econ", "mixed", "fast", "fp32"):
    out = lens.render_stack(img, dep, foc, mode=mode)
    torch.cuda.synchronize()
    print(mode, float(out.mean()))
print("pred", float(lens.pred(torch.rand(200, 4).cuda(), mode="parity").sum()))
psf = torch.rand(1, 24, 40, 11, 11, device="cuda")
print("gather", float(aadff_b200.local_psf_render(img, psf, 11).mean()))
img5 = torch.rand(2, 5, 19, 45, device="cuda")                   # ragged: partial groups / tiles, 3 + 1 + 1 channel passes
for ks in (3, 7, 31):
    psf = torch.rand(2, 19, 45, ks, ks, device="cuda")
    print("gather ragged ks", ks, float(aadff_b200.local_psf_render(img5, psf, ks).mean()))
tl = aadff_b200.ThinLens(50.0, 1.8, 11, [36.0, 24.0], (24, 40)).to("cuda")
print("thinlens", float(tl.render(img, dep, foc[:, 0]).mean()))
# ---- round 2: tile-row ranges, PSF-map convolution, device-side sign flag, fitting step
rows = lens.render_stack_rows(img, dep, foc, 1, 5, mode="parity")
print("rows", tuple(rows.shape), float(rows.mean()))
rows = lens.render_stack_rows(img, dep, foc, 0, 6, mode="fp32")
print("rows fp32", tuple(rows.shape), float(rows.mean()))
from deeplens.render_psf import render_psf, render_psf_map  # noqa: E402
print("render_psf", float(render_psf(img5, torch.rand(5, 7, 7, device="cuda")).mean()))
print("render_psf_map", float(render_psf_map(torch.rand(1, 3, 37, 41, device="cuda"), torch.rand(3, 15, 15, device="cuda"), 5).mean()))
print("thinlens +depth", float(tl.render(img, -dep.clamp(max=-300.0), -foc[:, 0]).mean()))
import torch.nn as nn  # noqa: E402
lin = [m for m in lens.psfnet.net if isinstance(m, nn.Linear)]
tr = aadff_b200.native.NativeTrainer([l.weight.detach().cpu().numpy() for l in lin], [l.bias.detach().cpu().numpy() for l in lin], 48, 0)
x, t = torch.rand(48, 4, device="cuda"), torch.rand(48, 121, device="cuda")
loss = torch.zeros(1, device="cuda")
for _ in range(2):
    aadff_b200.native.check(aadff_b200.native.lib.aadff_trainer_step(tr.handle, x.data_ptr(), t.data_ptr(), 1e-4, loss.data_ptr(), None))
torch.cuda.synchronize()
print("trainer loss", float(loss))
tr.close()
# ---- thin lens with TMA tensor-tile halo (interior tiles) and the cp.async border path, large kernel (single buffer), preparation
tl2 = aadff_b200.ThinLens(50.0, 1.8, 11, [36.0, 24.0], (72, 200)).to("cuda")
im2 = torch.rand(2, 3, 72, 200, device="cuda")
dp2 = 300 + 6000 * torch.rand(2, 1, 72, 200, device="cuda")
print("thinlens TMA", float(tl2.render(im2, dp2, torch.tensor([1500.0, 2500.0], device="cuda")).mean()))
tl3 = aadff_b200.ThinLens(50.0, 1.8, 31, [36.0, 24.0], (96, 160)).to("cuda")
print("thinlens k31", float(tl3.render(torch.rand(1, 4, 96, 160, device="cuda"), 300 + 6000 * torch.rand(1, 1, 96, 160, device="cuda"),
                                       torch.tensor([1500.0], device="cuda")).mean()))
bgr = torch.randint(0, 255, (2, 96, 130, 3), dtype=torch.uint8, device="cuda")
d16 = torch.randint(0, 8000, (2, 96, 130), dtype=torch.int16, device="cuda").view(torch.uint16)
a, d = aadff_b200.preprocess_rgbd(bgr, d16, (40, 56), jitter=torch.tensor([[0.5, 0.1], [-1.0, 0.0]]), flips=torch.tensor([3, 0], dtype=torch.uint8))
print("preprocess", float(a.mean()), float(d.mean()))
# ---- round 2, second half: strip-walking gather (every plan; W % 4 == 0, partial strips, runs crossing strips and
# images), two-pixel thin-lens kernel on odd widths, AutoAgument's spline rotation
for ks, (n_, h_, w_) in ((11, (2, 19, 68)), (7, (3, 9, 332)), (3, (1, 5, 4)), (13, (1, 33, 132)), (15, (1, 20, 64))):
    im = torch.rand(n_, 3, h_, w_, device="cuda")
    pf = torch.rand(n_, h_, w_, ks, ks, device="cuda")
    for flags in (0, 8192, 1024, 4096):
        aadff_b200.native.lib.aadff_debug_set_flags(flags)
        v = float(aadff_b200.local_psf_render(im, pf, ks).mean())
        aadff_b200.native.lib.aadff_debug_set_flags(0)
    print("strip gather ks", ks, (n_, h_, w_), v)
tl4 = aadff_b200.ThinLens(50.0, 1.8, 7, [36.0, 24.0], (33, 67)).to("cuda")
print("thinlens two-pixel odd W", float(tl4.render(torch.rand(1, 5, 33, 67, device="cuda"), 300 + 6000 * torch.rand(1, 1, 33, 67, device="cuda"),
                                                   torch.tensor([1500.0], device="cuda")).mean()))
a, d = aadff_b200.preprocess_rgbd(bgr, d16, (40, 56), jitter=torch.tensor([[0.5, 0.1], [-1.0, 0.0]]), flips=torch.tensor([3, 0], dtype=torch.uint8),
                                  rotate_deg=[33.0, None])
print("preprocess + rotation", float(a.mean()), float(d.mean()))
a, d = aadff_b200.preprocess_rgbd(bgr[:, :5, :23].contiguous(), d16[:, :5, :23].contiguous(), (5, 23), rotate_deg=[90.0, 171.0])
print("rotation of a 5 x 23 image", float(a.mean()), float(d.mean()))
