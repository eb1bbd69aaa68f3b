"""GPU parity tests (pytest -m gpu): the CUDA path, called the way the reference's scripts call
it (deeplens.psfnet.PSFNet / deeplens.render_psf.local_psf_render -> C ABI -> sm_100a kernels),
against (1) golden vectors produced by the reference itself, (2) the CPU oracle on seeded inputs,
(3) size-independent properties at BASELINE.json's full sizes.

Tolerances (max-abs on [0,1] images, fp32):
  parity mode (tcgen05, fp16 hi/lo split, 3 terms)   1e-4   -- north_star's bar; observed <= 1e-5, tested at 2e-5
  fp32 mode   (CUDA cores)                           5e-6
  mixed mode                                         1e-3
  fast mode   (single fp16 term)                     2e-2 max, 1e-4 mean  (stated tolerance of that mode; observed <= 1.4e-2 on noise images / 6e-5 mean)
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, analytic_rgbd, load_golden
from oracle import focal_stack_oracle as orc
from oracle import tc_arith_oracle as tao

pytestmark = pytest.mark.gpu

# north_star bar: 1e-4.  parity is tested at 2e-5 (observed <= 1e-5) and econ at 6e-5 (observed <= 3.4e-5 with the
# calibrated fp16 weights; plain rounding gave 6e-5 .. 9e-5) so that a regression shows before the bar is reached.
TOL = {"parity": 2e-5, "econ": 6e-5, "econ8": 4e-5, "fp32": 5e-6, "mixed": 1e-3, "fast": 2e-2}
CKPT = os.path.join(GOLDEN, "rf50mm_PSFNet480x640_ks11.pkl")
BASELINE_TOL = {"parity": 2e-5, "econ": 6e-5, "econ8": 4e-5, "fp32": 5e-6, "fast": 2e-2}        # fast: + mean-abs < 1e-4


def _report(tag, mode, err):
    print(f"[parity-at-size] {tag:28s} mode={mode:7s} max-abs vs reference = {err:.3e}")




def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


@pytest.fixture(scope="module")
def lens(pkg):
    from deeplens.psfnet import PSFNet          # the reference's import line
    l = PSFNet(filename='./lenses/rf50mm/lens.json', sensor_res=(480, 640), kernel_size=11)
    l.load_net(CKPT)
    l.analysis()
    return l


@pytest.fixture(scope="module")
def lens31(pkg):
    g = load_golden("kat_g_ks31_1x40x48.npz")
    Ws, bs = orc.seeded_psfnet_weights(31, seed=int(g["weight_seed"]))
    gen = torch.Generator().manual_seed(int(g["bias_seed"]))
    bs = [(torch.rand(b.shape, generator=gen) - 0.5) * 0.2 for b in bs]
    l = pkg.PSFNet(kernel_size=31, device="cuda")
    sd = {}
    for i, (W, b) in enumerate(zip(Ws, bs)):
        sd[f"net.{2 * i}.weight"], sd[f"net.{2 * i}.bias"] = W, b
    l.psfnet.load_state_dict(sd)
    return l


def maxabs(a, b):
    return float((a.detach().cpu().float() - b.detach().cpu().float()).abs().max())


# --------------------------------------------------------------------------- tensor-core plumbing
@pytest.mark.parametrize("K,N", [(32, 16), (64, 256), (256, 256), (256, 128), (256, 208)])
def test_umma_gemm_matches_fp16_product(pkg, K, N):
    """tcgen05.mma through the fused kernel's operand packing/descriptors/TMEM read-back."""
    rng = np.random.default_rng(K * 1000 + N)
    A = rng.standard_normal((128, K)).astype(np.float32)
    B = rng.standard_normal((N, K)).astype(np.float32)
    D = np.zeros((128, N), np.float32)
    pkg.native.check(pkg.native.lib.aadff_debug_umma_gemm(A.ctypes.data, B.ctypes.data, D.ctypes.data, K, N, 0))
    ref = A.astype(np.float16).astype(np.float64) @ B.astype(np.float16).astype(np.float64).T
    assert np.abs(D - ref).max() < 2e-4


# --------------------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("i", [0, 1, 2, 3, 4, "3d"])
def test_gather_golden(pkg, i):
    from deeplens.render_psf import local_psf_render
    g = load_golden(f"kat_d_gather_{i}.npz")
    out = local_psf_render(T(g["img"]).cuda(), T(g["psf"]).cuda(), int(g["ks"]))
    assert out.shape == g["out"].shape
    assert maxabs(out, T(g["out"])) < 5e-5 * int(g["ks"])


@pytest.mark.parametrize("ks", list(range(1, 35, 2)))
def test_gather_every_kernel_size_vs_oracle(pkg, ks):
    """Register-streaming gather (gather_coalesced_kernel.cuh): every odd ks in 3..31, ragged W/H (partial groups,
    partial tiles, rows beyond H), C = 1..5 (3-channel and 1-channel passes), against the oracle's direct definition.
    ks = 1 and 33 run the generic kernel (gather_kernel.cuh), with W % 4 == 0 and W % 4 != 0."""
    from deeplens.render_psf import local_psf_render
    gen = torch.Generator().manual_seed(100 + ks)
    for (N, C, H, W) in [(2, 3, 19, 45), (1, 5, 33, 36), (1, 1, 5, 7), (1, 2, 16, 64)]:
        img = torch.rand(N, C, H, W, generator=gen)
        psf = torch.rand(N, H, W, ks, ks, generator=gen)
        psf = psf / psf.sum((-1, -2), keepdim=True)
        ref = orc.local_psf_render(img, psf, ks)
        out = local_psf_render(img.cuda(), psf.cuda(), ks)
        assert out.shape == ref.shape
        assert maxabs(out, ref) < 2e-6, (ks, N, C, H, W)


@pytest.mark.parametrize("ks", [3, 5, 7, 9, 11, 13, 15, 17])
def test_gather_strip_kernel_vs_oracle_and_register_streaming(pkg, ks):
    """Strip-walking gather (gather_strip_kernel.cuh; taken when W % 4 == 0 and ks <= 15; ks = 17 exercises the fall-through): partial strips (W = 68, 132,
    200), a strip narrower than one lane pair (W = 4), images shorter than the kernel (H = 3), several images / strips
    per warp run, C = 1 / 3 / 4, the automatic plan and all three shared-memory plans forced (debug flags 8192 / 1024 / 4096: strips of 64 - 256
    columns taken in 64-column passes, deeper rings), against the oracle's direct definition and against the register-streaming
    kernel (debug flag 512)."""
    from deeplens.render_psf import local_psf_render
    gen = torch.Generator().manual_seed(300 + ks)
    for (N, C, H, W) in [(2, 3, 19, 68), (1, 4, 33, 132), (1, 1, 3, 4), (1, 3, 70, 64), (3, 3, 9, 200), (1, 3, 12, 332)]:
        img = torch.rand(N, C, H, W, generator=gen)
        psf = torch.rand(N, H, W, ks, ks, generator=gen)
        psf = psf / psf.sum((-1, -2), keepdim=True)
        ref = orc.local_psf_render(img, psf, ks)
        for flags in (0, 8192, 1024, 4096, 512):
            pkg.native.lib.aadff_debug_set_flags(flags)
            try:
                out = local_psf_render(img.cuda(), psf.cuda(), ks)
            finally:
                pkg.native.lib.aadff_debug_set_flags(0)
            assert out.shape == ref.shape
            assert maxabs(out, ref) < 2e-6, (ks, flags, N, C, H, W)
    # a launch that gives every warp of every SM a run crossing strip and image boundaries
    img = torch.rand(5, 3, 96, 320, generator=gen).cuda()
    psf = torch.rand(5, 96, 320, ks, ks, generator=gen).cuda()
    psf = psf / psf.sum((-1, -2), keepdim=True)
    new = local_psf_render(img, psf, ks)
    pkg.native.lib.aadff_debug_set_flags(512)
    try:
        old = local_psf_render(img, psf, ks)
    finally:
        pkg.native.lib.aadff_debug_set_flags(0)
    assert maxabs(new, old) < 2e-6, ks


@pytest.mark.parametrize("hidden_layers", [0, 2, 5])
def test_other_network_depths_vs_oracle(pkg, hidden_layers):
    """The C ABI takes any number of 256-wide hidden layers: shallower / deeper MLPs than the reference's
    MLP(4, k^2, 256, 8) exercise the other group counts of the kernel specialisations (all-three-term, econ and mixed
    patterns with fewer groups, the ring alignment check) against the CPU oracle."""
    from deeplens.psfnet_arch import MLP
    ks = 11
    l = pkg.PSFNet(kernel_size=ks, device="cuda")
    torch.manual_seed(40 + hidden_layers)
    l.psfnet = MLP(in_features=4, out_features=ks * ks, hidden_features=256, hidden_layers=hidden_layers).to("cuda")
    l.psfnet._evaluator = l._mlp_eval
    l._native = None
    gen = torch.Generator().manual_seed(7 + hidden_layers)
    with torch.no_grad():
        for lin in l.psfnet.linear_layers():
            lin.bias.copy_(((torch.rand(lin.bias.shape, generator=gen) - 0.5) * 0.2).cuda())
    Ws = [lin.weight.detach().cpu() for lin in l.psfnet.linear_layers()]
    bs = [lin.bias.detach().cpu() for lin in l.psfnet.linear_layers()]
    img, dm = orc.synthetic_rgbd(2, 24, 40, seed=3)
    foc = -orc.synthetic_focus(dm, 3) * 1e3
    ref = orc.render_stack(Ws, bs, img, -dm * 1e3, foc, ks)
    for mode in ("parity", "fp32", "fast", "econ", "econ8", "mixed"):
        out = l.render_stack(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode=mode)
        tol = TOL[mode]
        if mode in ("econ", "econ8"):
            # a net with fewer layer groups than the mode's first reduced group runs the parity pattern (launch_tc)
            reduced = 2 in tao.term_pattern(mode, hidden_layers, len(tao.head_blocks(ks)))
            tol = 1e-4 if reduced else TOL["parity"]
        assert maxabs(out, ref) < tol, (hidden_layers, mode)


def test_pred_golden(lens):
    g = load_golden("kat_a_pred.npz")
    psf = lens.pred(T(g["inp"]).cuda())
    assert psf.shape == (64, 11, 11)
    assert maxabs(psf, T(g["psf"])) < 1e-6
    assert abs(float(psf[1, 5, 5]) - 0.810939252) < 1e-6          # SURVEY.md 8c literal
    for mode, tol in (("parity", 1e-5), ("econ", 1e-4), ("fast", 5e-2)):   # tensor-core pred (PSF values, not images)
        tc = lens.pred(T(g["inp"]).cuda(), mode=mode)
        assert tc.shape == (64, 11, 11) and maxabs(tc, T(g["psf"])) < tol, mode
        assert float((tc.sum((-1, -2)) - 1).abs().max()) < 1e-5
    big = torch.rand(1000, 4, generator=torch.Generator().manual_seed(3))
    big[:, :2] = big[:, :2] * 2 - 1
    assert maxabs(lens.pred(big.cuda(), mode="parity"), lens.pred(big.cuda())) < 1e-5      # ragged M (not % 128)
    grid = lens.pred(T(g["inp"]).cuda().reshape(8, 8, 4))           # [H,W,4] -> [H,W,ks,ks]
    assert grid.shape == (8, 8, 11, 11) and maxabs(grid.reshape(64, 11, 11), psf) == 0.0


@pytest.mark.parametrize("mode", ["parity", "econ", "fp32", "mixed", "fast"])
@pytest.mark.parametrize("N,H,W", [(1, 48, 64), (2, 64, 64)])
def test_render_kat_b(lens, mode, N, H, W):
    g = load_golden(f"kat_b_{N}x{H}x{W}.npz")
    img, dm = analytic_rgbd(N, H, W)
    out = lens.render(img.cuda(), -dm.cuda() * 1e3, T(g["foc"]).cuda(), mode=mode)
    assert out.shape == (N, 3, H, W) and out.dtype == torch.float32 and out.is_cuda
    assert maxabs(out, T(g["out"])) < TOL[mode]


@pytest.mark.parametrize("mode", ["parity", "fp32"])
def test_render_kat_b_full_frame(lens, mode):
    """0_warm_up.py's shape (BASELINE config c1): 1 x 480 x 640, foc -2400 mm."""
    g = load_golden("kat_b_1x480x640.npz")
    img, dm = analytic_rgbd(1, 480, 640)
    out = lens.render(img.cuda(), -dm.cuda() * 1e3, T(g["foc"]).cuda(), mode=mode).cpu()
    assert (out[:, :, ::8, ::8] - T(g["out_sub"])).abs().max() < TOL[mode]
    assert (out[:, :, [0, 1, 239, 240, 478, 479], :] - T(g["out_rows"])).abs().max() < TOL[mode]
    assert abs(float(out.double().sum()) - float(g["sum"])) < 1.0


@pytest.mark.parametrize("mode", ["parity", "econ", "fp32"])
def test_warm_up_script_body_vs_reference_cpu_output(pkg, mode):
    """The body of 0_warm_up.py (lines 9-22, BASELINE config c1) through the shadow package, on the resolution chart
    + the real Adirondack depth map, against what the reference itself produced on the CPU
    (tests/golden/make_golden_warmup.py).  885 pixels of that depth map are invalid (0) -> z clamps."""
    from deeplens.psfnet import PSFNet                                    # 0_warm_up.py:3
    g = load_golden("kat_k_warmup_c1.npz")
    psfnet = PSFNet(filename='./lenses/rf50mm/lens.json', sensor_res=(480, 640), kernel_size=11, mode=mode)
    psfnet.load_net(CKPT)
    psfnet.analysis()
    img = torch.tensor(g["img_u8"]).permute(2, 0, 1).unsqueeze(0).float() / 255
    depth = torch.tensor(g["depth_m"]).unsqueeze(0).unsqueeze(0).float()
    depth = - depth * 1e3
    focus_dist = torch.tensor([-2400.])
    out = psfnet.render(img.to(psfnet.device), depth.to(psfnet.device), focus_dist.to(psfnet.device)).cpu()
    err = max(float((out[..., ::3, ::3] - T(g["out_sub"])).abs().max()),
              float((out[..., [0, 240, 479], :] - T(g["out_rows"])).abs().max()))
    _report("c1 0_warm_up.py body", mode, err)
    assert out.shape == (1, 3, 480, 640) and err < BASELINE_TOL[mode]
    assert abs(float(out.double().sum()) - float(g["sum"])) < 921600 * 1e-6


def test_econ_calibration_beats_plain_rounding(pkg, lens):
    """econ mode (2 terms for L5.. and the head) on a noise image at BASELINE c2 size, against the fp32 CUDA-core kernel:
    the calibrated weights (csrc/econ_calib.h) stay under 6e-5; plain fp16 rounding (debug flag 256) is >1.5x worse."""
    gen = torch.Generator().manual_seed(5)
    img = torch.rand(1, 3, 512, 512, generator=gen).cuda()
    _, dm = orc.synthetic_rgbd(1, 512, 512, seed=77)
    dep, foc = -dm.cuda() * 1e3, -orc.synthetic_focus(dm, 5).cuda() * 1e3
    ref = lens.render_stack(img, dep, foc, mode="fp32")
    cal = maxabs(lens.render_stack(img, dep, foc, mode="econ"), ref)
    pkg.native.lib.aadff_debug_set_flags(256)
    try:
        plain = maxabs(lens.render_stack(img, dep, foc, mode="econ"), ref)
    finally:
        pkg.native.lib.aadff_debug_set_flags(0)
    assert cal < 6e-5 and plain > 1.5 * cal, (cal, plain)
    assert maxabs(lens.render_stack(img, dep, foc, mode="parity"), ref) < 2e-5


@pytest.mark.parametrize("mode", ["parity", "fp32"])
def test_render_kat_c_depth_clamps(lens, mode):
    g = load_golden("kat_c_clamp.npz")
    img, dm = analytic_rgbd(1, 32, 32)
    dm[:, :, :8] = 0.0
    dm[:, :, 8:16] = 30.0
    out = lens.render(img.cuda(), -dm.cuda() * 1e3, T(g["foc"]).cuda(), mode=mode)
    assert maxabs(out, T(g["out"])) < TOL[mode]


@pytest.mark.parametrize("mode", ["parity", "econ", "fp32", "fast"])
def test_stack_golden_ragged(lens, mode):
    """2 x 40 x 56 (not a multiple of the 8x16 tile), S=5, focus from select_focus_dist."""
    from dff.utils import select_focus_dist
    g = load_golden("kat_e_stack_2x40x56.npz")
    img, dm = T(g["img"]).cuda(), T(g["depth_m"]).cuda()
    foc_m = select_focus_dist(dm, 5)
    assert torch.equal(foc_m.cpu(), T(g["foc_m"]))
    out = lens.render_stack(img, -dm * 1e3, -foc_m * 1e3, mode=mode)
    assert out.shape == (2, 3, 5, 40, 56)
    d = (out.cpu() - T(g["out"])).abs()
    assert float(d.max()) < TOL[mode]
    if mode == "fast":
        assert float(d.mean()) < 1e-4
    # the reference's own loop: one render per slice, stacked on dim 2 -- bit-identical
    loop = torch.stack([lens.render(img, -dm * 1e3, -foc_m[:, s] * 1e3, mode=mode) for s in range(5)], dim=2)
    assert torch.equal(loop, out)
    # DFVNet layout
    assert torch.equal(lens.render_stack(img, -dm * 1e3, -foc_m * 1e3, layout="BSCHW", mode=mode),
                       out.permute(0, 2, 1, 3, 4))


def test_render_3d_branch(lens):
    g = load_golden("kat_e_render3d.npz")
    out = lens.render(T(g["img"]).cuda(), -T(g["depth_m"]).cuda() * 1e3, float(g["foc"]))
    assert out.shape == (1, 3, 40, 56)
    assert maxabs(out, T(g["out"])) < TOL["parity"]
    with pytest.raises(ValueError):
        lens.render(torch.rand(4, 4).cuda(), torch.rand(4, 4).cuda(), -1000.0)


@pytest.mark.parametrize("mode", ["parity", "fp32", "fast", "econ", "mixed"])
def test_ks31_golden(lens31, mode):
    g = load_golden("kat_g_ks31_1x40x48.npz")
    out = lens31.render(T(g["img"]).cuda(), -T(g["depth_m"]).cuda() * 1e3, T(g["foc"]).cuda(), mode=mode)
    assert maxabs(out, T(g["out"])) < (1e-4 if mode == "econ" else TOL[mode])       # seeded random weights: north_star's bar
    probe = lens31.pred(torch.tensor([[0.1, -0.2, 0.3, 0.4]]).cuda())
    assert maxabs(probe, T(g["psf_probe"])) < 1e-6


def test_thinlens_and_focus_golden(pkg):
    from deeplens.psfnet import ThinLens
    from dff.utils import select_focus_dist
    g = load_golden("kat_h_thinlens.npz")
    tl = ThinLens(foc_len=float(g["foc_len"]), fnum=float(g["fnum"]), kernel_size=11,
                  sensor_size=[float(v) for v in g["sensor_size"]], sensor_res=(40, 56)).to("cuda")
    out = tl.render(T(g["img"]).cuda(), -T(g["depth_m"]).cuda() * 1e3, T(g["foc"]).cuda())      # fused kernel
    assert maxabs(out, T(g["out"])) < 5e-6
    # the reference's two-step formulation (materialised PSFs + gather kernel) agrees with the fused kernel
    from deeplens.render_psf import local_psf_render
    psf = tl.psf(-T(g["depth_m"]).cuda() * 1e3, T(g["foc"]).cuda())
    assert maxabs(local_psf_render(T(g["img"]).cuda(), psf, 11), T(g["out"])) < 5e-6
    # positive-depth convention (no sign flip), odd sizes, 1 and 5 channels
    gen = torch.Generator().manual_seed(5)
    for (N, C, H, W) in [(1, 1, 9, 13), (2, 5, 17, 40)]:
        img = torch.rand(N, C, H, W, generator=gen)
        dep = 300 + 6000 * torch.rand(N, 1, H, W, generator=gen)
        foc = 500 + 3000 * torch.rand(N, generator=gen)
        ref = orc.thinlens_render(img, dep, foc, 11, float(g["foc_len"]), float(g["fnum"]), tl.ps)
        assert maxabs(tl.render(img.cuda(), dep.cuda(), foc.cuda()), ref) < 5e-6
    g = load_golden("kat_f_select_focus.npz")
    # the CUDA kernel keeps the reference's arithmetic order with IEEE division: bit-exact vs the CPU golden
    assert torch.equal(select_focus_dist(T(g["depth_m"]).cuda(), 5).cpu(), T(g["out"]))
    assert torch.equal(select_focus_dist(T(g["depth_m"]).cuda(), 8).cpu(), T(g["out8"]))
    big = torch.rand(3, 1, 1080, 1920, generator=torch.Generator().manual_seed(1)) * 5
    big[big < 0.02] = 0.0
    assert torch.equal(select_focus_dist(big.cuda(), 7).cpu(), orc.select_focus_dist(big, 7))


@pytest.mark.parametrize("ks", [3, 7, 11, 15, 17, 31])
def test_thinlens_two_pixel_kernel_vs_oracle(pkg, ks):
    """ThinLens.render's kernel gives every thread two adjacent pixels (thinlens_render2_kernel: per-|dy| weight rows,
    LDS.64 windows).  Odd widths (the second pixel of the last thread does not exist), W % 4 != 0 (no TMA), border-only
    and interior tiles, C = 1 / 3 / 5, against the oracle."""
    from deeplens.psfnet import ThinLens
    gen = torch.Generator().manual_seed(700 + ks)
    for (N, C, H, W) in [(1, 1, 9, 13), (2, 3, 72, 200), (1, 5, 33, 67), (1, 3, 40, 264), (1, 2, 5, 64)]:
        tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=ks, sensor_size=[36.0, 24.0], sensor_res=(H, W)).to("cuda")
        im = torch.rand(N, C, H, W, generator=gen)
        dp = 300 + 6000 * torch.rand(N, 1, H, W, generator=gen)
        fc = 500 + 3000 * torch.rand(N, generator=gen)
        got = tl.render(im.cuda(), dp.cuda(), fc.cuda())
        ref = orc.thinlens_render(im, dp, fc, ks, 50.0, 1.8, tl.ps)
        assert maxabs(got, ref) < 5e-6, (ks, N, C, H, W)


def test_render_psf_and_psf_map_golden(pkg):
    """f4 row: render_psf / render_psf_map (deeplens/render_psf.py:12-73) -- reflect padding, flipped PSF, per-channel
    PSFs, grid of patches with int(i/grid*H) bounds (non-divisible sizes) -- against the reference's own outputs."""
    from deeplens.render_psf import render_psf, render_psf_map, local_psf_render_high_res, local_psf_render
    g = load_golden("kat_i_psf_conv.npz")
    for i in range(4):
        out = render_psf(T(g[f"conv{i}_img"]).cuda(), T(g[f"conv{i}_psf"]).cuda())
        assert out.shape == g[f"conv{i}_out"].shape and maxabs(out, T(g[f"conv{i}_out"])) < 2e-6, i
    for i in range(3):
        out = render_psf_map(T(g[f"map{i}_img"]).cuda(), T(g[f"map{i}_psf"]).cuda(), int(g[f"map{i}_grid"]))
        ks = g[f"map{i}_psf"].shape[1] // int(g[f"map{i}_grid"])
        assert maxabs(out, T(g[f"map{i}_out"])) < 2e-6 * ks * ks, i          # un-normalised random PSFs: sums up to ks^2/2
    with pytest.raises(ValueError):
        render_psf(torch.rand(1, 3, 8, 8).cuda(), torch.rand(3, 4, 4).cuda())
    # the patch-wise gather keeps the reference's semantics: each patch replicate-padded on its own
    gen = torch.Generator().manual_seed(9)
    img, psf = torch.rand(1, 3, 40, 50, generator=gen), torch.rand(1, 40, 50, 5, 5, generator=gen)
    hi = local_psf_render_high_res(img.cuda(), psf.cuda(), patch_size=[16, 32], kernel_size=5)
    ref = torch.zeros_like(img)
    for (a, b) in [(0, 16), (16, 32), (32, 40)]:
        for (c, d) in [(0, 32), (32, 50)]:
            ref[:, :, a:b, c:d] = orc.local_psf_render(img[:, :, a:b, c:d], psf[:, a:b, c:d], 5)
    assert maxabs(hi, ref) < 2e-5                                                # un-normalised 5x5 PSFs: values ~ 8
    assert maxabs(hi, local_psf_render(img.cuda(), psf.cuda(), 5)) > 1e-3        # ... which is NOT the full-frame gather


def test_train_psfnet_matches_torch_autograd(pkg):
    """f3 row: forward + MSE + backward + AdamW of PSFNet.train_psfnet (deeplens/psfnet.py:79-132) on the device
    against the same step in fp32 torch on the CPU (the reference's operators: nn.Linear/ReLU/Sigmoid/F.normalize,
    nn.MSELoss, torch.optim.AdamW): gradients of the first step, then parameters and losses over several steps."""
    import torch.nn as nn
    nat = pkg.native
    ks, bs = 11, 128
    Ws, Bs = orc.seeded_psfnet_weights(ks, seed=3)
    gen = torch.Generator().manual_seed(17)
    Bs = [(torch.rand(b.shape, generator=gen) - 0.5) * 0.2 for b in Bs]
    dims = [4, 64, 256] + [256] * 8 + [ks * ks]
    mods = []
    for a, b in zip(dims[:-2], dims[1:-1]):
        mods += [nn.Linear(a, b), nn.ReLU(inplace=True)]
    mods += [nn.Linear(dims[-2], dims[-1]), nn.Sigmoid()]
    net = nn.Sequential(*mods)
    with torch.no_grad():
        for lin, W, b in zip([m for m in net if isinstance(m, nn.Linear)], Ws, Bs):
            lin.weight.copy_(W)
            lin.bias.copy_(b)
    opt = torch.optim.AdamW(net.parameters(), 1e-4)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=8, eta_min=0)
    trainer = nat.NativeTrainer([w.numpy() for w in Ws], [b.numpy() for b in Bs], bs, 0)
    loss_dev = torch.zeros(1, device="cuda")
    for it in range(5):
        inp = torch.rand(bs, 4, generator=gen)
        inp[:, :2] = inp[:, :2] * 2 - 1
        tgt = torch.rand(bs, ks * ks, generator=gen)
        tgt = tgt / tgt.sum(1, keepdim=True)
        pred = torch.nn.functional.normalize(net(inp), p=1, dim=-1)
        opt.zero_grad()
        loss = nn.MSELoss()(pred, tgt)
        loss.backward()
        lr_i = opt.param_groups[0]["lr"]
        inp_d, tgt_d = inp.cuda(), tgt.cuda()            # (keep both alive: a freed temporary's block would be reused)
        nat.check(nat.lib.aadff_trainer_step(trainer.handle, inp_d.data_ptr(), tgt_d.data_ptr(), lr_i,
                                             loss_dev.data_ptr(), None))
        torch.cuda.synchronize()
        assert abs(float(loss_dev) - float(loss.detach())) < 1e-6 * max(1.0, float(loss.detach())) + 1e-9, it
        if it == 0:
            gw, gb = trainer.read(1)
            for lin, a, b in zip([m for m in net if isinstance(m, nn.Linear)], gw, gb):
                scale = float(lin.weight.grad.abs().max()) + 1e-12
                assert float((torch.from_numpy(a) - lin.weight.grad).abs().max()) < 2e-5 * scale
                assert float((torch.from_numpy(b) - lin.bias.grad).abs().max()) < 2e-5 * (float(lin.bias.grad.abs().max()) + 1e-12)
        opt.step()
        sched.step()
    pw, pb = trainer.read(0)
    for lin, a, b in zip([m for m in net if isinstance(m, nn.Linear)], pw, pb):
        # AdamW moves every weight by ~lr per step whatever the gradient's size: agreement to a small fraction of lr
        assert float((torch.from_numpy(a) - lin.weight.detach()).abs().max()) < 2e-5
        assert float((torch.from_numpy(b) - lin.bias.detach()).abs().max()) < 2e-5
    trainer.close()
    # the Python surface: a fit on synthetic targets lowers the loss and writes the weights back
    lens = pkg.PSFNet(kernel_size=ks, device="cuda")
    target_net = pkg.PSFNet(kernel_size=ks, device="cuda")
    def data(bs, spp):
        x = torch.rand(bs, 4, device="cuda")
        x[:, :2] = x[:, :2] * 2 - 1
        return x, target_net.pred(x).reshape(bs, -1)
    before = [p.detach().clone() for p in lens.psfnet.parameters()]
    hist = lens.train_psfnet(iters=300, bs=128, lr=1e-3, evaluate_every=100, data=data, save=False)
    assert len(hist) == 3 and hist[-1][1] < hist[0][1]
    assert any(not torch.equal(a, b) for a, b in zip(before, lens.psfnet.parameters()))


def test_dataset_preparation_matches_reference_datasets(pkg):
    """f4 row, host data path: ToTensor + BGR->RGB + /255 + AutoAgument jitter/flips + Resize(antialias=True) (and
    cv.resize for Middlebury's depth) on the device, against what the reference's own Dataset classes returned for
    the same decoded arrays (tests/golden/make_golden_f4_data.py ran dff/dataset.py: Matterport3D, Middlebury)."""
    g = load_golden("kat_j_dataset_prep.npz")
    bgr = T(g["mp_bgr"]).cuda()[None]
    dep = torch.from_numpy(g["mp_depth"].astype(np.int16)).view(torch.uint16).cuda()[None]
    for tag in "abc":                                   # down-scale by 2, non-integer factor, identity
        aif, d = pkg.preprocess_rgbd(bgr, dep, tuple(int(v) for v in g[f"mp_{tag}_size"]), depth_div=4000.0)
        assert aif.shape[1:] == g[f"mp_{tag}_aif"].shape and maxabs(aif[0], T(g[f"mp_{tag}_aif"])) < 2e-6, tag
        assert maxabs(d[0], T(g[f"mp_{tag}_depth"])) < 2e-6, tag
    aif, d = pkg.preprocess_rgbd(bgr, dep, (48, 65), depth_div=4000.0, jitter=T(g["mp_aug_jitter"])[None],
                                 flips=torch.tensor([int(g["mp_aug_flips"])], dtype=torch.uint8))
    assert maxabs(aif[0], T(g["mp_aug_aif"])) < 2e-6 and maxabs(d[0], T(g["mp_aug_depth"])) < 2e-6
    mb_dep = torch.from_numpy(g["mb_depth"].astype(np.int16)).view(torch.uint16).cuda()[None]
    aif, d = pkg.preprocess_rgbd(T(g["mb_bgr"]).cuda()[None], mb_dep, (48, 64), depth_div=1000.0, depth_mode="cv2")
    assert maxabs(aif[0], T(g["mb_aif"])) < 2e-6 and maxabs(d[0], T(g["mb_depth_out"])) < 5e-6
    # a batch: per-image jitter / flips, image-only and depth-only calls
    b2 = torch.cat([bgr, bgr.flip(1)]), torch.cat([dep, dep.flip(1)])
    aif2, d2 = pkg.preprocess_rgbd(b2[0], b2[1], (48, 65), jitter=torch.tensor([[-1.0, 0.0], [-1.0, 0.0]]),
                                   flips=torch.tensor([0, 2], dtype=torch.uint8))
    assert torch.equal(aif2[0], aif2[1]) and torch.equal(d2[0], d2[1])          # flipping a flipped image = the image
    only_img, none_d = pkg.preprocess_rgbd(bgr, None, (48, 65))
    assert none_d is None and maxabs(only_img[0], T(g["mp_a_aif"])) < 2e-6
    # straight into the simulator: decoded arrays -> focal stack without touching the host
    lens = pkg.PSFNet(kernel_size=11, device="cuda")
    lens.load_net(CKPT)
    a, dm = pkg.preprocess_rgbd(bgr, dep, (48, 64), depth_div=1000.0)
    stack, foc = lens.simulate_focal_stack(a, dm, 5)
    assert stack.shape == (1, 3, 5, 48, 64) and bool(torch.isfinite(stack).all())


def test_auto_augment_rotation_on_the_device(pkg):
    """f4 row, AutoAgument's rotation (dff/dataset.py:275-284: scipy.ndimage.rotate, order-3 spline, 'constant') on the
    device between the flips and the resize: against what the reference's own Matterport3D(train=True) returned for
    seeds that draw a rotation (alone / with jitter and both flips / with one flip), against scipy's full-resolution
    rotation of the decoded arrays, and against the oracle on odd shapes, multiples of 90 degrees and mixed batches."""
    from oracle import spline_rotate_oracle as so
    g = load_golden("kat_l_rotate.npz")
    bgr = T(g["bgr"]).cuda()[None]
    dep = torch.from_numpy(g["depth"].astype(np.int16)).view(torch.uint16).cuda()[None]
    for i in range(3):
        aif, d = pkg.preprocess_rgbd(bgr, dep, (48, 65), depth_div=4000.0, jitter=T(g[f"case{i}_jitter"])[None],
                                     flips=torch.tensor([int(g[f"case{i}_flips"])], dtype=torch.uint8),
                                     rotate_deg=[float(g[f"case{i}_degree"])])
        assert maxabs(aif[0], T(g[f"case{i}_aif"])) < 3e-6 and maxabs(d[0], T(g[f"case{i}_depth"])) < 3e-6, i
    # no resize: the rotation itself at full resolution
    H, W = g["bgr"].shape[:2]
    aif, d = pkg.preprocess_rgbd(bgr, dep, (H, W), depth_div=4000.0, rotate_deg=[float(g["full_degree"])])
    assert maxabs(aif[0], T(g["full_aif"]).permute(2, 0, 1)) < 3e-6 and maxabs(d[0, 0], T(g["full_depth"])) < 3e-6
    # a batch: sample 0 not rotated (== the one-launch path), samples 1.. at 90 / 180 / 33 degrees vs the oracle
    gen = np.random.default_rng(8)
    for (H, W) in [(37, 50), (16, 16), (5, 23)]:
        b8 = torch.from_numpy(gen.integers(0, 256, (4, H, W, 3), dtype=np.uint8)).cuda()
        d16 = torch.from_numpy(gen.integers(0, 8000, (4, H, W)).astype(np.int16)).view(torch.uint16).cuda()
        degs = [float("nan"), 90.0, 180.0, 33.0]
        aif, d = pkg.preprocess_rgbd(b8, d16, (H, W), depth_div=1000.0, rotate_deg=degs)
        plain_a, plain_d = pkg.preprocess_rgbd(b8[:1], d16[:1], (H, W), depth_div=1000.0)
        assert maxabs(aif[0], plain_a[0]) < 1e-6 and maxabs(d[0], plain_d[0]) < 1e-6
        for k in (1, 2, 3):
            oi, od = so.auto_augment_rotate(b8[k].cpu().numpy()[..., ::-1] / 255., d16[k].cpu().view(torch.int16).numpy().astype(np.float64) / 1000, degs[k])
            assert maxabs(aif[k], torch.from_numpy(oi).float().permute(2, 0, 1)) < 3e-6, (H, W, k)
            assert maxabs(d[k, 0], torch.from_numpy(od).float()) < 3e-5, (H, W, k)        # depths up to 8 m
        only_img, none_d = pkg.preprocess_rgbd(b8, None, (H, W), rotate_deg=degs)
        assert none_d is None and maxabs(only_img, aif) < 1e-6
        none_a, only_d = pkg.preprocess_rgbd(None, d16, (H, W), depth_div=1000.0, rotate_deg=degs)
        assert none_a is None and maxabs(only_d, d) < 1e-6


# --------------------------------------------------------------------------- oracle on seeded inputs, edge cases
@pytest.mark.parametrize("N,C,H,W", [(1, 3, 1, 1), (1, 3, 9, 1), (1, 3, 1, 21), (1, 1, 13, 37), (3, 4, 8, 16), (1, 5, 9, 17),
                                     (2, 3, 7, 130)])
def test_edge_shapes_vs_oracle(lens, rf50mm_weights, N, C, H, W):
    g = torch.Generator().manual_seed(N * 1000 + H * 10 + W)
    img = torch.rand(N, C, H, W, generator=g)
    dm = 0.3 + 6 * torch.rand(N, 1, H, W, generator=g)
    foc = -(500 + 4000 * torch.rand(N, generator=g))
    ref = orc.render(*rf50mm_weights, img, -dm * 1e3, foc, 11)
    for mode in ("parity", "fp32"):
        out = lens.render(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode=mode)
        assert out.shape == (N, C, H, W)
        assert maxabs(out, ref) < TOL[mode], mode


def test_empty_batch_and_inputs_untouched(lens):
    img = torch.rand(0, 3, 16, 16).cuda()
    out = lens.render(img, torch.rand(0, 1, 16, 16).cuda(), torch.rand(0).cuda())
    assert out.shape == (0, 3, 16, 16)
    img = torch.rand(1, 3, 24, 24).cuda()
    dep = -(torch.rand(1, 1, 24, 24).cuda() * 4000 + 300)
    foc = torch.tensor([-1500.0]).cuda()
    keep = (img.clone(), dep.clone(), foc.clone())
    lens.render(img, dep, foc)
    assert torch.equal(img, keep[0]) and torch.equal(dep, keep[1]) and torch.equal(foc, keep[2])


def test_weight_update_rebuilds_device_copy(pkg):
    l = pkg.PSFNet(kernel_size=11, device="cuda")
    l.load_net(CKPT)
    img, dm = analytic_rgbd(1, 32, 32)
    a = l.render(img.cuda(), -dm.cuda() * 1e3, torch.tensor([-900.0]).cuda())
    with torch.no_grad():
        l.psfnet.net[20].bias.add_(torch.linspace(-3, 3, 121, device="cuda"))
    b = l.render(img.cuda(), -dm.cuda() * 1e3, torch.tensor([-900.0]).cuda())
    assert maxabs(a, b) > 1e-3
    sd = torch.load(CKPT, map_location="cpu")
    assert set(l.psfnet.state_dict().keys()) == set(sd.keys())


def test_host_buffer_entry_point(pkg, lens):
    """aadff_render_stack_host_f32 (host buffers; upload / compute / download pipelined over two parts: image halves for
    N >= 2, row bands for a single image) returns exactly what the device-pointer call returns."""
    nat = pkg.native
    for (N, S, H, W, mode) in [(2, 4, 40, 48, "parity"), (3, 2, 24, 40, "parity"), (1, 3, 64, 48, "parity"), (1, 2, 37, 50, "fp32"),
                               (1, 1, 5, 9, "parity"), (1, 5, 128, 96, "econ")]:
        img, dm = orc.synthetic_rgbd(N, H, W, seed=3 + H)
        foc = -orc.synthetic_focus(dm, S) * 1e3
        dep = (-dm * 1e3).reshape(N, H, W).contiguous()
        out = torch.full((N, 3, S, H, W), -1.0)
        nat.check(nat.lib.aadff_render_stack_host_f32(lens.native().handle, img.data_ptr(), dep.data_ptr(),
                                                      foc.contiguous().data_ptr(), out.data_ptr(), N, 3, S, H, W,
                                                      -200.0, -20000.0, nat.MODES[mode]))
        dev = lens.render_stack(img.cuda(), dep.cuda(), foc.cuda(), mode=mode)
        assert torch.equal(out, dev.cpu()), (N, S, H, W, mode)


def test_c_abi_error_codes(pkg, lens):
    nat = pkg.native
    h = lens.native().handle
    s = (ctypes.c_int64 * 5)(1, 1, 1, 1, 1)
    assert nat.lib.aadff_render_stack_f32(h, None, None, None, None, s, 1, 3, 1, 8, 8, -200.0, -20000.0, 0, None) == -1
    assert nat.lib.aadff_render_stack_f32(h, 8, 8, 8, 8, s, 1, 3, 1, 8, 8, -200.0, -20000.0, 7, None) == -1
    assert nat.lib.aadff_local_psf_render_f32(8, 8, 8, 1, 3, 8, 8, 4, None) == -1          # even kernel size
    assert b"kernel size" in nat.lib.aadff_last_error()
    with pytest.raises(nat.AadffError):
        nat.NativePSFNet([np.zeros((64, 4), np.float32), np.zeros((9, 64), np.float32)],
                         [np.zeros(64, np.float32), np.zeros(9, np.float32)], 5, 0)      # 3*3 != 5*5


# --------------------------------------------------------------------------- properties at BASELINE sizes
def test_c2_constant_image_is_fixed_point(lens):
    """sum(PSF) = 1  =>  a constant image renders to itself (c2: 5 x 512 x 512)."""
    _, dm = orc.synthetic_rgbd(1, 512, 512, seed=1234)
    foc = -orc.synthetic_focus(dm, 5) * 1e3
    img = torch.full((1, 3, 512, 512), 0.625)
    for mode in ("parity", "fast"):
        out = lens.render_stack(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode=mode)
        assert float((out - 0.625).abs().max()) < 2e-6, mode


# --------------------------------------------------------------------------- BASELINE sizes against the REFERENCE's output
# (tests/golden/make_golden_baseline_sizes.py ran the reference itself on bench.py's seeded workloads; the inputs are
#  regenerated here from the same seed).  max-abs is printed (pytest -s / the GPU log) and asserted per mode.
@pytest.mark.parametrize("mode", ["parity", "econ", "econ8", "fp32", "fast"])
def test_c2_full_size_vs_reference_golden(lens, mode):
    """BASELINE config c2 (1 x 5 x 512 x 512, k = 11), all five slices, vs the reference's PSFNet.render."""
    g = load_golden("kat_c2_1x5x512x512.npz")
    img, dm = orc.synthetic_rgbd(1, 512, 512, seed=int(g["seed"]))
    foc_m = orc.synthetic_focus(dm, 5)
    assert torch.equal(foc_m, T(g["foc_m"]))
    out = lens.render_stack(img.cuda(), -dm.cuda() * 1e3, -foc_m.cuda() * 1e3, mode=mode).cpu()
    err = max(float((out[..., ::4, ::4] - T(g["out_sub"])).abs().max()),
              float((out[..., [0, 1, 255, 256, 510, 511], :] - T(g["out_rows"])).abs().max()))
    _report("c2 1x5x512x512 k=11", mode, err)
    assert err < BASELINE_TOL[mode]
    if mode == "fast":
        mean = float((out[..., ::4, ::4] - T(g["out_sub"])).abs().mean())
        print(f"[parity-at-size] c2 fast mean-abs = {mean:.3e}")
        assert mean < 1e-4
        return
    assert float((out.double().sum((1, 3, 4)) - T(g["sums"])).abs().max()) < 786432 * (1e-6 if mode.startswith("econ") else 5e-7)   # mean bias over ALL pixels of a slice


def test_econ8_mode_certified_between_parity_and_econ(pkg, lens):
    """AADFF_MODE_ECON8: two MMA terms only for L8, L9 and the head (calibrated fp16 weights), three before -- the earliest
    start whose worst case over ANY [0,1] image stays under north_star's 1e-4 (DESIGN.md section 5: the sweep).  Checked: that
    worst case (half the L1 distance between its PSFs and the fp32 PSFs) over 2^18 probes incl. faces and corners of
    the input box < 1e-4 and below econ's; the c1 golden of the reference; a noise image; pred(); bit-identical to
    parity on a network too shallow to have an eighth layer."""
    g = torch.Generator().manual_seed(5)
    x = torch.rand(1 << 18, 4, generator=g)
    x[:, :2] = x[:, :2] * 2 - 1
    m = x.shape[0] // 20
    x[:m, 0] = torch.sign(x[:m, 0]); x[m:2 * m, 1] = torch.sign(x[m:2 * m, 1])
    x[2 * m:3 * m, 2] = torch.round(x[2 * m:3 * m, 2]); x[3 * m:4 * m, 3] = torch.round(x[3 * m:4 * m, 3])
    x[4 * m:5 * m, :2] = torch.sign(x[4 * m:5 * m, :2]); x[5 * m:6 * m, 2:] = torch.round(x[5 * m:6 * m, 2:])
    x = x.cuda()
    ref = lens.pred(x).double()
    worst = {mode: float(((lens.pred(x, mode=mode).double() - ref).abs().sum((-1, -2)) / 2).max()) for mode in ("parity", "econ8", "econ")}
    print(f"[certificate] L1/2 max over {x.shape[0]} probes: {worst}")
    assert worst["econ8"] < 1e-4 and worst["parity"] <= worst["econ8"] <= worst["econ"]
    gold = load_golden("kat_b_1x480x640.npz")
    img, dm = analytic_rgbd(1, 480, 640)
    out = lens.render(img.cuda(), -dm.cuda() * 1e3, T(gold["foc"]).cuda(), mode="econ8")
    assert (out.cpu()[:, :, ::8, ::8] - T(gold["out_sub"])).abs().max() < TOL["econ8"]
    noise = torch.rand(1, 3, 256, 256, generator=g).cuda()
    dep = -(300 + 6000 * torch.rand(1, 1, 256, 256, generator=g)).cuda()
    foc = torch.tensor([[-800.0, -2500.0]]).cuda()
    exact = lens.render_stack(noise, dep, foc, mode="fp32")
    assert maxabs(lens.render_stack(noise, dep, foc, mode="econ8"), exact) < TOL["econ8"]
    # a network with two hidden 256-wide layers has no layer 8: econ8 = parity
    from deeplens.psfnet_arch import MLP
    shallow = pkg.PSFNet(kernel_size=11, device="cuda")
    shallow.psfnet = MLP(in_features=4, out_features=121, hidden_features=256, hidden_layers=2).to("cuda")
    a = shallow.render_stack(noise, dep, foc, mode="econ8")
    assert torch.equal(a, shallow.render_stack(noise, dep, foc, mode="parity"))


@pytest.mark.parametrize("mode", ["parity", "econ", "econ8", "fp32", "fast"])
def test_c3_full_size_vs_reference_golden(lens, mode):
    """BASELINE config c3 (16 x 5 x 256 x 256, k = 11): all 16 images, all slices (1/64 of the pixels of every slice,
    1/4 of image 3, sums over everything); fp32 on images 0..3 only (16.5 Mpix/s kernel)."""
    g = load_golden("kat_c3_16x5x256x256.npz")
    img, dm = orc.synthetic_rgbd(16, 256, 256, seed=int(g["seed"]))
    foc_m = orc.synthetic_focus(dm, 5)
    assert torch.equal(foc_m, T(g["foc_m"]))
    n = 4 if mode == "fp32" else 16
    out = lens.render_stack(img[:n].cuda(), -dm[:n].cuda() * 1e3, -foc_m[:n].cuda() * 1e3, mode=mode).cpu()
    err = max(float((out[..., ::8, ::8] - T(g["out_sub"])[:n]).abs().max()),
              float((out[3, :, :, ::2, ::2] - T(g["out_full_img3"])).abs().max()))
    _report("c3 16x5x256x256 k=11", mode, err)
    assert err < BASELINE_TOL[mode]
    if mode == "fast":
        assert float((out[..., ::8, ::8] - T(g["out_sub"])[:n]).abs().mean()) < 1e-4
        return
    assert float((out.double().sum((1, 3, 4)) - T(g["sums"])[:n]).abs().max()) < 196608 * (1e-6 if mode.startswith("econ") else 5e-7)


@pytest.fixture(scope="module")
def lens31_bench(pkg):
    """bench.py's c4 network: PSFNet(kernel_size=31) with the seeded kaiming-uniform weights, zero biases."""
    Ws, bs = orc.seeded_psfnet_weights(31, seed=0)
    l = pkg.PSFNet(kernel_size=31, device="cuda")
    sd = {}
    for i, (W, b) in enumerate(zip(Ws, bs)):
        sd[f"net.{2 * i}.weight"], sd[f"net.{2 * i}.bias"] = W, b
    l.psfnet.load_state_dict(sd)
    return l


@pytest.mark.parametrize("mode", ["parity", "econ", "econ8", "fp32"])
def test_c4_full_size_vs_reference_golden(lens31_bench, mode):
    """BASELINE config c4 (1 x 10 x 1080 x 1920, k = 31): the whole stack is rendered; the top-border, middle and
    bottom-border 8-row bands of slices 0, 5, 9 are compared with the reference's banded evaluation (its own
    PSFNet.pred + local_psf_render on the row-padded full frame, proven bit-equal to a full-frame call where that
    fits in memory -- see make_golden_baseline_sizes.py)."""
    g = load_golden("kat_c4_1x10x1080x1920_ks31.npz")
    img, dm = orc.synthetic_rgbd(1, 1080, 1920, seed=int(g["seed"]))
    foc_m = orc.synthetic_focus(dm, 10)
    assert torch.equal(foc_m, T(g["foc_m"]))
    slices = [int(s) for s in g["slices"]]
    sel = foc_m[:, slices] if mode == "fp32" else foc_m           # fp32 kernel: only the three compared slices
    out = lens31_bench.render_stack(img.cuda(), -dm.cuda() * 1e3, -sel.cuda() * 1e3, mode=mode)
    cs, err = int(g["col_stride"]), 0.0
    for i, s in enumerate(slices):
        for (h0, h1) in g["bands"]:
            got = out[0, :, i if mode == "fp32" else s, int(h0):int(h1), ::cs].cpu()
            err = max(err, float((got - T(g[f"s{s}_h{int(h0)}"])).abs().max()))
    _report("c4 1x10x1080x1920 k=31", mode, err)
    # seeded random weights (no k=31 checkpoint exists): econ's calibration is certified at the north_star bar there
    assert err < (1e-4 if mode == "econ" else BASELINE_TOL[mode])


def test_fast_mode_tile_rows_equal_the_full_launch(pkg, lens):
    """AADFF_MODE_FAST (single-term groups, 128 KB weight ring): a tile-row range reproduces the matching rows of the
    full launch bit for bit, and the stack stays within the mode's tolerance of parity; ragged shapes, odd tile counts,
    C = 1 / 3 / 4."""
    sh = pkg.sharding
    for (N, C, S, H, W) in [(1, 3, 1, 8, 16), (1, 3, 3, 37, 50), (2, 4, 2, 24, 40), (1, 1, 5, 64, 96), (3, 3, 4, 40, 56)]:
        gen = torch.Generator().manual_seed(H + W)
        img = torch.rand(N, C, H, W, generator=gen).cuda()
        _, dm = orc.synthetic_rgbd(N, H, W, seed=H)
        foc = -orc.synthetic_focus(dm, S).cuda() * 1e3
        dep = -dm.cuda() * 1e3
        full = lens.render_stack(img, dep, foc, mode="fast")
        R0, R1 = sh.tile_row_range(N, S, H, 3, 1)
        rows = lens.render_stack_rows(img, dep, foc, R0, R1, mode="fast")
        rows_full = full.permute(0, 2, 3, 1, 4).reshape(N * S * H, C, W)
        assert torch.equal(rows, rows_full[sh.flat_row(R0, H):sh.flat_row(R1, H)]), (N, C, S, H, W)
        assert maxabs(full, lens.render_stack(img, dep, foc, mode="parity")) < TOL["fast"]


def test_tile_row_ranges_are_bit_identical_to_the_full_launch(pkg, lens):
    """aadff_render_stack_rows_f32 (the multi-GPU partition unit): any split of the tile rows reproduces the full
    launch bit for bit, ragged H included, in the tensor-core and the fp32 kernel."""
    sh = pkg.sharding
    for (N, S, H, W) in [(2, 3, 37, 50), (1, 5, 64, 48)]:
        img, dm = orc.synthetic_rgbd(N, H, W, seed=H)
        foc = -orc.synthetic_focus(dm, S).cuda() * 1e3
        img, dep = img.cuda(), -dm.cuda() * 1e3
        for mode in ("parity", "fp32"):
            full = lens.render_stack(img, dep, foc, mode=mode)
            rows_full = full.permute(0, 2, 3, 1, 4).reshape(N * S * H, 3, W)
            for world in (1, 3, 8):
                parts = []
                for r in range(world):
                    R0, R1 = sh.tile_row_range(N, S, H, world, r)
                    part = lens.render_stack_rows(img, dep, foc, R0, R1, mode=mode)
                    assert part.shape[0] == sh.flat_row(R1, H) - sh.flat_row(R0, H)
                    parts.append(part)
                assert torch.equal(torch.cat(parts, 0), rows_full), (N, S, H, W, mode, world)
    nat = pkg.native
    s = (ctypes.c_int64 * 5)(1, 1, 1, 1, 1)
    assert nat.lib.aadff_render_stack_rows_f32(lens.native().handle, 8, 8, 8, 8, s, 1, 3, 1, 16, 8, -200.0, -20000.0,
                                               0, 1, 3, None) == -1            # only 2 tile rows exist


def test_thinlens_sign_decided_on_device_and_focus_sentinel(pkg):
    """ThinLens.render makes the reference's data-dependent sign decision (psfnet.py:504) on the device: no host
    synchronisation, so the call is CUDA-graph capturable; both sign conventions give the reference's result.
    select_focus_dist marks an image without valid depth with NaN instead of silently returning +inf."""
    from deeplens.psfnet import ThinLens
    from dff.utils import select_focus_dist
    tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=11, sensor_size=[36.0, 24.0], sensor_res=(40, 56)).to("cuda")
    gen = torch.Generator().manual_seed(3)
    img = torch.rand(1, 3, 40, 56, generator=gen).cuda()
    dep = (300 + 6000 * torch.rand(1, 1, 40, 56, generator=gen)).cuda()
    foc = torch.tensor([1500.0]).cuda()
    pos = tl.render(img, dep, foc)
    neg = tl.render(img, -dep, -foc)
    assert torch.equal(pos, neg)
    assert maxabs(pos, orc.thinlens_render(img.cpu(), dep.cpu(), foc.cpu(), 11, 50.0, 1.8, tl.ps)) < 5e-6
    # interior tiles take their halo as one TMA tensor tile, border tiles (and W % 4 != 0 images) by clamped cp.async:
    # both against the oracle, and the TMA path bit-equal to the all-cp.async path (debug flag 16)
    for (N, C, H, W, ks) in [(2, 3, 72, 200, 11), (1, 4, 40, 136, 7), (1, 3, 64, 130, 11), (1, 1, 96, 160, 31), (1, 5, 33, 68, 3)]:
        tlk = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=ks, sensor_size=[36.0, 24.0], sensor_res=(H, W)).to("cuda")
        im = torch.rand(N, C, H, W, generator=gen)
        dp = 300 + 6000 * torch.rand(N, 1, H, W, generator=gen)
        fc = 500 + 3000 * torch.rand(N, generator=gen)
        ref = orc.thinlens_render(im, dp, fc, ks, 50.0, 1.8, tlk.ps)
        got = tlk.render(im.cuda(), dp.cuda(), fc.cuda())
        assert maxabs(got, ref) < 5e-6, (N, C, H, W, ks)
        pkg.native.lib.aadff_debug_set_flags(16)
        try:
            assert torch.equal(tlk.render(im.cuda(), dp.cuda(), fc.cuda()), got)
        finally:
            pkg.native.lib.aadff_debug_set_flags(0)
    graph, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        tl.render(img, -dep, -foc)
        with torch.cuda.graph(graph, stream=side):
            captured = tl.render(img, -dep, -foc)
    torch.cuda.current_stream().wait_stream(side)
    captured.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, pos)
    d = torch.rand(3, 1, 16, 16).cuda() + 0.5
    d[1] = 0.0                                               # image 1: no valid depth at all
    f = select_focus_dist(d, 5)
    assert bool(torch.isnan(f[1]).all()) and bool(torch.isfinite(f[[0, 2]]).all())
    lens = pkg.PSFNet(kernel_size=11, device="cuda")
    with pytest.raises(ValueError):
        lens.simulate_focal_stack(torch.rand(3, 3, 16, 16).cuda(), d, 5, check=True)


def test_c2_tensor_core_vs_fp32_full_size(lens):
    img, dm = orc.synthetic_rgbd(1, 512, 512, seed=1234)
    foc = -orc.synthetic_focus(dm, 5) * 1e3
    ref = lens.render_stack(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode="fp32")
    out = lens.render_stack(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode="parity")
    assert float((out - ref).abs().max()) < TOL["parity"]
    lo = torch.nn.functional.pad(img, (5, 5, 5, 5), mode="replicate").cuda()
    mn = -torch.nn.functional.max_pool2d(-lo, 11, 1)
    mx = torch.nn.functional.max_pool2d(lo, 11, 1)
    assert bool(((out >= mn.unsqueeze(2) - 1e-5) & (out <= mx.unsqueeze(2) + 1e-5)).all())   # convex combination


def test_c3_linearity_in_the_image_at_full_size(lens):
    """For fixed depth and focus the render is linear in the image (the PSFs do not depend on it): a size-independent
    property checked on the whole c3 batch (16 x 5 x 256 x 256) -- render(a*x + b*y) == a*render(x) + b*render(y) up to
    fp32 rounding of the 121-tap sums, and the constant offset passes through unchanged (sum of a PSF = 1)."""
    img, dm = orc.synthetic_rgbd(16, 256, 256, seed=31)
    img2, _ = orc.synthetic_rgbd(16, 256, 256, seed=32)
    foc = -orc.synthetic_focus(dm, 5).cuda() * 1e3
    dep = -dm.cuda() * 1e3
    x, y = img.cuda(), img2.cuda()
    rx, ry = lens.render_stack(x, dep, foc), lens.render_stack(y, dep, foc)
    mix = lens.render_stack(0.25 * x + 0.5 * y + 0.125, dep, foc)
    assert float((mix - (0.25 * rx + 0.5 * ry + 0.125)).abs().max()) < 2e-6


def test_c3_batch_independence(lens):
    """c3 (16 x 5 x 256 x 256): rendering the batch == rendering each image alone, bit for bit."""
    img, dm = orc.synthetic_rgbd(16, 256, 256, seed=77)
    foc = -orc.synthetic_focus(dm, 5) * 1e3
    img, dep, foc = img.cuda(), -dm.cuda() * 1e3, foc.cuda()
    full = lens.render_stack(img, dep, foc)
    for n in (0, 7, 15):
        assert torch.equal(full[n:n + 1], lens.render_stack(img[n:n + 1], dep[n:n + 1], foc[n:n + 1]))
    ref = lens.render_stack(img[3:5], dep[3:5], foc[3:5], mode="fp32")
    assert float((full[3:5] - ref).abs().max()) < TOL["parity"]


def test_c4_large_kernel_full_frame(lens31):
    """c4's frame (1080 x 1920, k = 31), two slices: tensor-core path vs fp32 path + fixed point."""
    img, dm = orc.synthetic_rgbd(1, 1080, 1920, seed=9)
    foc = -orc.synthetic_focus(dm, 2) * 1e3
    img, dep, foc = img.cuda(), -dm.cuda() * 1e3, foc.cuda()
    out = lens31.render_stack(img, dep, foc, mode="parity")
    ref = lens31.render_stack(img, dep, foc[:, :1], mode="fp32")
    assert float((out[:, :, :1] - ref).abs().max()) < TOL["parity"]
    const = lens31.render_stack(torch.full_like(img, 0.25), dep, foc[:, 1:], mode="parity")
    assert float((const - 0.25).abs().max()) < 2e-6


def test_multi_gpu_sharded_render_matches_single_gpu():
    """2 ranks over NCCL: shares rendered per rank, all_gathered, bit-identical to one GPU (skips on 1 GPU)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29613",
                          os.path.join(root, "tests", "gpu_multi_verify.py")], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "MULTI_GPU_VERIFY PASS" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_second_device_in_one_process(pkg):
    """One process, two GPUs: everything on cuda:1 while cuda:0 stays the current device (the per-device shared-memory
    opt-in of the large-kernel gather / thin lens was once cached per process -- ADVICE r01).  Skips on one GPU."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    from deeplens.psfnet import ThinLens
    from deeplens.render_psf import local_psf_render
    dev = torch.device("cuda:1")
    assert torch.cuda.current_device() == 0
    l1 = pkg.PSFNet(kernel_size=11, device="cuda:1")
    l1.load_net(CKPT)
    l0 = pkg.PSFNet(kernel_size=11, device="cuda:0")
    l0.load_net(CKPT)
    img, dm = orc.synthetic_rgbd(1, 40, 56, seed=5)
    foc = -orc.synthetic_focus(dm, 3) * 1e3
    for mode in ("parity", "econ", "fp32"):
        a = l0.render_stack(img.cuda(0), -dm.cuda(0) * 1e3, foc.cuda(0), mode=mode)
        b = l1.render_stack(img.to(dev), -dm.to(dev) * 1e3, foc.to(dev), mode=mode)
        assert b.device == dev and torch.equal(a.cpu(), b.cpu()), mode
    gen = torch.Generator().manual_seed(1)
    im = torch.rand(1, 3, 20, 24, generator=gen)
    psf = torch.rand(1, 20, 24, 31, 31, generator=gen)                  # ks = 31, 3 channels: > 48 KB of shared memory
    for d in (dev, torch.device("cuda:0")):
        assert maxabs(local_psf_render(im.to(d), psf.to(d), 31), orc.local_psf_render(im, psf, 31)) < 5e-4
    tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=31, sensor_size=[36.0, 24.0], sensor_res=(96, 160)).to(dev)
    im = torch.rand(1, 3, 96, 160, generator=gen)
    dp = 300 + 6000 * torch.rand(1, 1, 96, 160, generator=gen)
    fc = torch.tensor([1500.0])
    assert maxabs(tl.render(im.to(dev), dp.to(dev), fc.to(dev)), orc.thinlens_render(im, dp, fc, 31, 50.0, 1.8, tl.ps)) < 5e-6
    assert torch.cuda.current_device() == 0


def test_install_grafts_cuda_path_onto_the_unmodified_reference():
    """aadff_b200.install() on the REAL reference (the unmodified copy in baseline/_ref, imported first): the reference's
    own PSFNet -- ray-traced Lensgroup constructor, its own MLP module -- renders through libaadff.so afterwards and
    reproduces the reference golden; uninstall() gives the eager path back.  Runs in a child process (the reference's
    `deeplens` and the shadow package cannot share an interpreter); skips where baseline/_ref is absent."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.isfile(os.path.join(root, "baseline", "_ref", "deeplens", "psfnet.py")):
        pytest.skip("baseline/_ref (copy of the reference) not present")
    code = f"""
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
from baseline import ref_import
ref_psfnet = ref_import.import_reference()
sd = torch.load({CKPT!r}, map_location='cpu')
lens = ref_import.make_lens(11, (480, 640), 'cuda', sd)
assert type(lens).__module__ == 'deeplens.psfnet' and 'baseline/_ref' in sys.modules['deeplens.psfnet'].__file__
g = np.load({os.path.join(GOLDEN, 'kat_b_2x64x64.npz')!r})
n, c, h, w = np.meshgrid(np.arange(2), np.arange(3), np.arange(64), np.arange(64), indexing='ij')
img = torch.tensor(((7 * h + 13 * w + 29 * c + 101 * n) % 256) / 255.0, dtype=torch.float32).cuda()
n, h, w = np.meshgrid(np.arange(2), np.arange(64), np.arange(64), indexing='ij')
dm = torch.tensor(0.5 + 4.5 * (((h * 64 + w) * 31 + 17 * n) % 1000) / 999.0, dtype=torch.float32).unsqueeze(1).cuda()
foc = torch.tensor(g['foc']).cuda()
eager = lens.render(img, -dm * 1e3, foc)                     # the reference's own eager path
import aadff_b200
launches0 = aadff_b200.native.lib.aadff_launch_count()
assert aadff_b200.install() is True
ours = lens.render(img, -dm * 1e3, foc)                      # same object, same call: now the fused kernel
assert aadff_b200.native.lib.aadff_launch_count() == launches0 + 1
gold = torch.tensor(g['out'])
assert float((ours.cpu() - gold).abs().max()) < 2e-5 and float((eager.cpu() - gold).abs().max()) < 2e-5
stack = lens.render_stack(img, -dm * 1e3, torch.stack([foc, foc * 1.5], 1))
assert stack.shape == (2, 3, 2, 64, 64) and torch.equal(stack[:, :, 0], ours)
psf = lens.pred(torch.tensor([[0., 0., .5, .5]]).cuda())
assert abs(float(psf[0, 5, 5]) - 0.810939252) < 1e-6         # SURVEY.md 8c literal, through the grafted pred
aadff_b200.uninstall()
back = lens.render(img, -dm * 1e3, foc)
assert aadff_b200.native.lib.aadff_launch_count() == launches0 + 3 and torch.equal(back, eager)
print('INSTALL-GPU-OK')
"""
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, PYTHONPATH=""))
    assert res.returncode == 0 and "INSTALL-GPU-OK" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]


def test_reference_training_script_runs_unchanged_on_the_shadow_package(tmp_path):
    """The reference's own 2_aber_aware_dff_aif.py -- byte for byte the copy in baseline/_ref -- executed with the shadow
    directory in front of the reference on PYTHONPATH: config(), get_lens, get_dataset (the reference's Matterport3D /
    Middlebury classes on a tiny synthetic dataset), two training iterations (select_focus_dist + 8 x lens.render +
    AiFDepthNet forward/backward) and one validate() pass.  Only data is adapted: the YAML (1 epoch, no pretrained DFF
    checkpoint, which the reference does not ship) and the dataset directory.  Optional packages this image lacks
    (wandb, skimage, matplotlib, lpips) are stubbed through sitecustomize.  Asserts that the fused kernel did the renders."""
    import shutil
    import subprocess
    import sys
    import cv2 as cv
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.path.join(root, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref, "2_aber_aware_dff_aif.py")):
        pytest.skip("baseline/_ref (copy of the reference) not present")
    work = tmp_path / "work"
    for d in ("configs", "lenses/rf50mm", "ckpt/rf50mm", "stubs"):
        (work / d).mkdir(parents=True)
    shutil.copy(os.path.join(ref, "2_aber_aware_dff_aif.py"), work / "2_aber_aware_dff_aif.py")
    shutil.copy(os.path.join(ref, "lenses/rf50mm/lens.json"), work / "lenses/rf50mm/lens.json")
    shutil.copy(os.path.join(ref, "ckpt/rf50mm/PSFNet480x640_ks11.pkl"), work / "ckpt/rf50mm/PSFNet480x640_ks11.pkl")
    with open(os.path.join(ref, "configs/aber_aware_dff_aif.yml")) as fh:
        yml = fh.read()
    yml = yml.replace("dffnet_pretrained: './ckpt/rf50mm/aifnet_stack8_480x640.pkl'", "dffnet_pretrained: ''").replace("epochs: 20", "epochs: 1")
    assert "dffnet_pretrained: ''" in yml and "epochs: 1 " in yml
    (work / "configs/aber_aware_dff_aif.yml").write_text(yml)
    rng = np.random.default_rng(3)
    yy, xx = np.mgrid[0:480, 0:640]
    for i in range(2):
        img = np.stack([(127 + 90 * np.sin(xx / (9.0 + i) + c) * np.cos(yy / 7.0)).clip(0, 255) for c in range(3)], -1).astype(np.uint8)
        dep = (6000 + 4000 * np.sin(xx / 50.0 + i) + 3000 * (yy > 200)).astype(np.uint16)          # / 4000 -> metres
        a = work / f"dataset/Matterport3D/train/aif/scene0/undistorted_color_images"
        b = work / f"dataset/Matterport3D/train/depth/scene0/render_depth"
        a.mkdir(parents=True, exist_ok=True); b.mkdir(parents=True, exist_ok=True)
        cv.imwrite(str(a / f"{i}.jpg"), img); cv.imwrite(str(b / f"{i}.png"), dep)
    m = work / "dataset/Middlebury2014/sceneA"
    m.mkdir(parents=True)
    cv.imwrite(str(m / "im0.png"), img); cv.imwrite(str(m / "depth.png"), (dep // 4).astype(np.uint16))   # mm
    (work / "stubs/sitecustomize.py").write_text("""
import sys, types, atexit
for name in ["matplotlib", "matplotlib.pyplot", "lpips", "skimage", "skimage.metrics", "skimage.morphology", "skimage.filters", "wandb"]:
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
sys.modules["skimage.metrics"].peak_signal_noise_ratio = lambda *a, **k: 0.0
sys.modules["skimage.metrics"].structural_similarity = lambda *a, **k: 0.0
sys.modules["skimage.morphology"].disk = sys.modules["skimage.morphology"].closing = lambda *a, **k: None
import scipy.ndimage
sys.modules.setdefault("scipy.ndimage.interpolation", scipy.ndimage)
def _report():
    nat = sys.modules.get("aadff_native")
    lens = sys.modules.get("deeplens.psfnet")
    print("AADFF-LAUNCHES", nat.lib.aadff_launch_count() if nat else -1, getattr(lens, "__file__", None), flush=True)
atexit.register(_report)
""")
    shadow = os.path.join(root, "aberration-aware-depth-from-focus_b200")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([str(work / "stubs"), shadow, ref]))
    res = subprocess.run([sys.executable, "2_aber_aware_dff_aif.py"], cwd=work, capture_output=True, text=True, timeout=900, env=env)
    tail = res.stdout[-1500:] + res.stderr[-3000:]
    assert res.returncode == 0, tail
    line = [l for l in res.stdout.splitlines() if l.startswith("AADFF-LAUNCHES")][-1].split()
    # 2 training iterations x (1 select_focus + 8 renders) + 1 validation image x (1 + 8) launches of libaadff kernels
    assert int(line[1]) >= 27 and "aberration-aware-depth-from-focus_b200" in line[2], line
    results = [d for d in (work / "results").iterdir()]
    assert results and (results[0] / "depth_net_last.pkl").exists(), tail


def test_reference_warm_up_script_runs_unchanged_on_the_shadow_package(tmp_path):
    """0_warm_up.py (BASELINE configs[0]) itself, byte for byte from baseline/_ref, on the shadow package: the script's
    image files are synthetic (the reference checkout ships no Middlebury RGB), everything else is the script."""
    import shutil
    import subprocess
    import sys
    import cv2 as cv
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.path.join(root, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref, "0_warm_up.py")):
        pytest.skip("baseline/_ref (copy of the reference) not present")
    work = tmp_path / "work"
    for d in ("lenses/rf50mm", "ckpt/rf50mm", "datasets/Middlebury2014/Adirondack-perfect"):
        (work / d).mkdir(parents=True)
    shutil.copy(os.path.join(ref, "0_warm_up.py"), work / "0_warm_up.py")
    shutil.copy(os.path.join(ref, "lenses/rf50mm/lens.json"), work / "lenses/rf50mm/lens.json")
    shutil.copy(os.path.join(ref, "ckpt/rf50mm/PSFNet480x640_ks11.pkl"), work / "ckpt/rf50mm/PSFNet480x640_ks11.pkl")
    g = load_golden("kat_k_warmup_c1.npz")
    cv.imwrite(str(work / "datasets/Middlebury2014/Adirondack-perfect/im0.png"), cv.cvtColor(g["img_u8"], cv.COLOR_RGB2BGR))
    cv.imwrite(str(work / "datasets/Middlebury2014/Adirondack-perfect/depth.png"), (g["depth_m"] * 1000).round().astype(np.uint16))
    shadow = os.path.join(root, "aberration-aware-depth-from-focus_b200")
    res = subprocess.run([sys.executable, "0_warm_up.py"], cwd=work, capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, PYTHONPATH=os.pathsep.join([shadow, ref])))
    assert res.returncode == 0, res.stdout[-1500:] + res.stderr[-3000:]
    out = cv.cvtColor(cv.imread(str(work / "aberrated_defocused_img.png")), cv.COLOR_BGR2RGB).astype(np.float32) / 255
    ref_sub = np.transpose(g["out_sub"][0], (1, 2, 0))                        # the reference's CPU render of the same inputs
    assert out.shape == (480, 640, 3) and float(np.abs(out[::3, ::3] - ref_sub).max()) < 1.5 / 255     # 8-bit PNG rounding


def test_fitting_with_the_reference_ray_tracer_and_the_device_trainer():
    """Row f3 as SURVEY 8f frames it: the ray-traced training targets stay in the reference's Python
    (PSFNet.get_training_data on the unmodified copy in baseline/_ref), the optimisation of train_psfnet runs on the
    device through the grafted method (tests/gpu_fit_with_reference_raytracer.py, child process)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.isfile(os.path.join(root, "baseline", "_ref", "deeplens", "psfnet.py")):
        pytest.skip("baseline/_ref (copy of the reference) not present")
    res = subprocess.run([sys.executable, os.path.join(root, "tests", "gpu_fit_with_reference_raytracer.py"), "20"],
                         capture_output=True, text=True, timeout=900, env=dict(os.environ, PYTHONPATH=""))
    assert res.returncode == 0 and "FIT-OK" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]
    losses = [float(x.strip("'")) for x in res.stdout.split("losses: [")[1].split("]")[0].split(", ")]
    assert len(losses) == 2 and all(0 < l < 1e-3 for l in losses), losses


def test_simulate_focal_stack_matches_training_loop(lens):
    """The block 2_aber_aware_dff_aif.py:101-114 (select_focus_dist + S renders + stack) as one call."""
    from dff.utils import select_focus_dist
    img, dm = orc.synthetic_rgbd(2, 64, 96, seed=11)
    img, dm = img.cuda(), dm.cuda()
    stack, foc = lens.simulate_focal_stack(img, dm, 5)
    ref_foc = select_focus_dist(dm, 5, mode='linear')
    loop = torch.stack([lens.render(img, depth=-dm * 1e3, foc_dist=-ref_foc[:, i] * 1e3) for i in range(5)], dim=2)
    assert torch.equal(foc, ref_foc) and torch.equal(stack, loop)


def test_render_is_cuda_graph_capturable(lens):
    """The C-ABI render never allocates or synchronises: it can be captured in a CUDA graph and replayed."""
    img, dm = orc.synthetic_rgbd(1, 64, 64, seed=21)
    foc = -orc.synthetic_focus(dm, 4).cuda() * 1e3
    img, dep = img.cuda(), -dm.cuda() * 1e3
    eager = lens.render_stack(img, dep, foc)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lens.render_stack(img, dep, foc)                  # warm-up on the capture stream
        with torch.cuda.graph(graph, stream=side):
            captured = lens.render_stack(img, dep, foc)
    torch.cuda.current_stream().wait_stream(side)
    captured.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)
    img.mul_(0.5)                                         # new data in the same buffers, replay again
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, lens.render_stack(img, dep, foc))


@pytest.mark.parametrize("ks", [1, 3, 5, 7, 9, 13, 21, 27])
def test_other_kernel_sizes_vs_oracle(pkg, ks):
    """Kernel sizes without a shipped checkpoint: seeded PSFNet weights (+ random biases) in the fused kernel
    (head padded to a multiple of 16 columns, 1..3 head blocks) against the CPU oracle."""
    Ws, bs = orc.seeded_psfnet_weights(ks, seed=ks)
    gen = torch.Generator().manual_seed(100 + ks)
    bs = [(torch.rand(b.shape, generator=gen) - 0.5) * 0.2 for b in bs]
    l = pkg.PSFNet(kernel_size=ks, device="cuda")
    sd = {}
    for i, (W, b) in enumerate(zip(Ws, bs)):
        sd[f"net.{2 * i}.weight"], sd[f"net.{2 * i}.bias"] = W, b
    l.psfnet.load_state_dict(sd)
    img, dm = orc.synthetic_rgbd(2, 24, 40, seed=ks)
    foc = -orc.synthetic_focus(dm, 2) * 1e3
    ref = orc.render_stack(Ws, bs, img, -dm * 1e3, foc, ks)
    for mode in ("parity", "fp32", "fast", "econ", "econ8", "mixed"):
        out = l.render_stack(img.cuda(), -dm.cuda() * 1e3, foc.cuda(), mode=mode)
        # econ / econ8: randomly initialised networks are not what their weight calibration was tuned on -> north_star's bar
        assert maxabs(out, ref) < (1e-4 if mode in ("econ", "econ8") else TOL[mode]), (ks, mode)
    probes = torch.rand(300, 4, generator=gen)
    ref_psf = orc.mlp_forward(Ws, bs, probes).reshape(-1, ks, ks)
    assert maxabs(l.pred(probes.cuda()), ref_psf) < 2e-6
    assert maxabs(l.pred(probes.cuda(), mode="parity"), ref_psf) < 1e-5
