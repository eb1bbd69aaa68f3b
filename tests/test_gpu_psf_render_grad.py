"""Gradients of local_psf_render, render_psf and render_psf_map (pytest -m gpu): the CUDA backward kernels
(psf_grad_kernel.cuh, psf_conv_grad_kernel.cuh) against torch autograd of the reference formulations in float64 on
the CPU, the autograd contract (which gradients, shapes, dtypes, devices), determinism, 64-bit indexing and CUDA-graph
capture.

Tolerances (max-abs over max|reference gradient|, fp32 sums of up to a few hundred terms): 1e-5 for the PSF
gradients, 2e-5 for the image gradients.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import focal_stack_oracle as orc

pytestmark = pytest.mark.gpu

TOL_PSF, TOL_IMG = 1e-5, 2e-5


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


def relerr(a, ref):
    ref = ref.detach().cpu().double()
    return float((a.detach().cpu().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def render_psf_map_ref(img, psf_map, grid):
    """deeplens/render_psf.py:31-73: per patch, reflect pad + grouped conv2d with the flipped PSF; zeros outside."""
    B, C, H, W = img.shape
    ks = psf_map.shape[-1] // grid
    p = (ks - 1) // 2
    pad = F.pad(img, (p, p, p, p), mode="reflect")
    out = torch.zeros_like(img)
    for i in range(grid):
        for j in range(grid):
            h0, h1 = int(i / grid * H), int((i + 1) / grid * H)
            w0, w1 = int(j / grid * W), int((j + 1) / grid * W)
            if h1 <= h0 or w1 <= w0:
                continue
            k = psf_map[:, i * ks:(i + 1) * ks, j * ks:(j + 1) * ks].flip(-2, -1).unsqueeze(1)
            out[:, :, h0:h1, w0:w1] = F.conv2d(pad[:, :, h0:h1 + 2 * p, w0:w1 + 2 * p], k, groups=C)
    return out


def check(what, got, ref, tol):
    """Assert relerr(got, ref) <= tol and print the observed value (pytest -s shows it)."""
    e = relerr(got, ref)
    print(f"relerr {what}: {e:.3g}")
    assert e <= tol, (what, e)


def oracle_grads(fn, img, psf, g):
    img64 = img.detach().double().requires_grad_(True)
    psf64 = psf.detach().double().requires_grad_(True)
    fn(img64, psf64).backward(g.double())
    return img64.grad, psf64.grad


def cuda_grads(fn, img, psf, g):
    img_c = img.detach().cuda().requires_grad_(True)
    psf_c = psf.detach().cuda().requires_grad_(True)
    fn(img_c, psf_c).backward(g.cuda())
    return img_c.grad, psf_c.grad


# --------------------------------------------------------------------------- local_psf_render
@pytest.mark.parametrize("ks", list(range(1, 35, 2)))
def test_local_psf_render_grads_vs_oracle(pkg, ks):
    """Every odd ks 1..33: W % 4 == 0 (strip dP kernel for ks 3..15, C <= 4) and W % 4 != 0, H and W smaller than
    ks (corners fold many clamped taps), C = 1, 3, 4, 5, N = 2."""
    from deeplens.render_psf import local_psf_render
    gen = torch.Generator().manual_seed(500 + ks)
    for (N, C, H, W) in [(2, 3, 21, 72), (2, 1, 13, 18), (2, 4, 5, 8), (2, 5, 7, 6), (2, 3, 3, 4)]:
        img = torch.rand(N, C, H, W, generator=gen)
        psf = torch.rand(N, H, W, ks, ks, generator=gen)
        g = torch.randn(N, C, H, W, generator=gen)
        ref_i, ref_p = oracle_grads(lambda a, b: orc.local_psf_render(a, b, ks), img, psf, g)
        gi, gp = cuda_grads(lambda a, b: local_psf_render(a, b, ks), img, psf, g)
        assert gi.shape == img.shape and gp.shape == psf.shape
        check(f"local dP ks={ks} {N}x{C}x{H}x{W}", gp, ref_p, TOL_PSF)
        check(f"local dimg ks={ks} {N}x{C}x{H}x{W}", gi, ref_i, TOL_IMG)


@pytest.mark.parametrize("ks,C", [(11, 3), (15, 4), (7, 5)])
def test_local_psf_render_strip_kernels_walk_many_rows_vs_oracle(pkg, ks, C):
    """8xCx256x300: N*H*ceil(W/64) = 10240 strip rows, so every warp of the strip dP and dimg kernels walks tens of
    rows (halo ring rotation, slot reuse after the bulk store has read it, source-row replay at run starts, runs that
    cross strip and image boundaries, a partial last strip).  C = 4 / 5: dimg in channel passes of 3 + 1 (+ 1); dP
    for C = 5 on the generic kernel."""
    from deeplens.render_psf import local_psf_render
    gen = torch.Generator().manual_seed(900 + ks)
    N, H, W = 8, 256, 300
    img = torch.rand(N, C, H, W, generator=gen)
    psf = torch.rand(N, H, W, ks, ks, generator=gen)
    g = torch.randn(N, C, H, W, generator=gen)
    ref_i, ref_p = oracle_grads(lambda a, b: orc.local_psf_render(a, b, ks), img, psf, g)
    gi, gp = cuda_grads(lambda a, b: local_psf_render(a, b, ks), img, psf, g)
    check(f"local dP ks={ks} {N}x{C}x{H}x{W}", gp, ref_p, TOL_PSF)
    check(f"local dimg ks={ks} {N}x{C}x{H}x{W}", gi, ref_i, TOL_IMG)


def test_local_psf_render_3d_input_and_flat_psf(pkg):
    """A [C,H,W] input and a psf given as [N,H,W,ks*ks]: gradients come back in those shapes."""
    from deeplens.render_psf import local_psf_render
    gen = torch.Generator().manual_seed(7)
    ks, C, H, W = 11, 3, 17, 40
    img = torch.rand(C, H, W, generator=gen)
    psf = torch.rand(1, H, W, ks * ks, generator=gen)
    g = torch.randn(1, C, H, W, generator=gen)
    ref_i, ref_p = oracle_grads(lambda a, b: orc.local_psf_render(a, b, ks), img, psf, g)
    gi, gp = cuda_grads(lambda a, b: local_psf_render(a, b, ks), img, psf, g)
    assert gi.shape == (C, H, W) and gp.shape == (1, H, W, ks * ks)
    assert relerr(gp, ref_p) <= TOL_PSF and relerr(gi, ref_i) <= TOL_IMG


# --------------------------------------------------------------------------- render_psf / render_psf_map
@pytest.mark.parametrize("ks", [3, 11, 31])
@pytest.mark.parametrize("C", [1, 3])
def test_render_psf_grads_vs_oracle(pkg, ks, C):
    from deeplens.render_psf import render_psf
    gen = torch.Generator().manual_seed(600 + ks + C)
    B, H, W = 2, 37, 45
    img = torch.rand(B, C, H, W, generator=gen)
    psf = torch.rand(C, ks, ks, generator=gen)
    g = torch.randn(B, C, H, W, generator=gen)
    ref_i, ref_p = oracle_grads(lambda a, b: render_psf_map_ref(a, b, 1), img, psf, g)
    gi, gp = cuda_grads(render_psf, img, psf, g)
    check(f"render_psf dK ks={ks} C={C}", gp, ref_p, TOL_PSF)
    check(f"render_psf dimg ks={ks} C={C}", gi, ref_i, TOL_IMG)


@pytest.mark.parametrize("ks", [3, 11, 31])
@pytest.mark.parametrize("grid", [2, 3, 32])
def test_render_psf_map_grads_vs_oracle(pkg, ks, grid):
    """Uneven int(i/grid*H) bounds, empty cells (grid 32 on small images), H and W just above 2p (several reflect
    preimages per pixel) and a larger image."""
    from deeplens.render_psf import render_psf_map
    gen = torch.Generator().manual_seed(700 + ks + grid)
    p = (ks - 1) // 2
    for (B, C, H, W) in [(2, 3, 2 * p + 2, 2 * p + 3), (1, 3, 70, 101)]:
        img = torch.rand(B, C, H, W, generator=gen)
        psf = torch.rand(C, grid * ks, grid * ks, generator=gen)
        g = torch.randn(B, C, H, W, generator=gen)
        ref_i, ref_p = oracle_grads(lambda a, b: render_psf_map_ref(a, b, grid), img, psf, g)
        gi, gp = cuda_grads(lambda a, b: render_psf_map(a, b, grid), img, psf, g)
        check(f"render_psf_map dK ks={ks} grid={grid} {B}x{C}x{H}x{W}", gp, ref_p, TOL_PSF)
        check(f"render_psf_map dimg ks={ks} grid={grid} {B}x{C}x{H}x{W}", gi, ref_i, TOL_IMG)


def test_render_psf_map_uint8_image_psf_grad(pkg):
    from deeplens.render_psf import render_psf_map
    rng = np.random.default_rng(3)
    img_u8 = rng.integers(0, 256, size=(40, 52, 3), dtype=np.uint8)
    ks, grid = 11, 3
    psf = torch.rand(3, grid * ks, grid * ks, generator=torch.Generator().manual_seed(3))
    img = torch.tensor((img_u8 / 255.).astype(np.float32)).permute(2, 0, 1).unsqueeze(0)
    g = torch.randn(1, 3, 40, 52, generator=torch.Generator().manual_seed(4))
    _, ref_p = oracle_grads(lambda a, b: render_psf_map_ref(a, b, grid), img, psf, g)
    psf_c = psf.cuda().requires_grad_(True)
    render_psf_map(img_u8, psf_c, grid).backward(g.cuda())
    assert relerr(psf_c.grad, ref_p) <= TOL_PSF


# --------------------------------------------------------------------------- contract
def _ops():
    from deeplens.render_psf import local_psf_render, render_psf_map
    gen = torch.Generator().manual_seed(11)
    lp = (lambda a, b: local_psf_render(a, b, 11), torch.rand(2, 3, 24, 64, generator=gen),
          torch.rand(2, 24, 64, 11, 11, generator=gen))
    pm = (lambda a, b: render_psf_map(a, b, 2), torch.rand(2, 3, 24, 64, generator=gen),
          torch.rand(3, 22, 22, generator=gen))
    return {"local_psf_render": lp, "render_psf_map": pm}


@pytest.mark.parametrize("op", ["local_psf_render", "render_psf_map"])
def test_only_the_requested_gradient_is_computed(pkg, op):
    """Only img (or only psf) requires grad: the other gradient is None and its kernel is not launched."""
    fn, img, psf = _ops()[op]
    lib = pkg.native.lib
    launches = {}
    for which in ("img", "psf", "both"):
        a = img.cuda().requires_grad_(which in ("img", "both"))
        b = psf.cuda().requires_grad_(which in ("psf", "both"))
        out = fn(a, b)
        torch.cuda.synchronize()
        n0 = lib.aadff_launch_count()
        out.sum().backward()
        torch.cuda.synchronize()
        launches[which] = lib.aadff_launch_count() - n0
        assert (a.grad is None) == (which == "psf") and (b.grad is None) == (which == "img")
    assert launches["img"] >= 1 and launches["psf"] >= 1
    assert launches["both"] == launches["img"] + launches["psf"]


@pytest.mark.parametrize("op", ["local_psf_render", "render_psf_map"])
def test_gradient_contract(pkg, op):
    """Non-contiguous grad_out, float64 inputs -> float64 gradients, a CPU psf -> a CPU gradient, and the forward
    output is bit-identical with and without requires_grad (and under no_grad)."""
    fn, img, psf = _ops()[op]
    plain = fn(img.cuda(), psf.cuda())
    with torch.no_grad():
        nograd = fn(img.cuda().requires_grad_(True), psf.cuda().requires_grad_(True))
    a, b = img.cuda().requires_grad_(True), psf.cuda().requires_grad_(True)
    out = fn(a, b)
    assert torch.equal(out.detach(), plain) and torch.equal(nograd, plain) and out.requires_grad
    g_nc = torch.randn(*img.shape[:-1], 2 * img.shape[-1], generator=torch.Generator().manual_seed(5))
    g_nc = g_nc.cuda()[..., ::2]                               # a strided grad_out
    assert not g_nc.is_contiguous()
    out.backward(g_nc)
    ref = cuda_grads(fn, img, psf, g_nc.contiguous())
    assert torch.equal(a.grad, ref[0]) and torch.equal(b.grad, ref[1])

    a64 = img.double().cuda().requires_grad_(True)
    b_cpu = psf.double().requires_grad_(True)
    fn(a64, b_cpu).sum().backward()
    assert a64.grad.dtype == torch.float64 and b_cpu.grad.dtype == torch.float64
    assert b_cpu.grad.device.type == "cpu" and a64.grad.is_cuda
    ones = torch.ones_like(img)
    ref = cuda_grads(fn, img, psf, ones)
    assert torch.equal(a64.grad.float(), ref[0]) and torch.equal(b_cpu.grad.float(), ref[1].cpu())


@pytest.mark.parametrize("op,ks", [("local_psf_render", 11), ("local_psf_render", 17), ("render_psf_map", 11)])
def test_backward_is_deterministic(pkg, op, ks):
    """5x3x96x320: every SM runs several warps' runs across strip and image boundaries; two backward passes are
    bit-identical."""
    from deeplens.render_psf import local_psf_render, render_psf_map
    gen = torch.Generator().manual_seed(13)
    img = torch.rand(5, 3, 96, 320, generator=gen).cuda()
    g = torch.randn(5, 3, 96, 320, generator=gen).cuda()
    if op == "local_psf_render":
        psf = torch.rand(5, 96, 320, ks, ks, generator=gen).cuda()
        fn = lambda a, b: local_psf_render(a, b, ks)
    else:
        psf = torch.rand(3, 8 * ks, 8 * ks, generator=gen).cuda()
        fn = lambda a, b: render_psf_map(a, b, 8)
    r1 = cuda_grads(fn, img, psf, g)
    r2 = cuda_grads(fn, img, psf, g)
    assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])


@pytest.mark.parametrize("N,C,ks", [(9, 3, 31), (40, 1, 15)])
def test_local_psf_render_grads_past_2_31_elements(pkg, N, C, ks):
    """More than 2^31 PSF elements (generic dP kernel at ks = 31, strip dP kernel at ks = 15): gradient elements
    past the 2^31 offset against the direct formula."""
    from deeplens.render_psf import local_psf_render
    H = W = 512
    r = (ks - 1) // 2
    assert N * H * W * ks * ks > 2 ** 31
    torch.manual_seed(17)
    img = torch.rand(N, C, H, W, device="cuda", requires_grad=True)
    psf = torch.rand(N, H, W, ks, ks, device="cuda", requires_grad=True)
    g = torch.randn(N, C, H, W, device="cuda")
    local_psf_render(img, psf, ks).backward(g)
    dP = psf.grad.view(-1)
    kk = ks * ks
    for flat in [2 ** 31 + 5, 2 ** 31 + 12345 * kk + 7, dP.numel() - 1]:
        px, t = divmod(flat, kk)
        n, hw = divmod(px, H * W)
        h, w = divmod(hw, W)
        i, j = divmod(t, ks)
        y, x = min(max(h + i - r, 0), H - 1), min(max(w + j - r, 0), W - 1)
        want = (g[n, :, h, w].double() * img.detach()[n, :, y, x].double()).sum()
        assert abs(float(dP[flat]) - float(want)) <= 1e-5 * max(1.0, abs(float(want))), flat
    n = N - 1                                                  # last image: its P offsets are past 2^31
    P = psf.detach()[n].double()
    taps = torch.arange(ks, device="cuda")
    for (y, x) in [(200, 300), (0, 0), (H - 1, 77)]:
        hs = torch.arange(max(0, y - r), min(H, y + r + 1), device="cuda")
        ws = torch.arange(max(0, x - r), min(W, x + r + 1), device="cuda")
        my = ((hs[:, None] + taps[None, :] - r).clamp(0, H - 1) == y).double()      # [h, i]
        mx = ((ws[:, None] + taps[None, :] - r).clamp(0, W - 1) == x).double()      # [w, j]
        Pw = P[hs[0]:hs[-1] + 1, ws[0]:ws[-1] + 1]                                  # [h, w, i, j]
        gw = g[n, :, hs[0]:hs[-1] + 1, ws[0]:ws[-1] + 1].double()                   # [c, h, w]
        want = torch.einsum("chw,hwij,hi,wj->c", gw, Pw, my, mx)
        got = img.grad[n, :, y, x].double()
        assert float((got - want).abs().max()) <= 2e-5 * max(1.0, float(want.abs().max())), (y, x)


@pytest.mark.parametrize("op", ["local_psf_render", "render_psf_map"])
def test_forward_and_backward_are_cuda_graph_capturable(pkg, op):
    fn, img, psf = _ops()[op]
    a, b = img.cuda().requires_grad_(True), psf.cuda().requires_grad_(True)
    g = torch.randn_like(a)
    eager = cuda_grads(fn, img, psf, g)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):                                     # warm-up on the capture stream
            a.grad = b.grad = None
            fn(a, b).backward(g)
    torch.cuda.current_stream().wait_stream(side)
    a.grad = b.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn(a, b).backward(g)
    a.grad.zero_()
    b.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(a.grad, eager[0]) and torch.equal(b.grad, eager[1])
