"""Gradients of ``PSFNet.render`` / ``render_stack`` with differentiable=True (aadff_render_stack_backward_f32,
csrc/render_grad_kernel.cuh) against float64 autograd through the reference's definition (oracle/render_grad_oracle.py),
against the hand-built chain lens.psfnet(probes) -> local_psf_render -> backward(), and the autograd contract: output
bit-identical to the no-grad path, grad_img independent of the other requested gradients, exact zeros on depth2z's
clamp, empty batch, accumulation, frozen layers, version checks, handle rebuilds, determinism across calls and streams,
CUDA-graph capture, and an Adam loop recovering an all-in-focus image.

Tolerances (max |ours - float64| over each tensor's largest element): 1e-5 for every gradient of the fp32 chain
(ddepth, dfoc, dW, db; as for the MLP backward), and for dimg in mode fp32.  dimg in the tensor-core modes is held to
each mode's own bound (DIMG_TOL): its PSFs are the forward's, whose error against float64 it inherits.
Depths come from the oracle's sampler, which keeps the fp32 and float64 forwards on the same ReLU and clamp branches.
With AADFF_GRAD_REPORT=<path> the largest observed error of every case is written there as JSON."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import focal_stack_oracle as orc
from oracle import render_grad_oracle as rgo
from oracle import train_oracle as tor

pytestmark = pytest.mark.gpu

CKPT = os.path.join(os.path.dirname(__file__), "golden", "rf50mm_PSFNet480x640_ks11.pkl")
TOL = 1e-5
# dimg against float64 per mode, rf50mm, 2 x 40 x 56 (B200 at 1000 W): fp32 4.3e-7, parity 4.4e-6, econ8 1.2e-5,
# econ 1.6e-5, mixed 1.6e-4, fast 3.9e-4 of the largest element
# dfoc sums H*W terms of either sign: with a random-sign (L1) upstream gradient the sum cancels far below its terms, and
# its largest element is a poor scale (1.79e-5 of a 5.0e-10 maximum observed at 15 x 18, S = 1)
DFOC_TOL = 4e-5
DIMG_TOL = {"fp32": 1e-5, "parity": 1e-5, "econ8": 3e-5, "econ": 4e-5, "mixed": 5e-4, "fast": 2e-3}
REPORT = {}


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    path = os.environ.get("AADFF_GRAD_REPORT")
    if path:
        os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
        with open(path, "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import aadff_b200
    return aadff_b200


def make_lens(pkg, Ws, bs, mode="fp32"):
    """A PSFNet whose MLP holds (Ws, bs): hidden layers = len(Ws) - 3."""
    from aadff_arch import MLP
    ks = int(round(np.sqrt(Ws[-1].shape[0])))
    lens = pkg.PSFNet(kernel_size=ks, device="cuda", mode=mode)
    lens.psfnet = MLP(in_features=4, out_features=ks * ks, hidden_features=256, hidden_layers=len(Ws) - 3).to("cuda")
    lens.psfnet._evaluator = lens._mlp_eval
    with torch.no_grad():
        for lin, W, b in zip(lens.psfnet.linear_layers(), Ws, bs):
            lin.weight.copy_(torch.as_tensor(np.asarray(W)))
            lin.bias.copy_(torch.as_tensor(np.asarray(b)))
    return lens


def rf50mm():
    Ws, bs = orc.split_state_dict(torch.load(CKPT, map_location="cpu"))
    return [w.numpy() for w in Ws], [b.numpy() for b in bs]


def seeded(ks, hidden, seed):
    gen = torch.Generator().manual_seed(seed)
    return tor.kaiming_net([4, 64, 256] + [256] * hidden + [ks * ks], gen, bias_scale=0.1)


def kaiming(ks, seed):
    gen = torch.Generator().manual_seed(seed)
    return tor.kaiming_net([4, 64, 256] + [256] * 8 + [ks * ks], gen)


def inputs(Ws, bs, N, C, S, H, W, seed, fixed=None):
    """img U[0,1] [N,C,H,W], depth [N,1,H,W] and foc [N,S] in mm from the oracle's sampler (float64 on the GPU)."""
    gen = torch.Generator().manual_seed(seed)
    foc_z = 0.05 + 0.9 * torch.rand(N, S, generator=gen, dtype=torch.float64)
    depth, foc = rgo.sample_depths(Ws, bs, N, H, W, foc_z, gen, fixed=fixed, dev="cuda")
    img = torch.rand(N, C, H, W, generator=gen)
    return img.cuda(), depth.view(N, 1, H, W).cuda(), foc.cuda()


def upstream(kind, out64, gen):
    """dL/dout for a random upstream gradient, an MSE or an L1 loss against random targets ([N,C,S,H,W] float64)."""
    if kind == "random":
        return torch.randn(out64.shape, generator=gen, dtype=torch.float64).to(out64.device)
    t = torch.rand(out64.shape, generator=gen, dtype=torch.float64).to(out64.device)
    if kind == "mse":
        return 2.0 * (out64 - t) / out64.numel()
    return torch.sign(out64 - t) / out64.numel()


def to_layout(G, layout):
    """[N,C,S,H,W] -> the layout of the output: BCSHW, BSCHW or NCHW (render, S = 1)."""
    if layout == "BSCHW":
        return G.permute(0, 2, 1, 3, 4).contiguous()
    if layout == "NCHW":
        return G[:, :, 0].contiguous()
    return G


def ours(lens, img, depth, foc, G, layout="BCSHW", mode=None, need=("img", "depth", "foc", "params")):
    """-> (out, grads dict) of render_stack (or render for layout NCHW) with differentiable=True."""
    x = img.clone().requires_grad_("img" in need)
    d = depth.clone().requires_grad_("depth" in need)
    f = foc.clone().requires_grad_("foc" in need)
    for p in lens.psfnet.parameters():
        p.grad = None
        p.requires_grad_("params" in need)
    if layout == "NCHW":
        out = lens.render(x, d, f[:, 0], mode=mode, differentiable=True)
    else:
        out = lens.render_stack(x, d, f, layout=layout, mode=mode, differentiable=True)
    out.backward(to_layout(G, layout).to(torch.float32))
    lins = lens.psfnet.linear_layers()
    for p in lens.psfnet.parameters():
        p.requires_grad_(True)
    return out.detach(), {"img": x.grad, "depth": None if d.grad is None else d.grad[:, 0], "foc": f.grad,
                          "W": [l.weight.grad for l in lins], "b": [l.bias.grad for l in lins]}


def reference(Ws, bs, img, depth, foc, ks, kind, seed):
    """float64 gradients for the upstream gradient `kind` -> (G [N,C,S,H,W] float64, grads dict)."""
    N, _, H, W = depth.shape
    d = depth.view(N, H, W).double()
    out64 = rgo.render_stack_f64([torch.as_tensor(w) for w in Ws], [torch.as_tensor(b) for b in bs], img.double(), d,
                                 foc.double(), ks)
    G = upstream(kind, out64, torch.Generator().manual_seed(seed))
    return G, rgo.grads_f64(Ws, bs, img, d, foc, ks, G)


def compare(case, got, ref, dimg_tol=TOL, tol=TOL, names=None):
    """max |got - ref| / max |ref| per tensor, asserted; records the worst of the fp32 chain and of dimg in REPORT."""
    names = names or ["img", "depth", "foc"] + [f"W{l}" for l in range(len(ref["W"]))] + \
        [f"b{l}" for l in range(len(ref["b"]))]
    worst, worst_img = 0.0, 0.0
    for name in names:
        if name[0] in "Wb" and name[1:].isdigit():
            a, r = got[name[0]][int(name[1:])], ref[name[0]][int(name[1:])]
        else:
            a, r = got[name], ref[name]
        r = r.to("cuda", torch.float64)
        a = a.to(torch.float64)
        assert a.shape == r.shape, f"{case} {name}: shape {tuple(a.shape)} != {tuple(r.shape)}"
        if not r.numel():
            continue
        scale = float(r.abs().max())
        if scale == 0.0:
            assert float(a.abs().max()) == 0.0, f"{case} {name}: reference is 0"
            continue
        err = float((a - r).abs().max()) / scale
        bound = dimg_tol if name == "img" else DFOC_TOL if name == "foc" else tol
        assert err <= bound, f"{case} d{name}: {err:.3e} of max {scale:.3e} (bound {bound:.1e})"
        if name == "img":
            worst_img = max(worst_img, err)
        else:
            worst = max(worst, err)
    REPORT[case] = {"chain": worst, "dimg": worst_img}


def run_case(pkg, case, Ws, bs, N, C, S, H, W, seed, kind="random", layout="BCSHW", mode="fp32"):
    ks = int(round(np.sqrt(Ws[-1].shape[0])))
    img, depth, foc = inputs(Ws, bs, N, C, S, H, W, seed)
    G, ref = reference(Ws, bs, img, depth, foc, ks, kind, seed + 1)
    lens = make_lens(pkg, Ws, bs, mode)
    out, got = ours(lens, img, depth, foc, G, layout)
    # at ks = 1 the PSF is the constant 1: only dimg is nonzero, and every other gradient is fp32 round-off of 0
    compare(case, got, ref, dimg_tol=DIMG_TOL[mode], names=["img"] if ks == 1 else None)
    return out, ref


# ---------------------------------------------------------------------------------------------- against float64
@pytest.mark.parametrize("ks", list(range(1, 32, 2)))
def test_every_kernel_size_vs_f64(pkg, ks):
    Ws, bs = seeded(ks, 2, 100 + ks)
    run_case(pkg, f"ks{ks}", Ws, bs, 1, 3, 2, 11, 13, seed=ks)


@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("S", [1, 5])
@pytest.mark.parametrize("C", [1, 3, 4, 5])
def test_batch_slices_channels_vs_f64(pkg, N, S, C):
    Ws, bs = seeded(7, 2, 7)
    run_case(pkg, f"N{N}_S{S}_C{C}", Ws, bs, N, C, S, 9, 10, seed=N * 100 + S * 10 + C)


@pytest.mark.parametrize("H,W,ks", [(170, 100, 5), (130, 129, 3), (3, 16384, 3), (40, 16384 // 3 + 1, 7),
                                    (17, 23, 31)])
def test_band_edges_vs_f64(pkg, H, W, ks):
    """Bands of floor(16384 / W) rows: the last band ragged, one-row bands, and a PSF wider than the band."""
    Ws, bs = seeded(ks, 1, H + W)
    run_case(pkg, f"band_{H}x{W}_ks{ks}", Ws, bs, 1, 3, 2, H, W, seed=H * W)


def test_full_frame_rf50mm_vs_f64(pkg):
    Ws, bs = rf50mm()
    run_case(pkg, "rf50mm_480x640", Ws, bs, 1, 3, 1, 480, 640, seed=5)


def test_from_scratch_init_vs_f64(pkg):
    Ws, bs = kaiming(11, 3)
    run_case(pkg, "kaiming_ks11", Ws, bs, 2, 3, 3, 24, 20, seed=3)


@pytest.mark.parametrize("kind", ["random", "mse", "l1"])
@pytest.mark.parametrize("layout", ["BCSHW", "BSCHW", "NCHW"])
def test_upstream_and_layouts_vs_f64(pkg, kind, layout):
    Ws, bs = seeded(9, 3, 9)
    S = 1 if layout == "NCHW" else 3
    run_case(pkg, f"{kind}_{layout}", Ws, bs, 2, 3, S, 15, 18, seed=len(kind) * 7 + len(layout), kind=kind,
             layout=layout)


@pytest.mark.parametrize("mode", ["parity", "econ8", "econ", "mixed", "fast", "fp32"])
def test_each_mode_vs_f64(pkg, mode):
    """rf50mm (the tensor-core modes need its 8 hidden layers): dimg to the mode's bound, the fp32 chain to 1e-5."""
    Ws, bs = rf50mm()
    run_case(pkg, f"mode_{mode}", Ws, bs, 1, 3, 2, 40, 56, seed=17, mode=mode)


@pytest.mark.parametrize("mode", ["parity", "econ8", "econ", "mixed", "fast", "fp32"])
def test_adjoint_each_mode(pkg, mode):
    """<render_stack(x), G> = <x, dimg(G)>: the image gradient is the transpose of the forward, within fp32 rounding."""
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs, mode)
    img, depth, foc = inputs(Ws, bs, 2, 3, 3, 33, 47, seed=23)
    G = torch.randn(2, 3, 3, 33, 47, generator=torch.Generator().manual_seed(2), dtype=torch.float64).cuda()
    out, got = ours(lens, img, depth, foc, G, need=("img",))
    lhs = float((out.double() * G).sum())
    rhs = float((img.double() * got["img"].double()).sum())
    mag = float((out.double().abs() * G.abs()).sum())
    REPORT[f"adjoint_{mode}"] = abs(lhs - rhs) / mag
    assert abs(lhs - rhs) <= 1e-6 * mag, (lhs, rhs, mag)


# ---------------------------------------------------------------------------------------------- hand-built chain
def hand_chain(pkg, lens, img, depth, foc, G):
    """lens.psfnet(probes) -> local_psf_render -> backward(), one slice at a time (mode fp32)."""
    N, C, H, W = img.shape
    S = foc.shape[1]
    ks = lens.kernel_size
    x = img.clone().requires_grad_(True)
    d = depth.clone().requires_grad_(True)
    f = foc.clone().requires_grad_(True)
    for p in lens.psfnet.parameters():
        p.grad = None
    xs = torch.from_numpy(orc.linspace_f32(-1.0, 1.0, W)).cuda().view(1, 1, W).expand(N, H, W)
    ys = torch.from_numpy(orc.linspace_f32(1.0, -1.0, H)).cuda().view(1, H, 1).expand(N, H, W)
    z = torch.clamp((d[:, 0] - lens.d_min) / (lens.d_max - lens.d_min), 0, 1)
    outs = []
    for s in range(S):
        fz = torch.clamp((f[:, s] - lens.d_min) / (lens.d_max - lens.d_min), 0, 1).view(N, 1, 1).expand(N, H, W)
        psf = lens.psfnet(torch.stack((xs, ys, z, fz), -1))
        outs.append(pkg.local_psf_render(x, psf.view(N, H, W, ks, ks), ks))
    out = torch.stack(outs, 2)
    out.backward(G.to(torch.float32))
    lins = lens.psfnet.linear_layers()
    return out.detach(), {"img": x.grad, "depth": d.grad[:, 0], "foc": f.grad,
                          "W": [l.weight.grad.clone() for l in lins], "b": [l.bias.grad.clone() for l in lins]}


def test_cross_check_hand_built_chain(pkg):
    Ws, bs = seeded(11, 3, 31)
    lens = make_lens(pkg, Ws, bs, "fp32")
    img, depth, foc = inputs(Ws, bs, 2, 3, 3, 37, 41, seed=31)
    G = torch.randn(2, 3, 3, 37, 41, generator=torch.Generator().manual_seed(4), dtype=torch.float64).cuda()
    out_h, hand = hand_chain(pkg, lens, img, depth, foc, G)
    out_o, got = ours(lens, img, depth, foc, G)
    REPORT["hand_chain_out"] = float((out_o - out_h).abs().max())
    assert float((out_o - out_h).abs().max()) <= 1e-6
    compare("hand_chain", got, hand)


def test_adam_recovers_aif_like_hand_chain(pkg):
    """10 Adam steps on the all-in-focus image from a rendered 5-slice stack: the same trajectory as the hand chain."""
    Ws, bs = seeded(7, 2, 41)
    lens = make_lens(pkg, Ws, bs, "fp32")
    for p in lens.psfnet.parameters():
        p.requires_grad_(False)
    img, depth, foc = inputs(Ws, bs, 1, 3, 5, 48, 64, seed=41)
    with torch.no_grad():
        target = lens.render_stack(img, depth, foc)
    N, C, H, W = img.shape
    ks = lens.kernel_size
    xs = torch.from_numpy(orc.linspace_f32(-1.0, 1.0, W)).cuda().view(1, 1, W).expand(N, H, W)
    ys = torch.from_numpy(orc.linspace_f32(1.0, -1.0, H)).cuda().view(1, H, 1).expand(N, H, W)
    z = torch.clamp((depth[:, 0] - lens.d_min) / (lens.d_max - lens.d_min), 0, 1)
    with torch.no_grad():
        psfs = [lens.psfnet(torch.stack((xs, ys, z, torch.clamp((foc[:, s] - lens.d_min) / (lens.d_max - lens.d_min),
                                                                 0, 1).view(N, 1, 1).expand(N, H, W)), -1))
                .view(N, H, W, ks, ks) for s in range(5)]

    def run(render):
        x = torch.full_like(img, 0.5).requires_grad_(True)
        opt = torch.optim.Adam([x], lr=0.05)
        losses = []
        for _ in range(10):
            opt.zero_grad()
            loss = ((render(x) - target) ** 2).mean()
            loss.backward()
            opt.step()
            losses.append(float(loss))
        return x.detach(), losses

    x_o, l_o = run(lambda x: lens.render_stack(x, depth, foc, differentiable=True))
    x_h, l_h = run(lambda x: torch.stack([pkg.local_psf_render(x, p, ks) for p in psfs], 2))
    dx = float((x_o - x_h).abs().max())
    dl = max(abs(a - b) / b for a, b in zip(l_o, l_h))
    REPORT["adam_traj"] = {"x": dx, "loss_rel": dl}
    assert l_o[-1] < 0.5 * l_o[0]
    # measured on a B200 at 1000 W: images 1.8e-6 apart, losses 1.9e-7 relative
    assert dx <= 1e-5 and dl <= 1e-6, (dx, dl)


# ---------------------------------------------------------------------------------------------- contract
@pytest.mark.parametrize("mode", ["parity", "econ8", "fp32", "fast"])
def test_output_bit_identical_to_no_grad(pkg, mode):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs, mode)
    img, depth, foc = inputs(Ws, bs, 2, 3, 3, 24, 40, seed=8)
    with torch.no_grad():
        ref = lens.render_stack(img, depth, foc)
        ref1 = lens.render(img, depth, foc[:, 1])
    x = img.clone().requires_grad_(True)
    out = lens.render_stack(x, depth, foc, differentiable=True)
    assert out.requires_grad and torch.equal(out, ref)
    assert torch.equal(lens.render(x, depth, foc[:, 1], differentiable=True), ref1)
    assert torch.equal(lens.render_stack(x, depth, foc, differentiable=False), ref)
    assert not lens.render_stack(x, depth, foc).requires_grad
    # one image with a 1-D row of focus distances, as the no-grad path accepts it
    with torch.no_grad():
        ref0 = lens.render_stack(img[:1], depth[:1], foc[0])
    assert torch.equal(lens.render_stack(x[:1], depth[:1], foc[0], differentiable=True), ref0)
    with torch.no_grad():
        o2 = lens.render_stack(x, depth, foc, differentiable=True)
    assert not o2.requires_grad and torch.equal(o2, ref)


@pytest.mark.parametrize("mode", ["parity", "econ", "fp32"])
def test_grad_img_independent_of_request(pkg, mode):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs, mode)
    img, depth, foc = inputs(Ws, bs, 2, 4, 2, 19, 31, seed=9)
    G = torch.randn(2, 4, 2, 19, 31, generator=torch.Generator().manual_seed(9), dtype=torch.float64).cuda()
    base = ours(lens, img, depth, foc, G, need=("img",))[1]["img"]
    for need in [("img", "depth"), ("img", "foc"), ("img", "params"), ("img", "depth", "foc", "params")]:
        assert torch.equal(ours(lens, img, depth, foc, G, need=need)[1]["img"], base), need


def test_clamped_and_invalid_depths_get_exact_zeros(pkg):
    Ws, bs = seeded(5, 2, 12)
    N, H, W = 2, 12, 14
    mask = torch.zeros(N, H, W, dtype=torch.bool)
    val = torch.zeros(N, H, W)
    for (n, h, w), v in {(0, 0, 0): 0.0, (0, 5, 6): -100.0, (1, 11, 13): -30000.0, (1, 3, 4): 0.0}.items():
        mask[n, h, w] = True
        val[n, h, w] = v
    img, depth, foc = inputs(Ws, bs, N, 3, 3, H, W, seed=12, fixed=(mask, val))
    foc[1, 2] = -25000.0            # focus beyond d_max: its z is clamped to 1
    foc[0, 1] = -150.0              # nearer than d_min: clamped to 0
    lens = make_lens(pkg, Ws, bs, "fp32")
    G = torch.randn(N, 3, 3, H, W, generator=torch.Generator().manual_seed(1), dtype=torch.float64).cuda()
    _, got = ours(lens, img, depth, foc, G)
    assert bool((got["depth"][mask.cuda()] == 0).all())
    assert float(got["foc"][1, 2]) == 0.0 and float(got["foc"][0, 1]) == 0.0
    assert bool((got["depth"][~mask.cuda()] != 0).any()) and float(got["foc"][0, 0]) != 0.0
    ref = rgo.grads_f64(Ws, bs, img, depth.view(N, H, W).double(), foc.double(), 5, G)
    compare("clamp_zeros", got, ref)


def test_empty_batch(pkg):
    Ws, bs = seeded(5, 1, 2)
    lens = make_lens(pkg, Ws, bs, "fp32")
    x = torch.rand(0, 3, 8, 8, device="cuda", requires_grad=True)
    out = lens.render_stack(x, -1000 * torch.ones(0, 1, 8, 8, device="cuda"), -900 * torch.ones(0, 2, device="cuda"),
                            differentiable=True)
    out.sum().backward()
    assert x.grad.shape == x.shape
    assert all(float(p.grad.abs().max()) == 0.0 for p in lens.psfnet.parameters())


def test_accumulation_dtypes_and_frozen_layers(pkg):
    Ws, bs = seeded(5, 2, 13)
    lens = make_lens(pkg, Ws, bs, "fp32")
    img, depth, foc = inputs(Ws, bs, 1, 3, 2, 10, 12, seed=13)
    G = torch.randn(1, 3, 2, 10, 12, generator=torch.Generator().manual_seed(3), dtype=torch.float64).cuda()
    _, full = ours(lens, img, depth, foc, G)
    lins = lens.psfnet.linear_layers()
    lins[0].weight.requires_grad_(False)
    lins[2].bias.requires_grad_(False)
    x = img.double().cpu().requires_grad_(True)            # another dtype and device: gradients come back there
    d = depth.double().requires_grad_(True)
    for p in lens.psfnet.parameters():
        p.grad = None
    for _ in range(2):
        lens.render_stack(x, d, foc, differentiable=True).backward(G.float())
    assert x.grad.dtype == torch.float64 and x.grad.device.type == "cpu" and d.grad.shape == (1, 1, 10, 12)
    torch.testing.assert_close(x.grad.float().cuda(), 2 * full["img"], rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(d.grad[:, 0].float(), 2 * full["depth"], rtol=1e-5, atol=1e-12)
    assert lins[0].weight.grad is None and lins[2].bias.grad is None
    torch.testing.assert_close(lins[1].weight.grad, 2 * full["W"][1], rtol=1e-6, atol=0)
    for p in lens.psfnet.parameters():
        p.requires_grad_(True)


def test_version_check_and_handle_rebuild(pkg):
    Ws, bs = seeded(5, 2, 14)
    lens = make_lens(pkg, Ws, bs, "fp32")
    img, depth, foc = inputs(Ws, bs, 1, 3, 2, 10, 12, seed=14)
    G = torch.randn(1, 3, 2, 10, 12, generator=torch.Generator().manual_seed(5), dtype=torch.float64).cuda()
    _, ref = ours(lens, img, depth, foc, G)
    x = img.clone().requires_grad_(True)
    out = lens.render_stack(x, depth, foc, differentiable=True)
    with torch.no_grad():
        x.add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        out.backward(G.float())
    # the handle the forward ran on is rebuilt before the backward: the graph keeps the old one alive
    x = img.clone().requires_grad_(True)
    for p in lens.psfnet.parameters():
        p.grad = None
    out = lens.render_stack(x, depth, foc, differentiable=True)
    lens.refresh()
    lens.native()
    out.backward(G.float())
    assert torch.equal(x.grad, ref["img"])
    assert torch.equal(lens.psfnet.linear_layers()[0].weight.grad, ref["W"][0])


def test_deterministic_across_calls_and_streams(pkg):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs, "parity")
    img, depth, foc = inputs(Ws, bs, 1, 3, 2, 64, 300, seed=15)      # several bands per slice
    G = torch.randn(1, 3, 2, 64, 300, generator=torch.Generator().manual_seed(6), dtype=torch.float64).cuda()
    a = ours(lens, img, depth, foc, G)[1]
    b = ours(lens, img, depth, foc, G)[1]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = ours(lens, img, depth, foc, G)[1]
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    for o in (b, c):
        for k in ("img", "depth", "foc"):
            assert torch.equal(a[k], o[k]), k
        for k in ("W", "b"):
            assert all(torch.equal(u, v) for u, v in zip(a[k], o[k])), k


@pytest.mark.parametrize("mode", ["parity", "econ", "fp32"])
def test_cuda_graph_capture(pkg, mode):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs, mode)
    img, depth, foc = inputs(Ws, bs, 1, 3, 2, 32, 40, seed=16)
    G = torch.randn(1, 3, 2, 32, 40, generator=torch.Generator().manual_seed(7)).cuda()
    x = img.clone().requires_grad_(True)
    lens.render_stack(x, depth, foc, differentiable=True).backward(G)        # warm-up (econ calibrates here)
    ref = x.grad.clone()
    refW = lens.psfnet.linear_layers()[-1].weight.grad.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x.grad = None
        for p in lens.psfnet.parameters():
            p.grad = None
        lens.render_stack(x, depth, foc, differentiable=True).backward(G)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    x.grad = None
    for p in lens.psfnet.parameters():
        p.grad = None
    with torch.cuda.graph(g):
        out = lens.render_stack(x, depth, foc, differentiable=True)
        out.backward(G)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(x.grad, ref)
    assert torch.equal(lens.psfnet.linear_layers()[-1].weight.grad, refW)
