"""Gradients of ``lens.psfnet(inp)`` (aadff_psfnet_backward_f32, csrc/mlp_grad_kernel.cuh) against float64 autograd
through the reference's operators (oracle/mlp_grad_oracle.py: grads_f64), and the autograd contract of the
differentiable path: forward bit-identical to the no-grad path, frozen layers, dtypes and devices, accumulation,
version checks, handle lifetime, determinism, CUDA-graph capture, the fitting step's own gradients, and the chain
psfnet -> local_psf_render -> image loss.

Tolerance: every gradient tensor within 1e-5 of its largest element (as the fitting-step tests), widened in two
places where a B200 run measured more:
  - a random-sign upstream gradient summed over M probes: the result grows as sqrt(M) while the rounding of the sum
    grows with M, so the bound is 1e-5 * sqrt(M / 8192) above 8192 probes (1.19e-5 observed at M = 32785);
  - both sides of the normalisation clamp: there s = sigmoid(z) ~ exp(z) with z ~ -31, where the forward's own fp32
    rounding of z moves s by ~1e-5 relative; bound 2.5e-5 (2.0e-5 observed).
Probes come from the oracle's sampler, which keeps the fp32 and float64 forwards on the same ReLU and clamp branches.
With AADFF_GRAD_REPORT=<path> the largest observed error of every case is written there as JSON."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import focal_stack_oracle as orc
from oracle import mlp_grad_oracle as mgo
from oracle import train_oracle as tor

pytestmark = pytest.mark.gpu

CKPT = os.path.join(os.path.dirname(__file__), "golden", "rf50mm_PSFNet480x640_ks11.pkl")
CHUNK = 16384           # MG_CHUNK of csrc/mlp_grad_kernel.cuh: probes per recompute chunk
TOL = 1e-5
CLAMP_TOL = 2.5e-5
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


def make_lens(pkg, Ws, bs):
    """A PSFNet whose MLP holds (Ws, bs): hidden layers = len(Ws) - 3."""
    from aadff_arch import MLP
    ks = int(round(np.sqrt(Ws[-1].shape[0])))
    lens = pkg.PSFNet(kernel_size=ks, device="cuda")
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


def sample_probes_dev(Ws, bs, M, gen, dev="cuda"):
    """oracle.train_oracle.sample_probes with the float64 forward on the GPU (for M in the hundreds of thousands)."""
    Wd = [torch.as_tensor(np.asarray(w)).to(dev, torch.float64) for w in Ws]
    bd = [torch.as_tensor(np.asarray(b)).to(dev, torch.float64) for b in bs]
    inp = torch.from_numpy(tor.draw_probes(M, gen)).to(dev)
    for _ in range(100):
        pre, S, _ = tor.forward_f64(Wd, bd, inp)
        ok = (S - tor.NORMALIZE_EPS).abs() >= tor.CLAMP_MARGIN * tor.NORMALIZE_EPS
        for z in pre:
            a = z.abs()
            ok &= (a >= tor.RELU_MARGIN * a.amax(-1, keepdim=True)).all(-1) & (a.amax(-1) > 0)
        bad = torch.nonzero(~ok).flatten()
        if bad.numel() == 0:
            return inp
        inp[bad] = torch.from_numpy(tor.draw_probes(bad.numel(), gen)).to(dev)
    raise RuntimeError("sample_probes_dev: margins not reached")


def upstream(kind, p64, gen):
    """dL/dp for a random upstream gradient, an MSE loss or an L1 loss against random targets."""
    M, kk = p64.shape
    if kind == "random":
        return torch.randn(M, kk, generator=gen, dtype=torch.float64).to(p64.device)
    t = torch.from_numpy(tor.random_targets(M, kk, gen)).to(p64.device, torch.float64)
    if kind == "mse":
        return 2.0 * (p64 - t) / (M * kk)
    return torch.sign(p64 - t) / (M * kk)


def grads_ours(lens, inp, g):
    x = inp.detach().to("cuda", torch.float32).clone().requires_grad_(True)
    for p in lens.psfnet.parameters():
        p.grad = None
    psf = lens.psfnet(x)
    psf.backward(g.to("cuda", torch.float32))
    lins = lens.psfnet.linear_layers()
    return [l.weight.grad for l in lins], [l.bias.grad for l in lins], x.grad


def compare(case, ours, ref, exact_zero_dead=False, tol=TOL):
    """max |ours - ref| / max |ref| per tensor, asserted <= tol; records the worst in REPORT."""
    dWs, dbs, dX = ours
    rW, rb, rX = ref
    worst = 0.0
    names = [f"dW{l}" for l in range(len(dWs))] + [f"db{l}" for l in range(len(dbs))] + ["dX"]
    for name, a, r in zip(names, list(dWs) + list(dbs) + [dX], list(rW) + list(rb) + [rX]):
        r = r.to("cuda", torch.float64)
        a = a.to(torch.float64)
        scale = float(r.abs().max())
        if scale == 0.0:
            assert float(a.abs().max()) == 0.0, f"{case} {name}: reference is 0, ours {float(a.abs().max()):.3e}"
            continue
        err = float((a - r).abs().max()) / scale
        worst = max(worst, err)
        assert err <= tol, f"{case} {name}: {err:.3e} of max {scale:.3e} (bound {tol:.2e})"
        if exact_zero_dead:
            assert bool((a[r == 0] == 0).all()), f"{case} {name}: dead units got nonzero gradients"
    REPORT[case] = worst
    return worst


def random_tol(M):
    return TOL * max(1.0, (M / 8192) ** 0.5)


def run_case(pkg, case, Ws, bs, M, kind, seed, exact_zero_dead=False, probes=None, tol=None):
    gen = torch.Generator().manual_seed(seed)
    if tol is None:
        tol = random_tol(M) if kind == "random" else TOL
    lens = make_lens(pkg, Ws, bs)
    inp = probes if probes is not None else (
        sample_probes_dev(Ws, bs, M, gen) if M > 4096 else torch.from_numpy(tor.sample_probes(Ws, bs, M, gen)[0]).cuda())
    _, _, p64 = tor.forward_f64([torch.as_tensor(np.asarray(w)).cuda() for w in Ws],
                                [torch.as_tensor(np.asarray(b)).cuda() for b in bs], inp)
    g = upstream(kind, p64, gen)
    ref = mgo.grads_f64([torch.as_tensor(np.asarray(w)).cuda() for w in Ws],
                        [torch.as_tensor(np.asarray(b)).cuda() for b in bs], inp, g)
    return compare(case, grads_ours(lens, inp, g), ref, exact_zero_dead, tol), lens, inp, g


# ---------------------------------------------------------------------------------------------------- 1. vs float64
@pytest.mark.parametrize("ks", [1, 3, 5, 11, 13, 17, 31])
@pytest.mark.parametrize("kind", ["random", "mse", "l1"])
def test_kernel_sizes_vs_f64(pkg, ks, kind):
    Ws, bs = seeded(ks, 2, seed=ks)
    if ks == 1:            # p = 1 whatever the network: every gradient is exactly 0
        lens = make_lens(pkg, Ws, bs)
        gen = torch.Generator().manual_seed(1)
        inp = torch.from_numpy(tor.draw_probes(300, gen)).cuda()
        dWs, dbs, dX = grads_ours(lens, inp, torch.randn(300, 1, generator=gen).cuda())
        assert all(bool((t == 0).all()) for t in dWs + dbs + [dX])
        REPORT[f"ks1_{kind}"] = 0.0
        return
    run_case(pkg, f"ks{ks}_{kind}", Ws, bs, 1000, kind, seed=100 + ks)


@pytest.mark.parametrize("M", [1, 63, 64, 65, 1000, CHUNK - 1, CHUNK, CHUNK + 1, 2 * CHUNK + 17])
def test_probe_counts_rf50mm_vs_f64(pkg, M):
    Ws, bs = rf50mm()
    run_case(pkg, f"rf50mm_M{M}", Ws, bs, M, "random", seed=M)


@pytest.mark.parametrize("hidden", [0, 2, 8])
@pytest.mark.parametrize("kind", ["random", "mse", "l1"])
@pytest.mark.parametrize("M", [65, CHUNK + 1])
def test_network_depths_vs_f64(pkg, hidden, kind, M):
    Ws, bs = seeded(11, hidden, seed=7 + hidden)
    run_case(pkg, f"seeded_h{hidden}_{kind}_M{M}", Ws, bs, M, kind, seed=hidden * 3 + M)


@pytest.mark.parametrize("ks", [5, 11])
@pytest.mark.parametrize("kind", ["random", "mse"])
def test_from_scratch_kaiming_dead_units_exact_zero(pkg, ks, kind):
    Ws, bs = kaiming(ks, seed=ks)
    run_case(pkg, f"kaiming_ks{ks}_{kind}", Ws, bs, 1000, kind, seed=ks + 50, exact_zero_dead=True)


@pytest.mark.parametrize("kind", ["random", "mse", "l1"])
def test_rf50mm_losses_vs_f64(pkg, kind):
    Ws, bs = rf50mm()
    run_case(pkg, f"rf50mm_{kind}", Ws, bs, 1000, kind, seed=9)


# ------------------------------------------------------------------------------------ 2. the normalisation clamp
@pytest.mark.parametrize("side", ["below", "above", "both"])
def test_normalisation_clamp_both_sides(pkg, side):
    gen = torch.Generator().manual_seed(21)
    Ws, bs = seeded(11, 2, seed=21)
    bs = tor.saturate_head(Ws, bs, gen)
    inp, _ = tor.sample_probes(Ws, bs, 2000, gen)
    _, S, _ = tor.forward_f64(Ws, bs, inp)
    below = (S < tor.NORMALIZE_EPS).numpy()
    assert 200 < below.sum() < 1800, below.sum()
    sel = {"below": below, "above": ~below, "both": np.ones_like(below)}[side]
    run_case(pkg, f"clamp_{side}", Ws, bs, int(sel.sum()), "random", seed=22, probes=torch.from_numpy(inp[sel]).cuda(),
             tol=CLAMP_TOL)


# ----------------------------------------------------------------------------------------------- 3. full frame
def test_full_frame_rf50mm_vs_f64(pkg):
    Ws, bs = rf50mm()
    run_case(pkg, "rf50mm_full_frame_480x640", Ws, bs, 480 * 640, "mse", seed=480)


# ------------------------------------------------------------------------------- 4. forward is the no-grad forward
@pytest.mark.parametrize("ks", [5, 11, 31])
def test_forward_bit_identical_in_every_grad_setting(pkg, ks):
    Ws, bs = rf50mm() if ks == 11 else seeded(ks, 2, seed=ks)
    lens = make_lens(pkg, Ws, bs)
    x = torch.from_numpy(tor.draw_probes(CHUNK + 5, torch.Generator().manual_seed(ks))).cuda()
    ref = lens.pred(x).reshape(x.shape[0], ks * ks)
    outs = []
    for grad_mode in (False, True):
        for probes_grad in (False, True):
            for frozen in (False, True):
                for p in lens.psfnet.parameters():
                    p.requires_grad_(not frozen)
                with torch.set_grad_enabled(grad_mode):
                    outs.append(lens.psfnet(x.clone().requires_grad_(probes_grad)).detach())
    for p in lens.psfnet.parameters():
        p.requires_grad_(True)
    for o in outs:
        assert torch.equal(o, ref)


def test_grad_path_runs_the_no_grad_kernels(pkg):
    """The no-grad call launches exactly one kernel (mlp_fp32_kernel<false>), as before this path existed."""
    Ws, bs = seeded(11, 2, seed=3)
    lens = make_lens(pkg, Ws, bs)
    x = torch.rand(100, 4, device="cuda")
    lens.psfnet(x)
    lib = pkg.native.lib
    with torch.no_grad():
        n0 = lib.aadff_launch_count()
        lens.psfnet(x)
        assert lib.aadff_launch_count() - n0 == 1
    n0 = lib.aadff_launch_count()
    y = lens.psfnet(x)
    assert lib.aadff_launch_count() - n0 == 1 and y.grad_fn is not None


# ------------------------------------------------------------------------------------------ 5. autograd contract
def test_probes_only_parameters_only_and_frozen_layers(pkg):
    Ws, bs = seeded(11, 2, seed=5)
    lens = make_lens(pkg, Ws, bs)
    gen = torch.Generator().manual_seed(5)
    inp = torch.from_numpy(tor.sample_probes(Ws, bs, 500, gen)[0]).cuda()
    g = torch.randn(500, 121, generator=gen).cuda()
    full = grads_ours(lens, inp, g)
    lins = lens.psfnet.linear_layers()
    # probes only
    for p in lens.psfnet.parameters():
        p.requires_grad_(False)
        p.grad = None
    x = inp.clone().requires_grad_(True)
    lens.psfnet(x).backward(g)
    assert torch.equal(x.grad, full[2]) and all(p.grad is None for p in lens.psfnet.parameters())
    # parameters only
    for p in lens.psfnet.parameters():
        p.requires_grad_(True)
    lens.psfnet(inp).backward(g)
    assert all(torch.equal(l.weight.grad, w) for l, w in zip(lins, full[0]))
    assert all(torch.equal(l.bias.grad, b) for l, b in zip(lins, full[1]))
    # layers 0 and 2 frozen, bias of layer 3 frozen
    for p in lens.psfnet.parameters():
        p.grad = None
    for p in (lins[0].weight, lins[0].bias, lins[2].weight, lins[2].bias, lins[3].bias):
        p.requires_grad_(False)
    lens.psfnet(inp).backward(g)
    for l, lin in enumerate(lins):
        for p, ref in ((lin.weight, full[0][l]), (lin.bias, full[1][l])):
            if p.requires_grad:
                assert torch.equal(p.grad, ref)
            else:
                assert p.grad is None


def test_shapes_dtypes_devices_float64_probes(pkg):
    Ws, bs = seeded(5, 2, seed=6)
    lens = make_lens(pkg, Ws, bs)
    x = torch.rand(2, 3, 5, 4, dtype=torch.float64, device="cuda", requires_grad=True)
    psf = lens.psfnet(x)
    assert psf.shape == (2, 3, 5, 25) and psf.dtype == torch.float32
    psf.pow(2).sum().backward()
    assert x.grad.shape == x.shape and x.grad.dtype == torch.float64 and x.grad.device == x.device
    for p in lens.psfnet.parameters():
        assert p.grad.shape == p.shape and p.grad.dtype == p.dtype and p.grad.device == p.device
    xc = torch.rand(7, 4, dtype=torch.float64, requires_grad=True)          # CPU probes, CUDA network
    lens.psfnet(xc).sum().backward()
    assert xc.grad.device.type == "cpu" and xc.grad.dtype == torch.float64


def test_two_backwards_accumulate_exactly_twice(pkg):
    Ws, bs = seeded(11, 2, seed=8)
    lens = make_lens(pkg, Ws, bs)
    x = torch.rand(300, 4, device="cuda", requires_grad=True)
    g = torch.randn(300, 121, device="cuda")
    psf = lens.psfnet(x)
    psf.backward(g, retain_graph=True)
    once = [p.grad.clone() for p in lens.psfnet.parameters()] + [x.grad.clone()]
    psf.backward(g)
    twice = [p.grad for p in lens.psfnet.parameters()] + [x.grad]
    assert all(torch.equal(b, 2 * a) for a, b in zip(once, twice))


def test_zero_probes(pkg):
    Ws, bs = seeded(11, 2, seed=9)
    lens = make_lens(pkg, Ws, bs)
    x = torch.zeros(0, 4, device="cuda", requires_grad=True)
    psf = lens.psfnet(x)
    assert psf.shape == (0, 121)
    psf.sum().backward()
    assert x.grad.shape == (0, 4)
    assert all(bool((p.grad == 0).all()) for p in lens.psfnet.parameters())


def test_in_place_parameter_change_raises(pkg):
    Ws, bs = seeded(11, 2, seed=10)
    lens = make_lens(pkg, Ws, bs)
    psf = lens.psfnet(torch.rand(50, 4, device="cuda"))
    with torch.no_grad():
        lens.psfnet.linear_layers()[1].weight.mul_(1.01)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        psf.sum().backward()


def test_backward_after_handle_rebuild(pkg):
    """forward, refresh(), another forward (a new handle), then the first graph's backward: the first handle must
    still be alive and give the first forward's gradients."""
    Ws, bs = seeded(11, 2, seed=11)
    lens = make_lens(pkg, Ws, bs)
    gen = torch.Generator().manual_seed(11)
    inp = torch.from_numpy(tor.sample_probes(Ws, bs, 400, gen)[0]).cuda()
    g = torch.randn(400, 121, generator=gen, dtype=torch.float64).cuda()
    ref = mgo.grads_f64([torch.as_tensor(w).cuda() for w in Ws], [torch.as_tensor(b).cuda() for b in bs], inp, g)
    x = inp.clone().requires_grad_(True)
    psf = lens.psfnet(x)
    first = lens._native
    lens.refresh()
    lens.psfnet(torch.rand(1000, 4, device="cuda"))
    assert lens._native is not first
    del first
    torch.cuda.synchronize()
    psf.backward(g.float())
    lins = lens.psfnet.linear_layers()
    compare("handle_rebuild", ([l.weight.grad for l in lins], [l.bias.grad for l in lins], x.grad), ref)


# ------------------------------------------------------------------------------------------------ 6. determinism
def test_deterministic_across_calls_and_streams(pkg):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs)
    x = torch.rand(CHUNK + 999, 4, device="cuda")
    g = torch.randn(CHUNK + 999, 121, device="cuda")

    def grads():
        xx = x.clone().requires_grad_(True)
        for p in lens.psfnet.parameters():
            p.grad = None
        lens.psfnet(xx).backward(g)
        return [p.grad.clone() for p in lens.psfnet.parameters()] + [xx.grad]

    a = grads()
    b = grads()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s1):
        c = grads()
    with torch.cuda.stream(s2):
        d = grads()
    torch.cuda.synchronize()
    for r in (b, c, d):
        assert all(torch.equal(u, v) for u, v in zip(a, r))


# ------------------------------------------------------------------------------------------------ 7. CUDA graphs
def test_cuda_graph_capture_replays_eager_results(pkg):
    Ws, bs = seeded(11, 8, seed=12)
    lens = make_lens(pkg, Ws, bs)
    M = CHUNK + 300
    x = torch.rand(M, 4, device="cuda", requires_grad=True)
    g = torch.randn(M, 121, device="cuda")
    params = list(lens.psfnet.parameters())

    def step():
        psf = lens.psfnet(x)
        grads = torch.autograd.grad(psf, params + [x], g)
        return psf.detach(), grads

    eager_psf, eager_grads = step()
    lens.psfnet(x)                       # the handle exists before the capture (its creation copies weights)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                           # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cap_psf, cap_grads = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(cap_psf, eager_psf)
    assert all(torch.equal(a, b) for a, b in zip(cap_grads, eager_grads))


# ------------------------------------------------------------------------------- 8. the fitting step's gradients
@pytest.mark.parametrize("ks", [5, 11])
def test_matches_native_trainer_gradients(pkg, ks):
    Ws, bs = rf50mm() if ks == 11 else seeded(ks, 2, seed=ks)
    lens = make_lens(pkg, Ws, bs)
    gen = torch.Generator().manual_seed(13)
    inp = torch.from_numpy(tor.sample_probes(Ws, bs, 128, gen)[0]).cuda()
    tgt = torch.from_numpy(tor.random_targets(128, ks * ks, gen)).cuda()
    loss = nn.MSELoss()(lens.psfnet(inp), tgt)
    loss.backward()
    trainer = pkg.native.NativeTrainer(Ws, bs, 128, torch.cuda.current_device())
    try:
        with torch.cuda.device(0):
            pkg.native.check(pkg.native.lib.aadff_trainer_step(trainer.handle, inp.data_ptr(), tgt.data_ptr(), 0.0, None,
                                                               torch.cuda.current_stream().cuda_stream))
        tW, tb = trainer.read(1, torch.cuda.current_stream().cuda_stream)
    finally:
        trainer.close()
    lins = lens.psfnet.linear_layers()
    for l, lin in enumerate(lins):
        for ours, theirs in ((lin.weight.grad, tW[l]), (lin.bias.grad, tb[l])):
            theirs = torch.from_numpy(theirs).cuda()
            err = float((ours - theirs).abs().max() / theirs.abs().max())
            assert err <= TOL, (l, err)
            REPORT[f"trainer_ks{ks}_l{l}"] = err


# ------------------------------------------------------------------------------ 9. psfnet -> local_psf_render
def test_end_to_end_image_loss_vs_f64(pkg):
    Ws, bs = rf50mm()
    lens = make_lens(pkg, Ws, bs)
    ks, N, H, W = 11, 2, 24, 40
    gen = torch.Generator().manual_seed(14)
    foc = torch.tensor([-800.0, -3000.0])
    depth = -(300 + 5000 * torch.rand(N, H, W, generator=gen, dtype=torch.float64))
    for _ in range(200):                          # redraw pixels whose forward sits within the sampler's margins
        o = orc.model_input(depth.float(), foc).reshape(-1, 4).numpy()
        bad = ~tor.branch_margin_ok(Ws, bs, o)
        if not bad.any():
            break
        depth.view(-1)[torch.from_numpy(np.flatnonzero(bad))] = -(300 + 5000 * torch.rand(int(bad.sum()), generator=gen,
                                                                                            dtype=torch.float64))
    assert not bad.any()
    img = torch.rand(N, 3, H, W, generator=gen)
    target = torch.rand(N, 3, H, W, generator=gen)
    x, y = orc.coord_grid(H, W)

    def chain(depth_t, psf_fn, render_fn, dtype):
        z = lens.depth2z(depth_t)
        fz = lens.depth2z(foc.to(depth_t.device, dtype).view(N, 1, 1).expand(N, H, W))
        o = torch.stack((x.to(depth_t.device, dtype).expand(N, H, W), y.to(depth_t.device, dtype).expand(N, H, W),
                         z, fz), -1)
        psf = psf_fn(o).reshape(N, H, W, ks, ks)
        out = render_fn(img.to(depth_t.device, dtype), psf, ks)
        return ((out - target.to(depth_t.device, dtype)) ** 2).mean()

    d32 = depth.float().cuda().requires_grad_(True)
    import aadff_render
    chain(d32, lens.psfnet, aadff_render.local_psf_render, torch.float32).backward()
    W64 = [torch.as_tensor(w).double().requires_grad_(True) for w in Ws]
    b64 = [torch.as_tensor(b).double().requires_grad_(True) for b in bs]
    d64 = depth.clone().requires_grad_(True)
    chain(d64, lambda o: orc.mlp_forward(W64, b64, o, torch.float64), orc.local_psf_render, torch.float64).backward()
    lins = lens.psfnet.linear_layers()
    compare("end_to_end_image_loss", ([l.weight.grad for l in lins], [l.bias.grad for l in lins], d32.grad),
            ([w.grad for w in W64], [b.grad for b in b64], d64.grad))


# -------------------------------------------------------------------------------------- 10. an AdamW loop
def test_adamw_loop_gradients_vs_f64(pkg):
    Ws, bs = seeded(11, 2, seed=15)
    lens = make_lens(pkg, Ws, bs)
    opt = torch.optim.AdamW(lens.psfnet.parameters(), lr=1e-4)
    gen = torch.Generator().manual_seed(15)
    checked = 0
    for step in range(20):
        lins = lens.psfnet.linear_layers()
        Wc = [l.weight.detach().cpu().numpy() for l in lins]
        bc = [l.bias.detach().cpu().numpy() for l in lins]
        inp = torch.from_numpy(tor.sample_probes(Wc, bc, 128, gen)[0]).cuda()
        tgt = torch.from_numpy(tor.random_targets(128, 121, gen)).cuda()
        opt.zero_grad()
        handle = lens._native
        nn.MSELoss()(lens.psfnet(inp), tgt).backward()
        assert step == 0 or lens._native is not handle            # each update rebuilds the handle
        if step in (0, 10, 19):
            _, _, p64 = tor.forward_f64(Wc, bc, inp.cpu())
            g = 2.0 * (p64 - tgt.cpu().double()) / (128 * 121)
            ref = mgo.grads_f64([torch.as_tensor(w).cuda() for w in Wc], [torch.as_tensor(b).cuda() for b in bc],
                                inp, g.cuda())
            compare(f"adamw_step{step}", ([l.weight.grad for l in lins], [l.bias.grad for l in lins],
                                          torch.zeros(128, 4, device="cuda")), (ref[0], ref[1], torch.zeros(128, 4)))
            checked += 1
        opt.step()
    assert checked == 3
