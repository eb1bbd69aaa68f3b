"""The float64 fitting-step oracle (oracle/train_oracle.py) pinned to torch on the CPU: its AdamW to
torch.optim.AdamW, its forward / backward to autograd through the reference's MLP layout, and its probe sampler to
the margins it promises."""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import train_oracle as tro


def test_adamw_f64_matches_torch_adamw():
    gen = torch.Generator().manual_seed(1)
    shapes = [(7, 5), (5,), (3, 7)]
    params = [torch.randn(s, generator=gen, dtype=torch.float64).requires_grad_(True) for s in shapes]
    betas, eps, wd, lr0, steps = (0.8, 0.99), 1e-3, 0.05, 3e-2, 50
    opt = torch.optim.AdamW(params, lr=lr0, betas=betas, eps=eps, weight_decay=wd, foreach=False)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=steps)
    P = [p.detach().numpy().copy() for p in params]
    m, v = tro.zero_moments(P), tro.zero_moments(P)
    for step in range(1, steps + 1):
        # gradients over several orders of magnitude, some exactly zero, so eps matters for part of the elements
        G = [torch.randn(s, generator=gen, dtype=torch.float64) * 10.0 ** float(torch.randint(-6, 1, (1,), generator=gen))
             for s in shapes]
        G[1][::2] = 0.0
        lr = opt.param_groups[0]["lr"]
        for p, g in zip(params, G):
            p.grad = g.clone()
        opt.step()
        sched.step()
        P = tro.adamw_f64(P, G, m, v, step, lr, betas, eps, wd)
        for a, p in zip(P, params):
            ref = p.detach().numpy()
            assert np.abs(a - ref).max() <= 1e-12 * np.abs(ref).max(), step
    assert lr < lr0 * 1e-2                                   # the schedule really ran down


def _mlp_like_reference(dims):
    """nn.Sequential laid out as aadff_arch.MLP.net: Linear/ReLU pairs, then Linear + Sigmoid."""
    mods = []
    for a, b in zip(dims[:-2], dims[1:-1]):
        mods += [nn.Linear(a, b), nn.ReLU(inplace=True)]
    mods += [nn.Linear(dims[-2], dims[-1]), nn.Sigmoid()]
    return nn.Sequential(*mods).double()


def test_step_f64_matches_autograd_through_reference_layout():
    gen = torch.Generator().manual_seed(2)
    for dims in ([4, 16, 64, 64, 25], [4, 9]):
        Ws, bs = tro.kaiming_net(dims, gen, bias_scale=0.1)
        net = _mlp_like_reference(dims)
        lins = [m for m in net if isinstance(m, nn.Linear)]
        with torch.no_grad():
            for lin, W, b in zip(lins, Ws, bs):
                lin.weight.copy_(torch.from_numpy(W))
                lin.bias.copy_(torch.from_numpy(b))
        inp = tro.draw_probes(33, gen)
        tgt = tro.random_targets(33, dims[-1], gen)
        pred = F.normalize(net(torch.from_numpy(inp).double()), p=1, dim=-1)
        loss = nn.MSELoss()(pred, torch.from_numpy(tgt).double())
        loss.backward()
        l64, p64, dWs, dbs = tro.step_f64(Ws, bs, inp, tgt)
        assert abs(l64 - loss.item()) <= 1e-14 * loss.item()
        assert np.abs(p64 - pred.detach().numpy()).max() <= 1e-15
        for lin, dW, db in zip(lins, dWs, dbs):
            assert np.abs(dW - lin.weight.grad.numpy()).max() <= 1e-12 * np.abs(dW).max()
            assert np.abs(db - lin.bias.grad.numpy()).max() <= 1e-12 * np.abs(db).max()


def test_sampler_keeps_its_margins():
    gen = torch.Generator().manual_seed(3)
    dims = [4, 64, 256] + [256] * 8 + [121]
    Ws, bs = tro.kaiming_net(dims, gen, bias_scale=0.1)
    inp, redrawn = tro.sample_probes(Ws, bs, 512, gen)
    assert redrawn > 0                       # the deep net has probes next to a ReLU kink: the sampler has work to do
    pre, S, _ = tro.forward_f64(Ws, bs, inp)
    for z in pre:
        a = z.abs()
        assert bool((a >= tro.RELU_MARGIN * a.amax(-1, keepdim=True)).all())
    # a saturated head: the L1 sums straddle the clamp, and no kept probe is near it
    Ws, bs = tro.kaiming_net([4, 32, 9], gen, bias_scale=0.1)
    bs = tro.saturate_head(Ws, bs, gen)
    assert float(bs[-1].max()) < -20
    inp, redrawn = tro.sample_probes(Ws, bs, 256, gen)
    _, S, _ = tro.forward_f64(Ws, bs, inp)
    assert bool((S < tro.NORMALIZE_EPS).any()) and bool((S > tro.NORMALIZE_EPS).any())
    assert bool(((S - tro.NORMALIZE_EPS).abs() >= tro.CLAMP_MARGIN * tro.NORMALIZE_EPS).all())
    assert tro.branch_margin_ok(Ws, bs, inp).all()
