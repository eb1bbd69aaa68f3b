"""The backward of the focal-stack render (aadff_render_stack_backward_f32, csrc/render_grad_kernel.cuh) in float64.

``render_stack_f64`` is ``focal_stack_oracle.render_stack`` in float64 with the probes built from the fp32 grid values
(``linspace_f32``: the values the kernels use) and from depth and focus distances kept in float64, so that torch
autograd can differentiate through depth2z's clamp.  ``grads_f64`` back-propagates an arbitrary upstream gradient G
[N,C,S,H,W] through it.  ``sample_depths`` draws depth maps and focus distances on which the float64 forward keeps
the ReLU-kink and normalisation-clamp margins of ``train_oracle.sample_probes``, and keeps them off depth2z's clamp
edges, so that the fp32 kernels and float64 take the same branches.
"""
import numpy as np
import torch

from oracle import focal_stack_oracle as orc
from oracle import train_oracle as tor

D_MIN, D_MAX = -orc.DMIN, -orc.DMAX        # PSFNet.d_min / d_max [mm]


def _f64(x, dev):
    """A float64 copy of x on dev, detached from the caller's tensor."""
    return torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).detach().to(dev, torch.float64).clone()


def probes_f64(depth, foc, d_min=D_MIN, d_max=D_MAX):
    """(x, y, depth2z(depth), depth2z(foc)) [N,S,H,W,4] in float64 from depth [N,H,W] and foc [N,S] (float64; autograd
    follows them through the clamp)."""
    N, H, W = depth.shape
    S = foc.shape[1]
    xs = torch.from_numpy(orc.linspace_f32(-1.0, 1.0, W)).to(depth.device, torch.float64)
    ys = torch.from_numpy(orc.linspace_f32(1.0, -1.0, H)).to(depth.device, torch.float64)
    z = orc.depth2z(depth, d_min, d_max)[:, None].expand(N, S, H, W)
    fz = orc.depth2z(foc, d_min, d_max)[:, :, None, None].expand(N, S, H, W)
    return torch.stack((xs.view(1, 1, 1, W).expand(N, S, H, W), ys.view(1, 1, H, 1).expand(N, S, H, W), z, fz), -1)


def render_stack_f64(Ws, bs, img, depth, foc, ks, d_min=D_MIN, d_max=D_MAX):
    """out [N,C,S,H,W] = sum_{i,j} img[n,c,clamp(h+i-r),clamp(w+j-r)] P[n,s,h,w,i,j], P = MLP(probes), in float64."""
    S = foc.shape[1]
    as_t = lambda t: (t if torch.is_tensor(t) else torch.from_numpy(np.asarray(t))).to(img.device)
    P = orc.mlp_forward([as_t(w) for w in Ws], [as_t(b) for b in bs], probes_f64(depth, foc, d_min, d_max),
                        torch.float64)                                                     # [N,S,H,W,kk]
    outs = [orc.local_psf_render(img, P[:, s], ks) for s in range(S)]
    return torch.stack(outs, 2)


def grads_f64(Ws, bs, img, depth, foc, ks, G, d_min=D_MIN, d_max=D_MAX):
    """Gradients of sum(render_stack(img, depth, foc) * G) by float64 autograd -> dict with 'img' [N,C,H,W],
    'depth' [N,H,W], 'foc' [N,S], 'W' and 'b' (lists per layer) and 'out' (the float64 forward), on img's device."""
    dev = img.device
    W_ = [_f64(w, dev).requires_grad_(True) for w in Ws]
    b_ = [_f64(v, dev).requires_grad_(True) for v in bs]
    x = _f64(img, dev).requires_grad_(True)
    d = _f64(depth, dev).requires_grad_(True)
    f = _f64(foc, dev).requires_grad_(True)
    out = render_stack_f64(W_, b_, x, d, f, ks, d_min, d_max)
    out.backward(_f64(G, dev))
    return {"img": x.grad, "depth": d.grad, "foc": f.grad, "W": [w.grad for w in W_], "b": [v.grad for v in b_],
            "out": out.detach()}


def sample_depths(Ws, bs, N, H, W, foc_z, gen, fixed=None, z_lo=0.02, z_hi=0.98, max_rounds=200, dev="cpu"):
    """Depth maps [N,H,W] (mm, float32) whose probes, with the focus distances of foc_z [N,S] (depth2z values), keep
    every margin of train_oracle.branch_margin_ok in every slice; z is drawn in [z_lo, z_hi], off depth2z's clamp
    edges.  `fixed` = (mask [N,H,W] bool, depth [N,H,W] mm) places depths on purpose (invalid, clamped): those pixels
    are never redrawn.  -> (depth, foc) in mm, float32 CPU tensors."""
    foc_z = torch.as_tensor(foc_z, dtype=torch.float64)
    S = foc_z.shape[1]
    foc = (D_MIN + foc_z * (D_MAX - D_MIN)).to(torch.float32)
    z = z_lo + (z_hi - z_lo) * torch.rand(N, H, W, generator=gen, dtype=torch.float64)
    depth = (D_MIN + z * (D_MAX - D_MIN)).to(torch.float32)
    keep = torch.zeros(N, H, W, dtype=torch.bool)
    if fixed is not None:
        keep = fixed[0].clone()
        depth[keep] = fixed[1].to(torch.float32)[keep]
    Wd = [_f64(w, dev) for w in Ws]
    bd = [_f64(v, dev) for v in bs]
    for _ in range(max_rounds):
        pr = probes_f64(depth.to(dev, torch.float64), foc.to(dev, torch.float64)).to(torch.float32)   # fp32 probes
        ok = _margin_ok(Wd, bd, pr.reshape(-1, 4)).reshape(N, S, H, W).all(1).cpu() | keep
        bad = ~ok
        if not bool(bad.any()):
            return depth, foc
        nz = z_lo + (z_hi - z_lo) * torch.rand(int(bad.sum()), generator=gen, dtype=torch.float64)
        depth[bad] = (D_MIN + nz * (D_MAX - D_MIN)).to(torch.float32)
    raise RuntimeError(f"sample_depths: margins not reached after {max_rounds} rounds")


def _margin_ok(Wd, bd, inp):
    """train_oracle.branch_margin_ok for a float32 tensor of probes on any device -> bool tensor [M]."""
    pre, S, _ = tor.forward_f64(Wd, bd, inp)
    ok = (S - tor.NORMALIZE_EPS).abs() >= tor.CLAMP_MARGIN * tor.NORMALIZE_EPS
    for z in pre:
        a = z.abs()
        ok &= (a >= tor.RELU_MARGIN * a.amax(-1, keepdim=True)).all(-1) & (a.amax(-1) > 0)
    return ok
