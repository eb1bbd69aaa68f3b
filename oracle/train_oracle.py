"""The PSFNet fitting step (csrc/train_kernels.cuh, aadff_trainer_*) in float64.

PSFNet.train_psfnet (deeplens/psfnet.py:79-132) runs psfnet(inp) -> nn.MSELoss -> backward -> AdamW.step.
Here the same step goes through the reference's own operators in float64:

- ``step_f64``: forward, loss and gradients, by torch autograd through F.linear, ReLU, sigmoid, F.normalize(p=1)
  with its 1e-12 clamp, and nn.MSELoss;
- ``adamw_f64``: torch's single-tensor AdamW update (decoupled decay, lerp for m, addcmul for v, bias corrections);
- ``sample_probes``: probes on which an fp32 forward takes the same branches as the float64 one.  A hidden unit whose
  pre-activation sits next to zero may be switched on in one precision and off in the other, and that changes the
  probe's whole contribution to dW; a probe whose L1 sum sits next to the clamp may take the other side of it.
  Such probes are redrawn.
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

NORMALIZE_EPS = 1e-12       # F.normalize's default eps: the L1 sum is clamped to at least this
RELU_MARGIN = 1e-5          # |pre-activation| >= this times the largest |pre-activation| of its layer and probe
CLAMP_MARGIN = 1e-4         # |S - 1e-12| >= this times 1e-12.  Near the clamp the head pre-activations sit at about
                            # -31, where one fp32 ulp of z (1.9e-6) moves exp(z), and so S, by 1.9e-6 relative: a few
                            # roundings of z must not carry a probe across the clamp


def _f64(x):
    if isinstance(x, torch.Tensor):
        return x.detach().to(torch.float64)
    return torch.from_numpy(np.asarray(x, dtype=np.float64))


def forward_f64(Ws, bs, inp):
    """-> (hidden pre-activations [layer][M, width], L1 sums S [M], p [M, kk]), all float64, no autograd."""
    with torch.no_grad():
        x, pre = _f64(inp), []
        L = len(Ws)
        for l in range(L):
            z = F.linear(x, _f64(Ws[l]), _f64(bs[l]))
            if l < L - 1:
                pre.append(z)
                x = torch.relu(z)
            else:
                x = torch.sigmoid(z)
        S = x.abs().sum(-1)
        return pre, S, F.normalize(x, p=1, dim=-1)


def step_f64(Ws, bs, inp, tgt):
    """One forward + MSE loss + backward in float64 -> (loss, p [M, kk], dWs, dbs) as float / numpy float64."""
    W = [_f64(w).clone().requires_grad_(True) for w in Ws]
    b = [_f64(v).clone().requires_grad_(True) for v in bs]
    x = _f64(inp)
    for l in range(len(W)):
        x = F.linear(x, W[l], b[l])
        x = torch.relu(x) if l < len(W) - 1 else torch.sigmoid(x)
    p = F.normalize(x, p=1, dim=-1)
    loss = nn.MSELoss()(p, _f64(tgt))
    loss.backward()
    return (float(loss.detach()), p.detach().numpy(), [w.grad.numpy() for w in W], [v.grad.numpy() for v in b])


def adamw_f64(P, G, m, v, step, lr, betas, eps, wd):
    """torch.optim.AdamW's single-tensor update of the parameters P with the gradients G at step `step` (1-based).
    P, G: lists of arrays; m, v: lists of float64 tensors (start at zeros), updated in place.  -> new P (float64 numpy)."""
    beta1, beta2 = betas
    bias_correction1 = 1 - beta1 ** step
    bias_correction2_sqrt = (1 - beta2 ** step) ** 0.5
    step_size = lr / bias_correction1
    out = []
    for p, g, mi, vi in zip(P, G, m, v):
        p, g = _f64(p).clone(), _f64(g)
        p.mul_(1 - lr * wd)
        mi.lerp_(g, 1 - beta1)
        vi.mul_(beta2).addcmul_(g, g, value=1 - beta2)
        denom = (vi.sqrt() / bias_correction2_sqrt).add_(eps)
        p.addcdiv_(mi, denom, value=-step_size)
        out.append(p.numpy())
    return out


def zero_moments(P):
    return [torch.zeros(np.shape(p), dtype=torch.float64) for p in P]


def branch_margin_ok(Ws, bs, inp):
    """-> bool [M]: the probe keeps RELU_MARGIN at every hidden unit and CLAMP_MARGIN at the normalisation clamp."""
    pre, S, _ = forward_f64(Ws, bs, inp)
    ok = (S - NORMALIZE_EPS).abs() >= CLAMP_MARGIN * NORMALIZE_EPS
    for z in pre:
        a = z.abs()
        ok &= (a >= RELU_MARGIN * a.amax(-1, keepdim=True)).all(-1) & (a.amax(-1) > 0)
    return ok.numpy()


def draw_probes(M, gen):
    """M probes like PSFNet's training inputs: (x, y) in [-1, 1], (z, foc) in [0, 1]; float32."""
    x = torch.rand(M, 4, generator=gen)
    x[:, :2] = x[:, :2] * 2 - 1
    return x.numpy()


def sample_probes(Ws, bs, M, gen, max_rounds=1000):
    """M float32 probes on which the float64 forward keeps every margin at the parameters (Ws, bs)
    -> (probes [M, 4], number of probes redrawn)."""
    inp = draw_probes(M, gen)
    redrawn = 0
    for _ in range(max_rounds):
        bad = np.flatnonzero(~branch_margin_ok(Ws, bs, inp))
        if bad.size == 0:
            return inp, redrawn
        redrawn += bad.size
        inp[bad] = draw_probes(bad.size, gen)
    raise RuntimeError(f"sample_probes: no {M} probes keep the margins after {max_rounds} rounds")


def saturate_head(Ws, bs, gen):
    """Head biases shifted so that the L1 sum S of half of all probes falls below the 1e-12 clamp: for a head
    pre-activation z far below zero sigmoid(z) = exp(z), so S = exp(shift) * sum_j exp(z_j).  -> new bs (float32)."""
    with torch.no_grad():
        x = _f64(draw_probes(256, gen))
        for l in range(len(Ws)):
            x = F.linear(x, _f64(Ws[l]), _f64(bs[l]))
            if l < len(Ws) - 1:
                x = torch.relu(x)
        shift = math.log(NORMALIZE_EPS) - float(torch.logsumexp(x, -1).median())
    return list(bs[:-1]) + [(bs[-1] + shift).astype(np.float32)]


def random_targets(M, kk, gen):
    """M random L1-normalised PSFs of kk taps, float32."""
    t = torch.rand(M, kk, generator=gen) + 1e-3
    return (t / t.sum(1, keepdim=True)).numpy()


def kaiming_net(dims, gen, bias_scale=0.0):
    """Kaiming-uniform weights (a=0, fan_in: aadff_arch.initialize_weights) and biases uniform in
    [-bias_scale, bias_scale] (zero, as the reference initialises them, by default); float32 numpy."""
    Ws, bs = [], []
    for fin, fout in zip(dims[:-1], dims[1:]):
        bound = math.sqrt(2.0) * math.sqrt(3.0 / fin)
        Ws.append(((torch.rand(fout, fin, generator=gen) * 2 - 1) * bound).numpy())
        bs.append(((torch.rand(fout, generator=gen) * 2 - 1) * bias_scale).numpy())
    return Ws, bs
