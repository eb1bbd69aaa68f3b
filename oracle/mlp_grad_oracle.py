"""The backward of the PSFNet MLP (aadff_psfnet_backward_f32, csrc/mlp_grad_kernel.cuh) in float64.

``lens.psfnet(inp)`` is the reference's MLP (deeplens/psfnet_arch.py:24-47): Linear + ReLU layers, a sigmoid head and
F.normalize(p=1) with its 1e-12 clamp.  ``grads_f64`` runs that forward through torch autograd in float64 and back-
propagates an arbitrary upstream gradient g = dL/dp.  Probes for comparisons against fp32 come from
``oracle.train_oracle.sample_probes``, which keeps both precisions on the same ReLU and clamp branches.
"""
import torch
import torch.nn.functional as F

from oracle.train_oracle import _f64


def grads_f64(Ws, bs, inp, g):
    """Gradients of sum(p * g) for p = MLP(inp), i.e. the backward of the network for an arbitrary upstream gradient
    g = dL/dp [M, kk], by float64 autograd through F.linear, ReLU, sigmoid and F.normalize(p=1)
    -> (dWs, dbs, dX) as float64 tensors on the device of inp."""
    dev = inp.device if isinstance(inp, torch.Tensor) else torch.device("cpu")
    W = [_f64(w).to(dev).clone().requires_grad_(True) for w in Ws]
    b = [_f64(v).to(dev).clone().requires_grad_(True) for v in bs]
    x0 = _f64(inp).to(dev).clone().requires_grad_(True)
    x = x0
    for l in range(len(W)):
        x = F.linear(x, W[l], b[l])
        x = torch.relu(x) if l < len(W) - 1 else torch.sigmoid(x)
    p = F.normalize(x, p=1, dim=-1)
    p.backward(_f64(g).to(dev))
    return [w.grad for w in W], [v.grad for v in b], x0.grad
