"""Host-side checks of the PSFNet MLP backward (no GPU needed): the float64 oracle's gradients against torch autograd
through an nn.Sequential, the C ABI's refusals that need neither a handle nor a device, and the CPU lens refusing the
differentiable path."""
import ctypes

import pytest
import torch
import torch.nn as nn

from oracle import mlp_grad_oracle as mgo
from oracle import train_oracle as tor


@pytest.fixture(scope="module")
def lib():
    import aadff_b200
    return aadff_b200.native.lib


@pytest.mark.parametrize("dims", [[4, 16, 9], [4, 64, 256, 256, 121], [4, 8, 8, 1]])
@pytest.mark.parametrize("saturate", [False, True])
def test_grads_f64_matches_sequential_autograd(dims, saturate):
    gen = torch.Generator().manual_seed(len(dims) * 10 + saturate)
    Ws, bs = tor.kaiming_net(dims, gen, bias_scale=0.1)
    if saturate:
        bs = tor.saturate_head(Ws, bs, gen)
    inp = torch.from_numpy(tor.draw_probes(37, gen))
    g = torch.randn(37, dims[-1], generator=gen, dtype=torch.float64)
    dWs, dbs, dX = mgo.grads_f64(Ws, bs, inp, g)

    mods = []
    for l, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        mods += [nn.Linear(a, b), nn.ReLU() if l < len(dims) - 2 else nn.Sigmoid()]
    seq = nn.Sequential(*mods).double()
    with torch.no_grad():
        for lin, W, b in zip([m for m in seq if isinstance(m, nn.Linear)], Ws, bs):
            lin.weight.copy_(torch.from_numpy(W))
            lin.bias.copy_(torch.from_numpy(b))
    x = inp.double().clone().requires_grad_(True)
    p = seq(x)
    p = p / p.abs().sum(-1, keepdim=True).clamp_min(1e-12)
    (p * g).sum().backward()
    lins = [m for m in seq if isinstance(m, nn.Linear)]

    def close(a, r):          # two float64 formulations of the same maths: they differ in the last bits only
        torch.testing.assert_close(a, r, rtol=1e-9, atol=1e-9 * float(r.abs().max()))

    for l, lin in enumerate(lins):
        close(dWs[l], lin.weight.grad)
        close(dbs[l], lin.bias.grad)
    close(dX, x.grad)
    assert all(w.dtype == torch.float64 for w in dWs)


def test_grads_f64_head_clamp_branch():
    """Below the clamp the normalisation passes no gradient: dL/ds = g / 1e-12."""
    gen = torch.Generator().manual_seed(4)
    Ws, bs = tor.kaiming_net([4, 8, 3], gen)
    bs[-1] = bs[-1] - 80.0                       # sigmoid ~ exp(-80): S far below 1e-12
    inp = torch.from_numpy(tor.draw_probes(5, gen))
    g = torch.randn(5, 3, generator=gen, dtype=torch.float64)
    dWs, dbs, _ = mgo.grads_f64(Ws, bs, inp, g)
    pre, S, _ = tor.forward_f64(Ws, bs, inp)
    assert bool((S < 1e-12).all())
    z = torch.relu(pre[0]) @ torch.from_numpy(Ws[1]).double().T + torch.from_numpy(bs[1]).double()
    s = torch.sigmoid(z)
    torch.testing.assert_close(dbs[1], (g / 1e-12 * s * (1 - s)).sum(0), rtol=1e-10, atol=0)


def _fptrs(n, value=None):
    c_f32p = ctypes.POINTER(ctypes.c_float)
    return (c_f32p * n)(*([ctypes.cast(ctypes.c_void_p(value), c_f32p)] * n if value else [None] * n))


def test_backward_refusals_name_the_argument(lib):
    bwd = lib.aadff_psfnet_backward_f32
    ws = _fptrs(3, 256)
    assert bwd(None, 256, 256, 256, ws, ws, 256, 1 << 20, -1, None) == -1
    assert b"M must be >= 0" in lib.aadff_last_error()
    assert bwd(None, None, 256, 256, ws, ws, 256, 1 << 20, 8, None) == -1
    assert b"inp is NULL" in lib.aadff_last_error()
    assert bwd(None, 256, None, 256, ws, ws, 256, 1 << 20, 8, None) == -1
    assert b"grad_psf is NULL" in lib.aadff_last_error()
    assert bwd(None, 260, 256, 256, ws, ws, 256, 1 << 20, 8, None) == -1
    assert b"inp must be 16-byte aligned" in lib.aadff_last_error()
    assert bwd(None, 256, 256, None, None, None, 256, 1 << 20, 8, None) == -1
    assert b"no output requested" in lib.aadff_last_error()
    assert b"grad_inp" in lib.aadff_last_error()
    assert bwd(None, 256, 256, 256, ws, ws, 256, 1 << 20, 8, None) == -1
    assert b"net is NULL" in lib.aadff_last_error()


def test_backward_work_bytes_refusals(lib):
    q = lib.aadff_psfnet_backward_work_bytes
    assert q(None, -1) == -1
    assert b"M must be >= 0" in lib.aadff_last_error()
    assert q(None, 8) == -1
    assert b"net is NULL" in lib.aadff_last_error()


def test_cpu_lens_psfnet_raises_naming_cuda():
    import aadff_b200
    lens = aadff_b200.PSFNet(kernel_size=5, device="cpu")
    x = torch.rand(3, 4, requires_grad=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        lens.psfnet(x)
    with pytest.raises(RuntimeError, match="CUDA"):     # parameters requiring grad, probes not
        lens.psfnet(torch.rand(3, 4))
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        lens.psfnet(torch.rand(3, 4))


def test_header_declares_backward(lib):
    import aadff_b200
    syms = aadff_b200.native.exported_symbols()
    assert "aadff_psfnet_backward_f32" in syms and "aadff_psfnet_backward_work_bytes" in syms
