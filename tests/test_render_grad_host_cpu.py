"""Host-side checks of the focal-stack render backward (no GPU needed): the float64 oracle against autograd through the
reference's unfold formulation and against central finite differences, its sampler's margins, the C ABI's refusals
that need neither a handle nor a device, and the CPU lens refusing the differentiable path."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import focal_stack_oracle as orc
from oracle import render_grad_oracle as rgo
from oracle import train_oracle as tor


@pytest.fixture(scope="module")
def lib():
    import aadff_b200
    return aadff_b200.native.lib


def small_case(ks, N=2, C=2, S=2, H=5, W=6, seed=0):
    gen = torch.Generator().manual_seed(seed)
    Ws, bs = tor.kaiming_net([4, 16, 32, ks * ks], gen, bias_scale=0.1)
    foc_z = 0.1 + 0.8 * torch.rand(N, S, generator=gen, dtype=torch.float64)
    depth, foc = rgo.sample_depths(Ws, bs, N, H, W, foc_z, gen)
    img = torch.rand(N, C, H, W, generator=gen, dtype=torch.float64)
    G = torch.randn(N, C, S, H, W, generator=gen, dtype=torch.float64)
    return Ws, bs, img, depth, foc, G


def unfold_stack_f64(Ws, bs, img, depth, foc, ks):
    """render_reference_ops's formulation (replicate pad, unfold, broadcast multiply, sum over k^2) in float64."""
    N, C, H, W = img.shape
    S = foc.shape[1]
    P = orc.mlp_forward(Ws, bs, rgo.probes_f64(depth, foc), torch.float64)        # [N,S,H,W,kk]
    r = (ks - 1) // 2
    cols = F.unfold(F.pad(img, (r, r, r, r), mode="replicate"), (ks, ks)).view(N, C, 1, ks * ks, H * W)
    taps = P.reshape(N, S, H * W, ks * ks).permute(0, 1, 3, 2)[:, None]            # [N,1,S,kk,HW]
    return (cols * taps).sum(3).view(N, C, S, H, W)


@pytest.mark.parametrize("ks", [1, 3, 5])
def test_oracle_matches_unfold_autograd(ks):
    Ws, bs, img, depth, foc, G = small_case(ks, seed=ks)
    ref = rgo.grads_f64(Ws, bs, img, depth, foc, ks, G)
    W_ = [torch.as_tensor(w).double().requires_grad_(True) for w in Ws]
    b_ = [torch.as_tensor(b).double().requires_grad_(True) for b in bs]
    x = img.clone().requires_grad_(True)
    d = depth.double().requires_grad_(True)
    f = foc.double().requires_grad_(True)
    out = unfold_stack_f64(W_, b_, x, d, f, ks)
    torch.testing.assert_close(out, ref["out"], rtol=1e-12, atol=1e-12)
    out.backward(G)

    def close(a, r):
        torch.testing.assert_close(a, r, rtol=1e-9, atol=1e-9 * float(r.abs().max()))

    close(ref["img"], x.grad)
    close(ref["depth"], d.grad)
    close(ref["foc"], f.grad)
    for l in range(len(Ws)):
        close(ref["W"][l], W_[l].grad)
        close(ref["b"][l], b_[l].grad)


def test_oracle_matches_finite_differences():
    ks = 3
    Ws, bs, img, depth, foc, G = small_case(ks, seed=7)
    ref = rgo.grads_f64(Ws, bs, img, depth, foc, ks, G)
    d64, f64 = depth.double(), foc.double()

    def loss(img_=img, d_=d64, f_=f64, W0=None):
        Ws_ = [torch.as_tensor(w).double() for w in Ws]
        if W0 is not None:
            Ws_[0] = W0
        return float((rgo.render_stack_f64(Ws_, bs, img_, d_, f_, ks) * G).sum())

    def fd(t, idx, h, **kw):
        tp, tm = t.clone(), t.clone()
        tp[idx] += h
        tm[idx] -= h
        return (loss(**{kw["name"]: tp}) - loss(**{kw["name"]: tm})) / (2 * h)

    for idx in [(0, 0, 0, 0), (1, 1, 4, 5), (0, 1, 2, 3)]:
        assert fd(img, idx, 1e-4, name="img_") == pytest.approx(float(ref["img"][idx]), rel=1e-6, abs=1e-9)
    for idx in [(0, 0, 0), (1, 4, 5), (0, 2, 3)]:
        assert fd(d64, idx, 1e-2, name="d_") == pytest.approx(float(ref["depth"][idx]), rel=1e-5, abs=1e-12)
    for idx in [(0, 0), (1, 1)]:
        assert fd(f64, idx, 1e-2, name="f_") == pytest.approx(float(ref["foc"][idx]), rel=1e-5, abs=1e-12)
    W0 = torch.as_tensor(Ws[0]).double()
    for idx in [(0, 2), (5, 3)]:
        assert fd(W0, idx, 1e-5, name="W0") == pytest.approx(float(ref["W"][0][idx]), rel=1e-5, abs=1e-9)


def test_oracle_clamp_rule_gives_exact_zeros():
    """Invalid (0) and out-of-range depths, and a focus distance past d_max, get exactly 0; an in-range one does not."""
    ks = 3
    Ws, bs, img, depth, foc, G = small_case(ks, seed=3)
    depth = depth.clone()
    depth[0, 0, 0] = 0.0                 # invalid
    depth[0, 1, 1] = -100.0              # nearer than 200 mm: z < 0
    depth[1, 2, 2] = -30000.0            # farther than 20 m: z > 1
    foc = foc.clone()
    foc[1, 0] = -25000.0
    ref = rgo.grads_f64(Ws, bs, img, depth, foc, ks, G)
    for idx in [(0, 0, 0), (0, 1, 1), (1, 2, 2)]:
        assert float(ref["depth"][idx]) == 0.0
    assert float(ref["foc"][1, 0]) == 0.0
    assert float(ref["foc"][0, 0]) != 0.0 and float(ref["depth"][0, 3, 3]) != 0.0


def test_sampler_keeps_margins_and_fixed_pixels():
    gen = torch.Generator().manual_seed(11)
    Ws, bs = tor.kaiming_net([4, 16, 32, 9], gen, bias_scale=0.1)
    mask = torch.zeros(1, 6, 7, dtype=torch.bool)
    mask[0, 0, 0] = True
    fixed = torch.zeros(1, 6, 7)
    depth, foc = rgo.sample_depths(Ws, bs, 1, 6, 7, torch.tensor([[0.3, 0.7]]), gen, fixed=(mask, fixed))
    assert float(depth[0, 0, 0]) == 0.0
    z = orc.depth2z(depth[~mask].double())
    assert float(z.min()) >= 0.02 - 1e-6 and float(z.max()) <= 0.98 + 1e-6
    pr = rgo.probes_f64(depth.double(), foc.double()).to(torch.float32).reshape(-1, 4)
    ok = torch.as_tensor(tor.branch_margin_ok(Ws, bs, pr.numpy())).reshape(1, 2, 6, 7).all(1)
    assert bool((ok | mask).all())


def _fptrs(n, value=None):
    c_f32p = ctypes.POINTER(ctypes.c_float)
    return (c_f32p * n)(*([ctypes.cast(ctypes.c_void_p(value), c_f32p)] * n if value else [None] * n))


def test_backward_refusals_name_the_argument(lib):
    bwd = lib.aadff_render_stack_backward_f32
    st = (ctypes.c_int64 * 5)(1, 1, 1, 1, 1)
    ws = _fptrs(3, 256)

    def call(img=256, depth=256, foc=256, gout=256, strides=st, gimg=256, gdep=256, gfoc=256, gw=ws, gb=ws,
             N=1, C=3, S=2, H=8, W=8, d_min=-200.0, d_max=-20000.0, mode=0, work=256, wb=1 << 30):
        rc = bwd(None, img, depth, foc, gout, strides, gimg, gdep, gfoc, gw, gb, N, C, S, H, W, d_min, d_max, mode,
                 work, wb, None)
        assert rc == -1
        return lib.aadff_last_error()

    assert b"N must be >= 0" in call(N=-1)
    assert b"C must be >= 1" in call(C=0)
    assert b"S must be >= 1" in call(S=0)
    assert b"H and W must be >= 1" in call(H=0)
    assert b"H and W must be >= 1" in call(W=0)
    assert b"W must be <= 16384" in call(W=16385)
    assert b"mode is unknown" in call(mode=6)
    assert b"mode is unknown" in call(mode=-1)
    assert b"d_max must differ from d_min" in call(d_max=-200.0)
    assert b"img is NULL" in call(img=None)
    assert b"depth is NULL" in call(depth=None)
    assert b"foc is NULL" in call(foc=None)
    assert b"grad_out is NULL" in call(gout=None)
    assert b"grad_out_strides is NULL" in call(strides=None)
    msg = call(gimg=None, gdep=None, gfoc=None, gw=None, gb=None)
    assert b"no output requested" in msg and b"grad_img" in msg
    assert b"work must be 256-byte aligned" in call(work=256 + 16)
    assert b"net is NULL" in call()


def test_backward_work_bytes_refusals(lib):
    q = lib.aadff_render_stack_backward_work_bytes
    assert q(None, 0, 8) == -1
    assert b"H and W must be >= 1" in lib.aadff_last_error()
    assert q(None, 8, 16385) == -1
    assert b"W must be <= 16384" in lib.aadff_last_error()
    assert q(None, 8, 8) == -1
    assert b"net is NULL" in lib.aadff_last_error()


def test_cpu_lens_differentiable_render_raises_naming_cuda():
    import aadff_b200
    lens = aadff_b200.PSFNet(kernel_size=5, device="cpu")
    img = torch.rand(1, 3, 8, 8, requires_grad=True)
    depth = -1000.0 * torch.ones(1, 1, 8, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        lens.render(img, depth, torch.tensor([-900.0]), differentiable=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        lens.render_stack(img, depth, torch.tensor([[-900.0, -1500.0]]), differentiable=True)


def test_header_declares_render_backward():
    import aadff_b200
    syms = aadff_b200.native.exported_symbols()
    assert "aadff_render_stack_backward_f32" in syms and "aadff_render_stack_backward_work_bytes" in syms
