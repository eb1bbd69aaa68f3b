"""Per-pixel PSF rendering (mirror of the reference's deeplens/render_psf.py:76-107)."""
import torch
from torch.autograd.function import once_differentiable

import aadff_native as _nat


__all__ = ["local_psf_render", "render_psf", "render_psf_map", "local_psf_render_high_res"]


def _ptr(t):
    return None if t is None else t.data_ptr()


class _LocalPSFRender(torch.autograd.Function):
    """img [N,C,H,W], taps [N,H,W,ks,ks]: fp32, contiguous, on one CUDA device."""

    @staticmethod
    def forward(ctx, img, taps, ks):
        n, c, h, w = img.shape
        out = torch.empty_like(img)
        _nat.call("aadff_local_psf_render_f32", img.data_ptr(), taps.data_ptr(), out.data_ptr(), n, c, h, w, ks,
                  device=img.device)
        ctx.save_for_backward(img, taps)
        ctx.ks = ks
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        img, taps = ctx.saved_tensors
        need_img, need_psf = ctx.needs_input_grad[:2]
        g = grad_out.contiguous()
        grad_img = torch.empty_like(img) if need_img else None
        grad_psf = torch.empty_like(taps) if need_psf else None
        n, c, h, w = img.shape
        _nat.call("aadff_local_psf_render_backward_f32", img.data_ptr(), taps.data_ptr(), g.data_ptr(), _ptr(grad_img),
                  _ptr(grad_psf), n, c, h, w, ctx.ks, device=img.device)
        return grad_img, grad_psf, None


def local_psf_render(input, psf, kernel_size=11):
    """Blur ``input`` with a different PSF at every pixel.

    Same contract as the reference: input [N,C,H,W] (or [C,H,W] -> treated as N=1),
    psf [N,H,W,ks,ks] (any shape that reshapes to it), returns [N,C,H,W]; replicate border,
    no kernel flip, one PSF shared by all channels.  CUDA only.  Differentiable in ``input`` and ``psf``
    (CUDA backward kernels, deterministic; gradients come back in each input's own shape, dtype and device).
    """
    if input.dim() < 4:
        input = input.unsqueeze(0)
    if not input.is_cuda:
        raise RuntimeError("local_psf_render: CUDA tensors required (no CPU fallback in this build)")
    n, c, h, w = input.shape
    ks = int(kernel_size)
    img = input.contiguous().float()
    taps = psf.to(img.device).contiguous().float()
    if taps.numel() != n * h * w * ks * ks:
        raise ValueError(f"psf has {taps.numel()} elements, expected {n}*{h}*{w}*{ks}*{ks}")
    return _LocalPSFRender.apply(img, taps.reshape(n, h, w, ks, ks), ks)


def _bounds(grid, n):
    # the reference's patch limits int(i/grid*H) in Python arithmetic
    return (_nat.ctypes.c_int * (grid + 1))(*[int(i / grid * n) for i in range(grid + 1)])


class _PSFConv(torch.autograd.Function):
    """img [B,C,H,W], psf_map [C, grid*ks, grid*ks]: fp32, contiguous, on one CUDA device."""

    @staticmethod
    def forward(ctx, x, taps, ks, grid):
        B, C, H, W = x.shape
        out = torch.zeros_like(x)            # the reference starts from zeros (rows past the last patch stay 0)
        _nat.call("aadff_render_psf_map_f32", x.data_ptr(), taps.data_ptr(), out.data_ptr(), B, C, H, W, ks, grid,
                  _bounds(grid, H), _bounds(grid, W), device=x.device)
        ctx.save_for_backward(x, taps)
        ctx.ks, ctx.grid = ks, grid
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        x, taps = ctx.saved_tensors
        need_img, need_psf = ctx.needs_input_grad[:2]
        g = grad_out.contiguous()
        B, C, H, W = x.shape
        ks, grid = ctx.ks, ctx.grid
        hb, wb = _bounds(grid, H), _bounds(grid, W)
        grad_img = torch.empty_like(x) if need_img else None
        grad_psf = torch.empty_like(taps) if need_psf else None
        work = None         # only grad_psf_map needs a workspace
        if need_psf:
            work = _nat.workspace(_nat.lib.aadff_render_psf_map_backward_work_bytes(B, C, H, W, ks, grid, hb, wb),
                                  x.device)
        _nat.call("aadff_render_psf_map_backward_f32", x.data_ptr(), taps.data_ptr(), g.data_ptr(), _ptr(grad_img),
                  _ptr(grad_psf), _ptr(work), 0 if work is None else work.numel(), B, C, H, W, ks, grid, hb, wb,
                  device=x.device)
        return grad_img, grad_psf, None, None


def _psf_conv(img, psf_map, ks, grid):
    if not img.is_cuda:
        raise RuntimeError("render_psf / render_psf_map: CUDA tensors required (no CPU fallback in this build)")
    x = img.contiguous().float()
    taps = psf_map.to(x.device).contiguous().float()
    return _PSFConv.apply(x, taps, ks, grid)


def render_psf(img, psf):
    """Render an image with ONE PSF per channel (mirror of deeplens/render_psf.py:12-28): img [B,C,H,W],
    psf [C,ks,ks] -> [B,C,H,W]; reflect padding, true convolution (the PSF is flipped), grouped by channel.
    Differentiable in ``img`` and ``psf`` (CUDA backward kernels, deterministic)."""
    _, ks, ks2 = psf.shape
    if ks != ks2 or ks % 2 == 0:
        raise ValueError("render_psf: square PSFs of odd size only (an even size changes the output shape in the reference)")
    if psf.shape[0] != img.shape[1]:
        raise ValueError("render_psf: PSF must have one kernel per image channel")
    return _psf_conv(img, psf, ks, 1)


def render_psf_map(img, psf_map, grid):
    """Render an image with a grid x grid map of PSFs, one per image patch (mirror of deeplens/render_psf.py:31-73):
    img [B,C,H,W] (or an HxWx3 uint8 array), psf_map [C, grid*ks, grid*ks] -> [B,C,H,W].
    Differentiable in ``img`` and ``psf_map`` (CUDA backward kernels, deterministic)."""
    if not torch.is_tensor(img):
        import numpy as np
        img = torch.tensor((img / 255.).astype(np.float32)).permute(2, 0, 1).unsqueeze(0).to(psf_map.device)
    assert len(img.shape) == 4, 'Input image should be [B, C, H, W]'
    Cpsf, Hpsf, Wpsf = psf_map.shape
    assert Hpsf % grid == 0 and Wpsf % grid == 0, 'PSF map size should be divisible by grid'
    ks = int(Hpsf / grid)
    assert ks % 2 == 1, 'PSF kernel size should be odd'
    assert img.shape[1] == Cpsf, 'PSF map should have the same channel as image'
    return _psf_conv(img, psf_map, ks, grid)


def local_psf_render_high_res(input, psf, patch_size=[320, 480], kernel_size=11):
    """Patch-based local_psf_render (mirror of deeplens/render_psf.py:110-127), kept with the reference's semantics:
    every patch is replicate-padded on its own, so a (ks-1)/2-pixel band at each seam differs from the full-frame
    gather.  The fused kernels never need it (no [N,H,W,k,k] unfold exists to bound); it is here for callers.
    Differentiable through local_psf_render and the slice assignments."""
    import math
    B, C, H, W = input.shape
    out = torch.zeros_like(input)
    for pi in range(int(math.ceil(H / patch_size[0]))):
        for pj in range(int(math.ceil(W / patch_size[1]))):
            li, ui = pi * patch_size[0], min((pi + 1) * patch_size[0], H)
            lj, uj = pj * patch_size[1], min((pj + 1) * patch_size[1], W)
            out[:, :, li:ui, lj:uj] = local_psf_render(input[:, :, li:ui, lj:uj], psf[:, li:ui, lj:uj, :, :],
                                                       kernel_size=kernel_size)
    return out
