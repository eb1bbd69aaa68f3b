"""Device-side sample preparation (the CPU half of the reference's Dataset classes, dff/dataset.py, after decoding).

The reference decodes, augments and resizes every sample on the CPU with ``num_workers=0``
(2_aber_aware_dff_aif.py:74); once the focal-stack simulation runs at hundreds of Mpix*slices/s that is the
bottleneck of a training step.  ``preprocess_rgbd`` does ToTensor + colour jitter + flips + the antialiased resize
for a whole batch in one launch from the raw decoded arrays (uint8 BGR image as ``cv.imread`` returns it, uint16 depth).
With ``rotate_deg`` AutoAgument's rotation (scipy.ndimage.rotate, order-3 spline, between the flips and the resize) runs on
the device as well (csrc/spline_rotate_kernel.cuh).  File decoding itself stays with the reference.
"""
import math

import torch

import aadff_native as _nat

__all__ = ["preprocess_rgbd", "rotation_xform"]


@torch.no_grad()
def _cosdg_sindg(degree):
    """scipy.special.cosdg / sindg (what scipy.ndimage.rotate uses: exact at multiples of 90 degrees)."""
    try:
        from scipy import special
        return float(special.cosdg(degree)), float(special.sindg(degree))
    except Exception:
        table = {0: (1.0, 0.0), 90: (0.0, 1.0), 180: (-1.0, 0.0), 270: (0.0, -1.0)}
        return table.get(degree % 360, (math.cos(math.radians(degree)), math.sin(math.radians(degree))))


def rotation_xform(degree, H, W):
    """scipy.ndimage.rotate(x, degree, reshape=False) as (m00, m01, m10, m11, off0, off1): input (row, col) =
    M (output row, col) + off with M = [[cos, sin], [-sin, cos]], off = centre - M centre (float64, like scipy)."""
    c, s = _cosdg_sindg(degree)
    cy, cx = (H - 1) / 2.0, (W - 1) / 2.0
    return [c, s, -s, c, cy - (c * cy + s * cx), cx - (-s * cy + c * cx)]


@torch.no_grad()
def preprocess_rgbd(bgr_u8, depth_u16, size, depth_div=4000.0, depth_mode="antialias", jitter=None, flips=None,
                    rotate_deg=None):
    """bgr_u8 [B,H,W,3] uint8 (cv.imread order) and/or depth_u16 [B,H,W] uint16/int16-as-uint16, CUDA tensors ->
    (aif [B,3,h,w] float32 RGB in [0,1], depth [B,1,h,w] float32 = raw / depth_div), resized to ``size`` = (h, w).

    depth_div: 4000 for Matterport3D (dataset.py:45), 1000 for Middlebury (:199).  depth_mode 'antialias' =
    torchvision Resize(antialias=True) as Matterport3D's transform applies it to the depth; 'cv2' = cv.resize
    INTER_LINEAR as Middlebury does.  jitter [B,2] = (contrast, brightness) of AutoAgument's colour jitter
    (:259-262), contrast < 0 = none; flips [B] uint8: bit 0 = np.flip(axis=1), bit 1 = np.flip(axis=0).
    rotate_deg: sequence of B angles in degrees (AutoAgument draws np.random.randint(0, 180), :276), None / NaN / negative
    = this sample is not rotated: scipy.ndimage.rotate(order 3, 'constant', reshape=False) of every image plane and of the
    depth (then depth[depth<0] = 0) at full resolution between the flips and the resize -- three more launches
    (planes, B-spline prefilter x 2, affine gather) and a B x P x H x W fp32 workspace x 4."""
    ref = bgr_u8 if bgr_u8 is not None else depth_u16
    if not ref.is_cuda:
        raise RuntimeError("preprocess_rgbd: CUDA tensors required (no CPU fallback in this build)")
    dev = ref.device
    B, H, W = ref.shape[0], ref.shape[1], ref.shape[2]
    h, w = int(size[0]), int(size[1])
    aif = depth = None
    if bgr_u8 is not None:
        assert bgr_u8.dtype == torch.uint8 and bgr_u8.shape == (B, H, W, 3)
        bgr_u8 = bgr_u8.contiguous()
        aif = torch.empty(B, 3, h, w, device=dev, dtype=torch.float32)
    if depth_u16 is not None:
        assert depth_u16.dtype in (torch.uint16, torch.int16) and depth_u16.shape == (B, H, W)
        depth_u16 = depth_u16.contiguous()
        depth = torch.empty(B, 1, h, w, device=dev, dtype=torch.float32)
    jit = None if jitter is None else jitter.to(dev, torch.float32).reshape(B, 2).contiguous()
    flp = None if flips is None else flips.to(dev, torch.uint8).reshape(B).contiguous()
    ptr = lambda t: None if t is None else t.data_ptr()
    rot = None
    if rotate_deg is not None:
        rot = [None if (d is None or d != d or d < 0) else float(d) for d in
               (rotate_deg.tolist() if torch.is_tensor(rotate_deg) else list(rotate_deg))]
        assert len(rot) == B, "rotate_deg needs one entry per sample"
        if all(d is None for d in rot):
            rot = None
    if B and rot is not None:
        P = (3 if bgr_u8 is not None else 0) + (1 if depth_u16 is not None else 0)
        nan = float("nan")
        xf = torch.tensor([[nan] * 6 if d is None else rotation_xform(d, H, W) for d in rot], dtype=torch.float64).to(dev)
        planes = torch.empty(B, P, H, W, device=dev, dtype=torch.float32)
        work = torch.empty(2, B, P, H, W, device=dev, dtype=torch.float32)
        rotated = torch.empty_like(planes)
        _nat.call("aadff_prepare_planes_u8", ptr(bgr_u8), ptr(depth_u16), planes.data_ptr(), B, H, W, float(depth_div),
                  ptr(jit), ptr(flp), device=dev)
        _nat.call("aadff_spline_affine_f32", planes.data_ptr(), work.data_ptr(), rotated.data_ptr(), B, P, H, W,
                  xf.data_ptr(), P - 1 if depth_u16 is not None else -1, device=dev)
        _nat.call("aadff_resize_planes_f32", rotated.data_ptr(), ptr(aif), ptr(depth), B, P, H, W, h, w,
                  {"antialias": 0, "cv2": 1}[depth_mode], device=dev)
        return aif, depth
    if B:
        _nat.call("aadff_preprocess_rgbd_u8", ptr(bgr_u8), ptr(depth_u16), ptr(aif), ptr(depth), B, H, W, h, w,
                  float(depth_div), {"antialias": 0, "cv2": 1}[depth_mode], ptr(jit), ptr(flp), device=dev)
    return aif, depth
