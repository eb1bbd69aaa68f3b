"""CPU oracle for the sample preparation of the reference's Dataset classes (dff/dataset.py: Matterport3D :43-52,
Middlebury :190-205, AutoAgument :252-286), after file decoding.

TEST INFRASTRUCTURE ONLY (see focal_stack_oracle.py): only ``tests/`` may import this file.

The chain is restated here with the same third-party calls the reference makes, at the same precision:

* ``matterport_sample``  BGR -> RGB and ``/ 255`` in float64; AutoAgument's colour jitter
  ``clip(0.5 + contrast * (x - 0.5) + brightness, 0, 1)`` in float64; the flips; optionally
  ``scipy.ndimage.rotate(order=3, reshape=False)`` of the image and of the depth, then ``depth[depth < 0] = 0``, all
  on float64 arrays; ``astype(float32)``; torchvision ``Resize(antialias=True)`` on float32 CPU tensors (ATen's
  ``_upsample_bilinear2d_aa``).  The depth is ``depth_u16 / div`` in float64 and goes through the same flips,
  rotation, cast and resize.  The rotation sees float64 input: rotating the float32-cast arrays instead differs from
  the reference by 2-4 ulp after the resize.
* ``middlebury_depth``   ``cv2.resize(depth_u16 / div, (w, h), interpolation=INTER_LINEAR)`` on float64, cast to
  float32 (on float64 input cv2 evaluates the plain bilinear formula in double).
* ``antialias_f64``      the antialiased filter written out in float64 (see there for where ATen leaves it).
* ``bilinear_f64``       the bilinear formula cv2 evaluates, written out in float64 (see there for where cv2 leaves it).
* ``aa_taps``            the length of ATen's antialias filter window along one axis (what decides whether the device
  kernel keeps the column weights in registers).

Parity pin: ``tests/test_resize_oracle.py`` reproduces the reference's own outputs stored in
``tests/golden/kat_j_dataset_prep.npz`` and ``tests/golden/kat_l_rotate.npz``.
"""
import cv2
import numpy as np
import scipy.ndimage
import torch
import torchvision.transforms.functional as TF


def resize_aa(planes_f32, size):
    """[C,H,W] float32 numpy -> [C,h,w] float32: torchvision Resize(size, antialias=True) on a float32 CPU tensor."""
    return TF.resize(torch.from_numpy(np.ascontiguousarray(planes_f32)), list(size), antialias=True).numpy()


def matterport_sample(bgr_u8, depth_u16, size, jitter=None, flips=0, degree=None, div=4000.0):
    """One sample of Matterport3D(train=...) as __getitem__ returns it, for given AutoAgument draws.

    bgr_u8 [H,W,3] uint8 (cv.imread order) or None, depth_u16 [H,W] uint16 or None, size (h, w), or None for the
    float32 planes before the resize (so that one rotation can be resized to several sizes with ``resize_aa``);
    jitter (contrast, brightness) or None; flips bit 0 = np.flip(axis=1), bit 1 = np.flip(axis=0);
    degree: rotation angle in degrees or None.  Returns (aif [3,h,w], depth [1,h,w]) float32 numpy (None where the
    input is None)."""
    aif = depth = None
    if bgr_u8 is not None:
        x = bgr_u8[..., ::-1] / 255.0
        if jitter is not None:
            c, b = float(jitter[0]), float(jitter[1])
            x = np.clip(0.5 + c * (x - 0.5) + b, 0.0, 1.0)
        aif = x
    if depth_u16 is not None:
        depth = np.asarray(depth_u16, dtype=np.uint16) / div
    for bit, axis in ((1, 1), (2, 0)):
        if flips & bit:
            aif = None if aif is None else np.flip(aif, axis)
            depth = None if depth is None else np.flip(depth, axis)
    if degree is not None:
        if aif is not None:
            aif = scipy.ndimage.rotate(aif, degree, reshape=False)
        if depth is not None:
            depth = scipy.ndimage.rotate(depth, degree, reshape=False)
            depth[depth < 0] = 0
    aif = None if aif is None else aif.astype(np.float32).transpose(2, 0, 1)
    depth = None if depth is None else depth.astype(np.float32)[None]
    if size is not None:
        aif = None if aif is None else resize_aa(aif, size)
        depth = None if depth is None else resize_aa(depth, size)
    return aif, depth


def middlebury_depth(depth_u16, size, div=1000.0):
    """Middlebury's depth: cv2.resize(depth / div, (w, h), INTER_LINEAR) on float64 -> [1,h,w] float32."""
    h, w = int(size[0]), int(size[1])
    d = np.asarray(depth_u16, dtype=np.uint16) / div
    return cv2.resize(d, (w, h), interpolation=cv2.INTER_LINEAR).reshape(1, h, w).astype(np.float32)


def bilinear_f64(x, size):
    """[H,W] float64 -> [h,w] float64: the INTER_LINEAR formula written out -- source coordinate (o + 0.5) * (n / m) - 0.5,
    floor and fraction in double; below 0 -> index 0, fraction 0; at or beyond n - 1 -> index n - 1, fraction 0.  cv2.resize
    evaluates exactly this on float64 input with H, W > 1; a single-row or single-column input takes another OpenCV path
    with float32 coordinates and weights (up to ~1e-6 relative away)."""
    x = np.asarray(x, dtype=np.float64)
    (H, W), (h, w) = x.shape, (int(size[0]), int(size[1]))

    def axis(m, n):
        c = (np.arange(m) + 0.5) * (n / m) - 0.5
        s = np.floor(c)
        f = c - s
        s = s.astype(np.int64)
        f = np.where((s < 0) | (s >= n - 1), 0.0, f)
        s = np.clip(s, 0, n - 1)
        return s, np.minimum(s + 1, n - 1), f

    y0, y1, fy = axis(h, H)
    x0, x1, fx = axis(w, W)
    fy, fx = fy[:, None], fx[None, :]
    top = x[y0][:, x0] * (1 - fx) + x[y0][:, x1] * fx
    bot = x[y1][:, x0] * (1 - fx) + x[y1][:, x1] * fx
    return top * (1 - fy) + bot * fy


def _aa_matrix(n_in, n_out):
    """[n_out, n_in] float64 weights of ATen's antialiased bilinear filter along one axis (triangle of support
    max(n_in / n_out, 1), window as aa_taps, each row divided by its sum)."""
    scale = n_in / n_out
    support, inv = (scale, 1.0 / scale) if scale >= 1.0 else (1.0, 1.0)
    m = np.zeros((n_out, n_in))
    for i in range(n_out):
        centre = scale * (i + 0.5)
        lo = max(0, int(centre - support + 0.5))
        j = np.arange(lo, min(n_in, int(centre + support + 0.5)))
        w = np.maximum(0.0, 1.0 - np.abs((j - centre + 0.5) * inv))
        m[i, j] = w / w.sum()
    return m


def antialias_f64(planes, size):
    """[C,H,W] -> [C,h,w] float64: Resize(antialias=True) written out as the separable filter in float64.  ATen
    evaluates this formula, except that its CPU vertical pass is wrong on planes one column wide (torch 2.11:
    37x1 -> 9x1 is off by 0.4 on random data, in float32 and float64 alike), which Resize((h, 1)) runs into."""
    x = np.asarray(planes, dtype=np.float64)
    (H, W), (h, w) = x.shape[1:], (int(size[0]), int(size[1]))
    return _aa_matrix(H, h) @ x @ _aa_matrix(W, w).T


def aa_taps(n_in, n_out):
    """Largest window of ATen's antialiased bilinear filter along one axis: n_in -> n_out samples (the support grows
    with the down-scaling factor; at most 2 * ceil(scale) + 1 taps)."""
    scale = n_in / n_out
    support = max(scale, 1.0)
    taps = 0
    for i in range(n_out):
        centre = scale * (i + 0.5)
        lo = max(0, int(centre - support + 0.5))
        taps = max(taps, min(n_in, int(centre + support + 0.5)) - lo)
    return taps
