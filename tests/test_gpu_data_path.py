"""GPU (pytest -m gpu): the device data path -- preprocess_rgbd_kernel, the spline rotation kernels and
aadff_resize_planes_f32 -- against oracle/resize_oracle.py (torchvision, OpenCV and scipy on the CPU; anchored to the
reference's own Dataset outputs by tests/test_resize_oracle.py) at the sizes the datasets have: Matterport3D frames are
1024x1280, Middlebury 2014 frames about 2000x2900.

Inputs are seeded, piecewise-constant noise with hard edges (weight errors show), depths are uint16 including 0 and
values >= 32768.  Tolerances (max-abs):
  image against float32 ATen                         1e-6
  depth, antialias mode                              5e-7 * max|reference depth|     (about 4 ulp)
  depth, cv2 mode                                    2.5e-7 * max|reference depth|   (about 2 ulp)
  rotated image                                      3e-6
  rotated depth                                      3e-6 * max depth
The rotation is compared with scipy on float64 input while the device rotates the float32 planes; that input
rounding, amplified by the spline prefilter, is what the rotation tolerances cover.
"""
import math

import numpy as np
import pytest
import torch

from oracle import resize_oracle as ro
from oracle import spline_rotate_oracle as so

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")
ndimage = pytest.importorskip("scipy.ndimage")

# (H, W) -> (h, w)
SHAPES = [
    (1024, 1280, 480, 640),       # Matterport3D, the timed shape
    (1024, 1280, 256, 320),
    (1988, 2964, 480, 640),       # Middlebury-like, non-integer factors
    (2000, 2900, 128, 160),       # factors above 5.5 on both axes: windows of more than 12 taps
    (1080, 1920, 37, 50),
    (96, 130, 480, 640),          # up-scaling
    (480, 640, 1080, 320),        # up on one axis, down on the other
    (37, 50, 37, 50),             # identity
    (37, 50, 1, 9),               # one output row
    (37, 50, 9, 1),               # one output column
    (1, 50, 7, 9),                # one input row
    (50, 1, 9, 7),                # one input column
]
SHAPE_IDS = ["x".join(map(str, s[:2])) + "-" + "x".join(map(str, s[2:])) for s in SHAPES]
# the kernel keeps at most PP_MAXW = 12 column weights in registers and recomputes them beyond: keep a row that needs
# that on each axis
assert any(ro.aa_taps(H, h) > 12 and ro.aa_taps(W, w) > 12 for H, W, h, w in SHAPES)

# AutoAgument's colour jitter per image (contrast < 0 = none): none, contrast 0, and contrast 2 with brightness
# +-0.6 (clips at both ends); float32 as the device receives them
JITTER = np.float32([[-1.0, 0.0], [0.0, 0.0], [2.0, 0.6], [2.0, -0.6]])
FLIPS = [0, 1, 2, 3]


def blocks(rng, H, W, p=0.15):
    """Row and column block indices of a piecewise-constant field with random hard edges."""
    return np.cumsum(rng.random(H) < p), np.cumsum(rng.random(W) < p)


def sample_inputs(seed, B, H, W):
    """B images uint8 [B,H,W,3] (BGR) and depths uint16 [B,H,W] with 0 (invalid) and values up to 65535."""
    rng = np.random.default_rng(seed)
    bgr = np.empty((B, H, W, 3), np.uint8)
    dep = np.empty((B, H, W), np.uint16)
    for b in range(B):
        r, c = blocks(rng, H, W)
        bgr[b] = rng.integers(0, 256, (r[-1] + 1, c[-1] + 1, 3), dtype=np.uint8)[r][:, c]
        r, c = blocks(rng, H, W)
        d = rng.integers(1, 65536, (r[-1] + 1, c[-1] + 1)).astype(np.uint16)
        d[rng.random(d.shape) < 0.1] = 0
        d[0, 0], d[-1, -1] = 0, 65535
        dep[b] = d[r][:, c]
    return bgr, dep


def to_device(bgr, dep):
    """numpy uint8 / uint16 -> CUDA uint8 / uint16 tensors (uint16 through the int16 view)."""
    d16 = torch.from_numpy(np.ascontiguousarray(dep).view(np.int16)).view(torch.uint16)
    return torch.from_numpy(np.ascontiguousarray(bgr)).cuda(), d16.cuda()


def jitter_of(b):
    c, br = JITTER[b]
    return None if c < 0 else (float(c), float(br))


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def report(test, tag, **errs):
    print(f"[data-path] {test:10s} {tag:22s} " + "  ".join(f"{k} {v:.3e}" for k, v in errs.items()))


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


@pytest.mark.parametrize("H,W,h,w", SHAPES, ids=SHAPE_IDS)
def test_antialias_resize_matches_torchvision(pkg, H, W, h, w):
    """preprocess_rgbd in antialias mode (Matterport3D: /255, jitter, flips, Resize(antialias=True) of image and depth)
    for a batch of four with every jitter kind and every flip code, and image-only / depth-only calls.

    The depth tolerance is 5e-7 * max depth, not 2.5e-7: over windows of up to 78 taps per axis the kernel accumulates
    each row with FMAs from zero while ATen multiplies and adds separately, and the two fp32 sums drift apart by up to
    3.5e-7 * max depth (3 ulp) on the Middlebury-sized rows.  For one-column outputs the reference is the filter
    written out in float64 (oracle antialias_f64): ATen's CPU vertical pass is wrong on one-column planes."""
    B = 4
    bgr, dep = sample_inputs(H * 7 + W, B, H, W)
    gb, gd = to_device(bgr, dep)
    aif, d = pkg.preprocess_rgbd(gb, gd, (h, w), depth_div=4000.0, jitter=torch.from_numpy(JITTER),
                                 flips=torch.tensor(FLIPS, dtype=torch.uint8))
    only_img, none_d = pkg.preprocess_rgbd(gb, None, (h, w), jitter=torch.from_numpy(JITTER),
                                           flips=torch.tensor(FLIPS, dtype=torch.uint8))
    none_a, only_d = pkg.preprocess_rgbd(None, gd, (h, w), depth_div=4000.0, flips=torch.tensor(FLIPS, dtype=torch.uint8))
    assert none_d is None and none_a is None and aif.shape == (B, 3, h, w) and d.shape == (B, 1, h, w)
    aif, d, only_img, only_d = (t.cpu().numpy() for t in (aif, d, only_img, only_d))
    ea = ed = 0.0
    for b in range(B):
        ra, rd = ro.matterport_sample(bgr[b], dep[b], (h, w), jitter=jitter_of(b), flips=FLIPS[b], div=4000.0)
        if w == 1 and h != H:
            fa, fd = ro.matterport_sample(bgr[b], dep[b], None, jitter=jitter_of(b), flips=FLIPS[b], div=4000.0)
            ra, rd = ro.antialias_f64(fa, (h, w)), ro.antialias_f64(fd, (h, w))
        dmax = float(np.abs(rd).max())
        ea = max(ea, maxabs(aif[b], ra), maxabs(only_img[b], ra))
        ed = max(ed, max(maxabs(d[b], rd), maxabs(only_d[b], rd)) / dmax)
    report("antialias", f"{H}x{W}->{h}x{w}", image=ea, depth_rel=ed)
    assert ea <= 1e-6 and ed <= 5e-7


@pytest.mark.parametrize("H,W,h,w", SHAPES, ids=SHAPE_IDS)
def test_cv2_depth_resize_matches_opencv(pkg, H, W, h, w):
    """preprocess_rgbd(depth_mode='cv2') (Middlebury: cv2.resize(depth / 1000, INTER_LINEAR) on float64) against
    OpenCV, with flips.  On a single-row or single-column input OpenCV 4.13 leaves its double-precision formula for a
    path with float32 coordinates and weights (up to ~1e-6 relative away); there the depth is held to 2.5e-7 against
    that formula written out in float64 (oracle bilinear_f64) and to 2e-6 against cv2 itself."""
    B = 2
    bgr, dep = sample_inputs(H * 11 + W, B, H, W)
    gb, gd = to_device(bgr, dep)
    fl = [0, 3]
    _, d = pkg.preprocess_rgbd(None, gd, (h, w), depth_div=1000.0, depth_mode="cv2",
                               flips=torch.tensor(fl, dtype=torch.uint8))
    aif, d2 = pkg.preprocess_rgbd(gb, gd, (h, w), depth_div=1000.0, depth_mode="cv2",
                                  flips=torch.tensor(fl, dtype=torch.uint8))
    aa, _ = pkg.preprocess_rgbd(gb, None, (h, w), flips=torch.tensor(fl, dtype=torch.uint8))
    assert torch.equal(d, d2) and torch.equal(aif, aa)        # the image keeps the antialiased resize
    d = d.cpu().numpy()
    e_cv = e_f64 = e_abs = 0.0
    for b in range(B):
        src = dep[b]
        if fl[b] & 1:
            src = src[:, ::-1]
        if fl[b] & 2:
            src = src[::-1]
        ref = ro.middlebury_depth(src, (h, w), 1000.0)
        dmax = float(np.abs(ref).max())
        e_abs = max(e_abs, maxabs(d[b], ref))
        e_cv = max(e_cv, maxabs(d[b], ref) / dmax)
        e_f64 = max(e_f64, maxabs(d[b, 0], ro.bilinear_f64(src / 1000.0, (h, w))) / dmax)
    report("cv2", f"{H}x{W}->{h}x{w}", depth_m_cv2=e_abs, depth_rel_cv2=e_cv, depth_rel_f64=e_f64)
    assert e_f64 <= 2.5e-7
    assert e_cv <= (2e-6 if min(H, W) == 1 else 2.5e-7)


def _rotation_refs(bgr, dep, degs, sizes):
    """Oracle outputs of matterport_sample with jitter_of(b), FLIPS[b] and degs[b] (None = not rotated) per sample,
    resized to each of ``sizes``: {size: [(aif, depth) per sample]}; scipy runs once per sample."""
    out = {s: [] for s in sizes}
    for b in range(len(degs)):
        fa, fd = ro.matterport_sample(bgr[b], dep[b], None, jitter=jitter_of(b), flips=FLIPS[b], degree=degs[b])
        H, W = fd.shape[1:]
        for s in sizes:
            out[s].append((fa, fd) if s == (H, W) else (ro.resize_aa(fa, s), ro.resize_aa(fd, s)))
    return out


def _check_rotation(pkg, bgr, dep, rot, sizes, tag):
    B = len(rot)
    gb, gd = to_device(bgr, dep)
    refs = _rotation_refs(bgr, dep, [None if d != d else d for d in rot], sizes)
    for s in sizes:
        aif, d = pkg.preprocess_rgbd(gb, gd, s, depth_div=4000.0, rotate_deg=rot, jitter=torch.from_numpy(JITTER[:B]),
                                     flips=torch.tensor(FLIPS[:B], dtype=torch.uint8))
        aif, d = aif.cpu().numpy(), d.cpu().numpy()
        ea = max(maxabs(aif[b], refs[s][b][0]) for b in range(B))
        ed = max(maxabs(d[b], refs[s][b][1]) / float(np.abs(refs[s][b][1]).max() or 1.0) for b in range(B))
        report("rotation", f"{tag}->{s[0]}x{s[1]}", image=ea, depth_rel=ed)
        assert ea <= 3e-6 and ed <= 3e-6, (tag, s)


def test_rotation_at_full_size(pkg):
    """AutoAgument's spline rotation of a 1024x1280 batch (17, 90 and 179 degrees and one sample without rotation, with
    the per-image jitter and flips) with the resize to 480x640 and without a resize, against scipy.ndimage.rotate."""
    bgr, dep = sample_inputs(5, 4, 1024, 1280)
    _check_rotation(pkg, bgr, dep, [17.0, 90.0, 179.0, float("nan")], [(480, 640), (1024, 1280)], "1024x1280")


@pytest.mark.parametrize("H,W", [(1, 40), (40, 1), (2, 37), (37, 2), (16, 45), (45, 16), (33, 47), (47, 33), (16, 16)])
def test_rotation_of_degenerate_planes(pkg, H, W):
    """Planes with H or W of 1, 2, 16 (every pixel on the mirror path of the 33-tap prefilter) and 33, with and without
    a resize."""
    bgr, dep = sample_inputs(H * 100 + W, 4, H, W)
    _check_rotation(pkg, bgr, dep, [17.0, 90.0, 179.0, float("nan")], [(H, W), (max(1, H // 2 + 3), W + 5)], f"{H}x{W}")


def _call_abi(pkg, fn, *args):
    nat = pkg.native
    nat.check(getattr(nat.lib, fn)(*args, torch.cuda.current_stream().cuda_stream))


@pytest.mark.parametrize("P,clamp", [(1, True), (1, False), (3, False), (4, True), (4, False)])
def test_three_step_abi_with_general_affine(pkg, P, clamp):
    """aadff_prepare_planes_u8 -> aadff_spline_affine_f32 -> aadff_resize_planes_f32 called directly, each step against
    its own reference on the previous step's device output: the planes against the oracle's float32 planes; a general
    affine map (scale and shear, and a rotation; one sample copied) against scipy.ndimage.affine_transform(order=3,
    'constant', prefilter=True), with the depth plane clamped at 0 or not; the resize in both depth modes against
    torchvision and OpenCV."""
    B, H, W, h, w = 3, 300, 410, 128, 170
    bgr, dep = sample_inputs(P * 10 + clamp, B, H, W)
    gb, gd = to_device(bgr, dep)
    img_on, dep_on = P >= 3, P != 3
    jit = torch.from_numpy(JITTER[:B]).cuda()
    fl = torch.tensor(FLIPS[1:B + 1], dtype=torch.uint8).cuda()
    planes = torch.empty(B, P, H, W, device="cuda")
    _call_abi(pkg, "aadff_prepare_planes_u8", gb.data_ptr() if img_on else None, gd.data_ptr() if dep_on else None,
              planes.data_ptr(), B, H, W, 1000.0, jit.data_ptr(), fl.data_ptr())
    pl = planes.cpu().numpy()
    for b in range(B):
        ra, rd = ro.matterport_sample(bgr[b] if img_on else None, dep[b] if dep_on else None, None,
                                      jitter=jitter_of(b), flips=FLIPS[b + 1], div=1000.0)
        ref = np.concatenate([x for x in (ra, rd) if x is not None])
        assert maxabs(pl[b], ref) <= 6e-8 * float(np.abs(ref).max()), b     # within half an ulp: /div in fp32

    # sample 0: scale + shear, sample 1: a rotation by 31 degrees, sample 2: NaN = copied
    shear = [1.13, 0.21, -0.17, 0.87, -7.5, 12.25]
    xf = torch.tensor([shear, so.rotation_xform(31.0, H, W).tolist(), [math.nan] * 6], dtype=torch.float64).cuda()
    work = torch.empty(2, B, P, H, W, device="cuda")
    out = torch.empty_like(planes)
    cp = P - 1 if (clamp and dep_on) else -1
    _call_abi(pkg, "aadff_spline_affine_f32", planes.data_ptr(), work.data_ptr(), out.data_ptr(), B, P, H, W,
              xf.data_ptr(), cp)
    rot = out.cpu().numpy()
    assert np.array_equal(rot[2], pl[2])
    negative = False
    for b in range(2):
        M = np.array(xf[b, :4].cpu().tolist()).reshape(2, 2)
        for p in range(P):
            ref = ndimage.affine_transform(pl[b, p].astype(np.float64), M, offset=xf[b, 4:].cpu().numpy(), order=3,
                                           mode="constant", cval=0.0, prefilter=True)
            is_depth = dep_on and p == P - 1
            if is_depth:
                negative |= bool((ref < -1e-3).any())
                if cp >= 0:
                    ref[ref < 0] = 0
            scale = float(np.abs(ref).max()) if is_depth else 1.0
            e = maxabs(rot[b, p], ref) / scale
            report("affine", f"P{P} clamp{cp} b{b} p{p}", err=e)
            assert e <= 3e-6, (b, p)
    if dep_on:
        assert negative          # the spline overshoots at the depth edges, so the clamp is exercised

    for mode in (0, 1):
        aif = torch.empty(B, 3, h, w, device="cuda") if img_on else None
        dd = torch.empty(B, 1, h, w, device="cuda") if dep_on else None
        _call_abi(pkg, "aadff_resize_planes_f32", out.data_ptr(), aif.data_ptr() if img_on else None,
                  dd.data_ptr() if dep_on else None, B, P, H, W, h, w, mode)
        for b in range(B):
            if img_on:
                e = maxabs(aif[b].cpu().numpy(), ro.resize_aa(rot[b, :3], (h, w)))
                report("resize", f"P{P} mode{mode} b{b} image", err=e)
                assert e <= 1e-6
            if dep_on:
                src = rot[b, P - 1]
                ref = ro.resize_aa(src[None], (h, w)) if mode == 0 else \
                    cv2.resize(src.astype(np.float64), (w, h), interpolation=cv2.INTER_LINEAR)[None]
                e = maxabs(dd[b].cpu().numpy(), ref) / float(np.abs(ref).max())
                report("resize", f"P{P} mode{mode} b{b} depth", depth_rel=e)
                assert e <= (5e-7 if mode == 0 else 2.5e-7)
