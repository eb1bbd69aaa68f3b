"""CPU: oracle/resize_oracle.py against what the reference's own Dataset classes returned
(tests/golden/make_golden_f4_data.py, make_golden_f4_rotate.py).  Every GPU tolerance of
tests/test_gpu_data_path.py rests on this restatement, so it is checked bit for bit."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import resize_oracle as ro

pytest.importorskip("cv2")
pytest.importorskip("torchvision")


def autoagument_draw(seed):
    """AutoAgument's random draws (dff/dataset.py:258-276) in float64, as make_golden_f4_rotate.py replays them:
    (jitter or None, flips, degree or None)."""
    rs = np.random.RandomState(seed)
    jit = (rs.rand(), rs.rand()) if rs.rand() > 0.5 else None
    fl = (1 if rs.rand() > 0.5 else 0) | (2 if rs.rand() > 0.5 else 0)
    deg = rs.randint(0, 180) if rs.rand() > 0.5 else None
    return jit, fl, deg


def test_resize_oracle_reproduces_reference_datasets_bit_for_bit():
    """Matterport3D (down-scale by 2, non-integer factor, identity; AutoAgument jitter with both flips) and
    Middlebury (image through the antialiased resize, depth through cv2.resize): equal to the golden outputs."""
    g = load_golden("kat_j_dataset_prep.npz")
    for tag in "abc":
        aif, dep = ro.matterport_sample(g["mp_bgr"], g["mp_depth"], tuple(g[f"mp_{tag}_size"]))
        assert np.array_equal(aif, g[f"mp_{tag}_aif"]) and np.array_equal(dep, g[f"mp_{tag}_depth"]), tag
    # the golden stores the jitter rounded to float32; the reference used the float64 draws of np.random
    jit, fl, deg = autoagument_draw(int(g["mp_aug_seed"]))
    assert fl == int(g["mp_aug_flips"]) and deg is None and np.array_equal(np.float32(jit), g["mp_aug_jitter"])
    for j in (jit, g["mp_aug_jitter"].astype(np.float64)):
        aif, dep = ro.matterport_sample(g["mp_bgr"], g["mp_depth"], (48, 65), jitter=j, flips=fl)
        assert np.array_equal(aif, g["mp_aug_aif"]) and np.array_equal(dep, g["mp_aug_depth"])
    aif, none = ro.matterport_sample(g["mb_bgr"], None, tuple(g["mb_size"]))
    assert none is None and np.array_equal(aif, g["mb_aif"])
    assert np.array_equal(ro.middlebury_depth(g["mb_depth"], tuple(g["mb_size"]), 1000.0), g["mb_depth_out"])


def test_resize_oracle_reproduces_reference_rotation_bit_for_bit():
    """Matterport3D(train=True) with AutoAgument's spline rotation (alone / with jitter and both flips / with one flip):
    equal to the golden outputs.  This pins the order of the chain: jitter, flips and scipy's rotation run on float64
    arrays and the cast to float32 comes after them (rotating float32 arrays lands 2-4 ulp away)."""
    g = load_golden("kat_l_rotate.npz")
    for i in range(3):
        jit, fl, deg = autoagument_draw(int(g[f"case{i}_seed"]))
        assert fl == int(g[f"case{i}_flips"]) and deg == float(g[f"case{i}_degree"]), i
        aif, dep = ro.matterport_sample(g["bgr"], g["depth"], (48, 65), jitter=jit, flips=fl, degree=deg)
        assert np.array_equal(aif, g[f"case{i}_aif"]) and np.array_equal(dep, g[f"case{i}_depth"]), i
    # the full-resolution rotation without a resize
    aif, dep = ro.matterport_sample(g["bgr"], g["depth"], None, degree=float(g["full_degree"]))
    assert np.array_equal(aif.transpose(1, 2, 0), g["full_aif"]) and np.array_equal(dep[0], g["full_depth"])


def test_bilinear_formula_is_what_cv2_computes():
    """middlebury_depth is cv2.resize itself; bilinear_f64 writes its formula out.  On float64 input with H, W > 1 the
    two agree to 1e-11 (2e-13 relative: double rounding) at every size of the GPU table (up, down, mixed, identity, 1-pixel outputs)."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    for (H, W, h, w) in [(96, 130, 48, 64), (1024, 1280, 480, 640), (1988, 2964, 480, 640), (96, 130, 480, 640),
                         (480, 640, 1080, 320), (37, 50, 37, 50), (37, 50, 1, 9), (37, 50, 9, 1), (2, 2, 7, 5)]:
        x = rng.random((H, W)) * 65.535
        ref = cv2.resize(x, (w, h), interpolation=cv2.INTER_LINEAR).reshape(h, w)
        assert np.abs(ro.bilinear_f64(x, (h, w)) - ref).max() < 1e-11, (H, W, h, w)


def test_antialias_formula_is_what_aten_computes():
    """antialias_f64 writes out the filter of Resize(antialias=True); ATen in float64 evaluates the same numbers (up,
    down, mixed, identity, one-row outputs and inputs), except on the vertical pass of one-column planes."""
    rng = np.random.default_rng(5)
    for (H, W, h, w) in [(96, 130, 48, 65), (1024, 1280, 480, 640), (2000, 2900, 128, 160), (96, 130, 480, 640),
                         (480, 640, 1080, 320), (37, 50, 37, 50), (37, 50, 1, 9), (1, 50, 7, 9), (50, 1, 9, 7),
                         (20, 50, 20, 1)]:
        x = rng.random((2, H, W))
        ref = torch.nn.functional.interpolate(torch.from_numpy(x)[None], (h, w), mode="bilinear", antialias=True,
                                              align_corners=False)[0].numpy()
        assert np.abs(ro.antialias_f64(x, (h, w)) - ref).max() < 1e-13, (H, W, h, w)


def test_antialias_tap_count():
    """aa_taps: ATen's window covers 2 * support input samples, support = max(n_in / n_out, 1)."""
    assert ro.aa_taps(1280, 640) == 4 and ro.aa_taps(1024, 480) == 5 and ro.aa_taps(130, 130) == 2
    assert ro.aa_taps(2900, 160) > 12 and ro.aa_taps(1, 37) == 1
