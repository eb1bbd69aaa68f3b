"""Which kernel specialisation each entry point launches (pytest -m gpu).

The host code of libaadff.so (csrc/aadff_api.cu) picks a template instantiation per launch: the fused render kernel's
<TRACE, PRED, UNI, TA> from the mode, the network depth and the weight ring; the strip / register-streaming / generic
gather and the strip plan <KS, CN, SL, NW, SPX> from ks, W and C; the kernel-size instantiation of the backward, PSF-map
and thin-lens kernels.  A wrong choice there leaves every output bit-identical (the specialisations compute the same
products in the same order) and only costs throughput, so no output test can see it.  This test records the kernel
names of each launch with torch.profiler and compares them with tests/golden/dispatch_kernels.json.

Regenerate the table (on a B200, only when a dispatch change is intended):
    python tests/test_gpu_dispatch.py --record tests/golden/dispatch_kernels.json
"""
import json
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import focal_stack_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu

TABLE = os.path.join(ROOT, "tests", "golden", "dispatch_kernels.json")
MODES = ("parity", "econ8", "econ", "mixed", "fast")
NAME = re.compile(r"aadff::(\w+(?:<[^()]*>)?)")


def launched(fn):
    """Names (with template arguments) of the libaadff kernels that fn() launches, in launch order."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kernels.sort(key=lambda e: e.time_range.start)
    return [m.group(1) for m in (NAME.search(e.name) for e in kernels) if m]


def lens(pkg, ks, hidden_layers=None):
    l = pkg.PSFNet(kernel_size=ks, device="cuda")
    if hidden_layers is not None:
        from deeplens.psfnet_arch import MLP
        torch.manual_seed(40 + hidden_layers)
        l.psfnet = MLP(in_features=4, out_features=ks * ks, hidden_features=256, hidden_layers=hidden_layers).to("cuda")
        l.psfnet._evaluator = l._mlp_eval
        l._native = None
    return l


def stack_inputs():
    img, dm = orc.synthetic_rgbd(1, 16, 24, seed=3)
    foc = -orc.synthetic_focus(dm, 2) * 1e3
    return img.cuda(), -dm.cuda() * 1e3, foc.cuda()


def record_render_stack(pkg):
    img, dep, foc = stack_inputs()
    out = {}
    for ks in (5, 11, 13, 15, 31):
        l = lens(pkg, ks)
        for mode in MODES:
            out[f"render_stack/ks{ks}/{mode}"] = launched(lambda: l.render_stack(img, dep, foc, mode=mode))
        if ks == 11:
            out["render_stack_rows/ks11/econ8"] = launched(lambda: l.render_stack_rows(img, dep, foc, 1, 3, mode="econ8"))
    for hl in (0, 2):
        l = lens(pkg, 11, hl)
        for mode in ("econ8", "mixed"):
            out[f"render_stack/ks11/hidden{hl}/{mode}"] = launched(lambda: l.render_stack(img, dep, foc, mode=mode))
    return out


def record_pred(pkg):
    x = torch.rand(300, 4, generator=torch.Generator().manual_seed(1)).cuda()
    out = {}
    for ks in (11, 13, 31):
        l = lens(pkg, ks)
        for mode in MODES:
            out[f"pred/ks{ks}/{mode}"] = launched(lambda: l.pred(x, mode=mode))
    return out


def record_local_psf_render(pkg):
    gen = torch.Generator().manual_seed(2)
    out = {}
    for ks in (1, 3, 7, 11, 15, 17, 31, 33):
        for W in (64, 66, 512, 640):
            for C in (1, 3, 4):
                img = torch.rand(1, C, 4, W, generator=gen).cuda()
                psf = torch.rand(1, 4, W, ks, ks, generator=gen).cuda()
                out[f"local_psf_render/ks{ks}/W{W}/C{C}"] = launched(lambda: pkg.local_psf_render(img, psf, ks))
    return out


def record_local_psf_render_backward(pkg):
    """dP and dimg: strip kernels for 3 <= ks <= 15 and W % 4 == 0 (dP: C <= 4), the generic kernels otherwise."""
    gen = torch.Generator().manual_seed(3)
    out = {}
    for ks in (3, 11, 15, 17):
        for W in (64, 66):
            for C in (1, 3, 5):
                img = torch.rand(1, C, 6, W, generator=gen).cuda().requires_grad_(True)
                psf = torch.rand(1, 6, W, ks, ks, generator=gen).cuda().requires_grad_(True)
                y = pkg.local_psf_render(img, psf, ks)
                g = torch.rand_like(y)
                out[f"local_psf_render_backward/ks{ks}/W{W}/C{C}"] = launched(lambda: y.backward(g))
    return out


def record_psf_map_and_thinlens(pkg):
    from deeplens.psfnet import ThinLens
    from deeplens.render_psf import render_psf_map
    gen = torch.Generator().manual_seed(4)
    out = {}
    for (B, C, H, W, ks, grid) in [(2, 3, 40, 48, 5, 3), (1, 3, 80, 96, 31, 2)]:
        img = torch.rand(B, C, H, W, generator=gen).cuda().requires_grad_(True)
        psf_map = torch.rand(C, grid * ks, grid * ks, generator=gen).cuda().requires_grad_(True)
        key = f"render_psf_map/ks{ks}/grid{grid}"
        out[key] = launched(lambda: render_psf_map(img, psf_map, grid))
        y = render_psf_map(img, psf_map, grid)
        g = torch.rand_like(y)
        out[key + "/backward"] = launched(lambda: y.backward(g))
    for (C, H, W, ks) in [(3, 40, 64, 11), (3, 72, 200, 31)]:
        tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=ks, sensor_size=[36.0, 24.0], sensor_res=(H, W)).to("cuda")
        im = torch.rand(1, C, H, W, generator=gen).cuda()
        dp = (300 + 6000 * torch.rand(1, 1, H, W, generator=gen)).cuda()
        fc = (500 + 3000 * torch.rand(1, generator=gen)).cuda()
        out[f"thinlens/ks{ks}/{H}x{W}"] = launched(lambda: tl.render(im, dp, fc))
    return out


GROUPS = [record_render_stack, record_pred, record_local_psf_render, record_local_psf_render_backward,
          record_psf_map_and_thinlens]


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


@pytest.fixture(scope="module")
def table():
    with open(TABLE) as f:
        return json.load(f)


@pytest.mark.parametrize("group", GROUPS, ids=lambda g: g.__name__[len("record_"):])
def test_dispatch_matches_table(pkg, table, group):
    got = group(pkg)
    assert all(got.values()), [k for k, v in got.items() if not v]      # every case launches a libaadff kernel
    expected = {k: table[k] for k in got if k in table}
    assert sorted(expected) == sorted(got), sorted(set(got) - set(table))
    wrong = {k: (got[k], expected[k]) for k in got if got[k] != expected[k]}
    assert not wrong, json.dumps(wrong, indent=1)


if __name__ == "__main__":
    if len(sys.argv) != 3 or sys.argv[1] != "--record":
        sys.exit("usage: python tests/test_gpu_dispatch.py --record TABLE.json")
    import aadff_b200
    rec = {}
    for group in GROUPS:
        rec.update(group(aadff_b200))
    with open(sys.argv[2], "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"{len(rec)} cases, {sum(len(v) for v in rec.values())} launches -> {sys.argv[2]}")
