"""CPU-side tests (pytest -m "not gpu"): the C-ABI library loads and exports every symbol the
header declares, argument validation works without a device, the Python drop-in surface mirrors
the reference's, nothing falls back to a CPU path, and the multi-rank partitioning logic gathers
to the single-rank result under a world_size-2 gloo group."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_golden

CKPT = os.path.join(GOLDEN, "rf50mm_PSFNet480x640_ks11.pkl")


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


def test_library_exports_every_header_symbol(pkg):
    nat = pkg.native
    with open(os.path.join(ROOT, "include", "aadff.h")) as f:
        declared = sorted(set(re.findall(r"\b(aadff_[a-z0-9_]+)\s*\(", f.read())))
    assert len(declared) >= 11
    for name in declared:
        assert hasattr(nat.lib, name), name
    assert nat.lib.aadff_version() == 200
    assert nat.lib.aadff_launch_count() >= 0
    sass_free = subprocess.run(["nm", "-D", nat.LIB_PATH], capture_output=True, text=True).stdout
    for name in declared:
        assert re.search(rf"\bT {name}\b", sass_free), f"{name} not an exported text symbol"


def test_argument_validation_needs_no_device(pkg):
    lib = pkg.native.lib
    assert lib.aadff_local_psf_render_f32(None, None, None, 1, 3, 8, 8, 11, None) == -1
    assert b"null" in lib.aadff_last_error()
    assert lib.aadff_local_psf_render_f32(8, 8, 8, 1, 3, 8, 8, 10, None) == -1
    assert lib.aadff_psfnet_pred_f32(None, None, None, 4, None) == -1
    assert lib.aadff_psfnet_create(None, None, None, 11, 11, 0, None) == -1
    assert lib.aadff_psfnet_destroy(None) == 0


def test_trainer_argument_validation_needs_no_device(pkg):
    """aadff_trainer_create / _step refuse what would make a step read outside its buffers (dims that are not
    [4, hidden widths, kk]) and the AdamW settings torch.optim.AdamW refuses, before touching a device."""
    lib = pkg.native.lib
    c_f32p = ctypes.POINTER(ctypes.c_float)

    def create(dims, batch=8, beta1=0.9, beta2=0.999, eps=1e-8, wd=1e-2, null_layer=None):
        # every layer gets buffers as large as its dims ask for, so that a call the library accepts (on a box with a
        # GPU it goes on to copy dims[l+1] * dims[l] weights and dims[l+1] biases per layer) reads only what it owns
        n = len(dims) - 1
        ws = [np.zeros(max(dims[l + 1], 1) * max(dims[l], 1), np.float32) for l in range(n)]
        bs = [np.zeros(max(dims[l + 1], 1), np.float32) for l in range(n)]
        wp = (c_f32p * n)(*[c_f32p() if l == null_layer else w.ctypes.data_as(c_f32p) for l, w in enumerate(ws)])
        bp = (c_f32p * n)(*[b.ctypes.data_as(c_f32p) for b in bs])
        handle = ctypes.c_void_p()
        rc = lib.aadff_trainer_create(wp, bp, (ctypes.c_int * (n + 1))(*dims), n, batch, beta1, beta2, eps, wd, 0,
                                      ctypes.byref(handle))
        return rc, lib.aadff_last_error().decode(), handle

    nan, inf = float("nan"), float("inf")
    bad = [
        (dict(dims=[5, 64, 9]), "start with 4"), (dict(dims=[3, 64, 9]), "start with 4"),
        (dict(dims=[4, 60, 9]), "hidden widths"), (dict(dims=[4, 0, 9]), "hidden widths"),
        (dict(dims=[4, -8, 9]), "hidden widths"), (dict(dims=[4, 264, 9]), "hidden widths"),
        (dict(dims=[4, 64, 256, 0]), "kk"), (dict(dims=[4, -1]), "kk"),
        (dict(dims=[4] + [64] * 16 + [9]), "n_layers"), (dict(dims=[4, 64, 9], batch=0), "batch"),
        (dict(dims=[4, 64, 9], null_layer=1), "null layer"),
        (dict(dims=[4, 64, 9], beta1=1.0), "beta1"), (dict(dims=[4, 64, 9], beta1=-0.1), "beta1"),
        (dict(dims=[4, 64, 9], beta1=nan), "beta1"), (dict(dims=[4, 64, 9], beta2=1.0), "beta2"),
        (dict(dims=[4, 64, 9], beta2=nan), "beta2"), (dict(dims=[4, 64, 9], eps=-1e-8), "eps"),
        (dict(dims=[4, 64, 9], eps=inf), "eps"), (dict(dims=[4, 64, 9], eps=nan), "eps"),
        (dict(dims=[4, 64, 9], wd=-1e-2), "weight_decay"), (dict(dims=[4, 64, 9], wd=inf), "weight_decay"),
        (dict(dims=[4, 64, 9], wd=nan), "weight_decay"),
    ]
    for kwargs, name in bad:
        rc, msg, _ = create(**kwargs)
        assert rc == -1 and name in msg, (kwargs, rc, msg)
    # the edges that are valid get past validation (on a box without a GPU, to the device selection)
    for kwargs in (dict(dims=[4, 1]), dict(dims=[4, 8, 256, 961], beta1=0.0, beta2=0.0, eps=0.0, wd=0.0)):
        rc, msg, handle = create(**kwargs)
        if rc == 0:
            lib.aadff_trainer_destroy(handle)
        else:
            assert rc == -2 and "CUDA device" in msg, (kwargs, rc, msg)
    for lr in (nan, inf, -inf, -1e-4):            # checked first, so no handle is needed (every pointer is null)
        assert lib.aadff_trainer_step(None, None, None, lr, None, None) == -1
        assert b"lr" in lib.aadff_last_error()
    # NativeTrainer checks layer shapes before the library copies dims[l+1] * dims[l] floats from each buffer
    Ws = [np.zeros((64, 4), np.float32), np.zeros((256, 64), np.float32), np.zeros((9, 256), np.float32)]
    bs = [np.zeros(64, np.float32), np.zeros(256, np.float32), np.zeros(9, np.float32)]
    for l, W in ((1, np.zeros((256, 63), np.float32)), (2, np.zeros((9, 255), np.float32))):
        with pytest.raises(ValueError, match=f"layer {l}"):
            pkg.native.NativeTrainer(Ws[:l] + [W] + Ws[l + 1:], bs, 8, 0)
    with pytest.raises(ValueError, match="layer 1"):
        pkg.native.NativeTrainer(Ws, bs[:1] + [np.zeros(255, np.float32)] + bs[2:], 8, 0)
    with pytest.raises(ValueError, match="biases"):
        pkg.native.NativeTrainer(Ws, bs[:2], 8, 0)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks behaviour on a box without a GPU")
def test_no_cpu_fallback(pkg):
    """Without a device every compute entry fails loudly; nothing silently computes on the host."""
    from deeplens.psfnet import PSFNet
    from deeplens.render_psf import local_psf_render
    lens = PSFNet(kernel_size=11, device="cpu")
    lens.load_net(CKPT)
    with pytest.raises(RuntimeError, match="CUDA"):
        lens.render(torch.rand(1, 3, 8, 8), -torch.rand(1, 1, 8, 8) * 1000, torch.tensor([-1000.0]))
    with pytest.raises(RuntimeError, match="CUDA"):
        lens.pred(torch.zeros(2, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        local_psf_render(torch.rand(1, 3, 8, 8), torch.rand(1, 8, 8, 3, 3), 3)
    with pytest.raises(pkg.native.AadffError):
        pkg.native.NativePSFNet([np.zeros((64, 4), np.float32), np.zeros((256, 64), np.float32),
                                 np.zeros((9, 256), np.float32)], [np.zeros(64, np.float32), np.zeros(256, np.float32),
                                                                   np.zeros(9, np.float32)], 3, 0)


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.join(ROOT, "aberration-aware-depth-from-focus_b200")
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                with open(os.path.join(dirpath, f)) as fh:
                    text = fh.read()
                assert "oracle" not in text.replace("no oracle", ""), os.path.join(dirpath, f)


def test_python_surface_mirrors_reference(pkg):
    from deeplens.psfnet import PSFNet, ThinLens, DMIN, DMAX
    from deeplens.psfnet_arch import MLP
    from dff.factory import get_lens
    lens = PSFNet(filename="./lenses/rf50mm/lens.json", model_name="mlp", kernel_size=11, sensor_res=(480, 640),
                  device="cpu")
    assert (lens.d_min, lens.d_max, lens.kernel_size, lens.device) == (-DMIN, -DMAX, 11, "cpu")
    assert isinstance(lens.psfnet, MLP) and sum(p.numel() for p in lens.psfnet.parameters()) == 574393
    sd = torch.load(CKPT, map_location="cpu")
    assert list(lens.psfnet.state_dict().keys()) == list(sd.keys())
    lens.load_net(CKPT)
    assert torch.equal(lens.psfnet.state_dict()["net.20.bias"], sd["net.20.bias"])
    d = torch.tensor([0.0, -200.0, -10100.0, -20000.0, -30000.0])
    assert torch.allclose(lens.depth2z(d), torch.tensor([0.0, 0.0, 0.5, 1.0, 1.0]))
    assert torch.allclose(lens.z2depth(lens.depth2z(d[1:4])), d[1:4])
    lens.analysis()
    with pytest.raises(NotImplementedError):
        PSFNet(model_name="siren", device="cpu")
    args = {"ks": 11, "res": (480, 640), "device": "cpu",
            "train": {"lens": "./lenses/rf50mm/lens.json", "psfnet_path": CKPT},
            "test": {"lens": "thinlens", "foc_len": 50.0, "fnum": 1.8, "sensor_size": ["36", "24"]}}
    train_lens, test_lens = get_lens(args)
    assert isinstance(train_lens, PSFNet) and isinstance(test_lens, ThinLens)
    assert abs(test_lens.ps - 36.0 / 480) < 1e-12
    coc = test_lens.coc(torch.tensor([-1000.0, -2000.0]), torch.tensor([-2000.0, -2000.0]))
    assert coc[1] == pytest.approx(0.1) and coc[0] > 1.0


def test_select_focus_dist_matches_reference_golden():
    from dff.utils import select_focus_dist
    g = load_golden("kat_f_select_focus.npz")
    d = torch.from_numpy(g["depth_m"])
    assert torch.equal(select_focus_dist(d, 5), torch.from_numpy(g["out"]))
    assert torch.equal(select_focus_dist(d, 8), torch.from_numpy(g["out8"]))
    with pytest.raises(AssertionError):
        select_focus_dist(d, 3)


def test_econ_weight_calibration_host_side(pkg):
    """csrc/econ_calib.h (econ mode's output-error-calibrated fp16 rounding) against a numpy restatement of the same
    recurrence: results are fp16 values, agree with the restatement almost everywhere (a near-tie may round the other
    way), and shrink the layer's output error several-fold compared with plain rounding.  Host code only: no GPU."""
    import ctypes
    rng = np.random.default_rng(0)
    N, K, NC = 48, 64, 512
    M = rng.standard_normal((6, K))

    def acts(n):                                        # correlated, ReLU-like, like a hidden layer fed from 4 inputs
        return np.maximum(rng.standard_normal((n, 6)) @ M + 0.02 * rng.standard_normal((n, K)), 0)
    A = acts(NC).astype(np.float32)
    W = (rng.standard_normal((N, K)) * 0.1).astype(np.float32)
    out = np.zeros_like(W)
    rc = pkg.native.lib.aadff_debug_econ_round(ctypes.c_void_p(W.ctypes.data), N, K, ctypes.c_void_p(A.ctypes.data), NC,
                                               ctypes.c_void_p(out.ctypes.data))
    assert rc == 0
    assert np.array_equal(out, out.astype(np.float16).astype(np.float32))

    def f16(x):
        return x.astype(np.float16).astype(np.float64)
    A64, W64 = A.astype(np.float64), W.astype(np.float64)
    H = A64.T @ A64 / NC
    H += 1e-6 * np.mean(np.diag(H)) * np.eye(K)
    U = np.linalg.cholesky(np.linalg.inv(H)).T
    Wc, Q = W64.copy(), np.zeros_like(W64)
    for k in range(K):
        Q[:, k] = f16(Wc[:, k])
        err = (Wc[:, k] - Q[:, k]) / U[k, k]
        Wc[:, k + 1:] -= np.outer(err, U[k, k + 1:])
    assert np.mean(out == Q) > 0.98
    At = acts(4096)                                     # fresh samples of the same distribution
    e_plain = np.linalg.norm(At @ (W64 - f16(W64)).T)
    e_cal = np.linalg.norm(At @ (W64 - out).T)
    assert e_cal < 0.6 * e_plain, (e_cal, e_plain)
    assert pkg.native.lib.aadff_debug_econ_round(None, N, K, None, NC, None) != 0


def test_product_synthetic_generators_match_the_oracle_copies(pkg):
    """bench.py's GPU arm draws its inputs from aadff_b200.synthetic, the CPU arms and the tests from the oracle's own
    copy: both must give identical tensors (same workload on both arms, no oracle import in the product)."""
    from aadff_b200 import synthetic
    from oracle import focal_stack_oracle as orc
    for (N, H, W, seed) in [(1, 48, 64, 1234), (2, 40, 56, 1251)]:
        a, b = synthetic.synthetic_rgbd(N, H, W, seed), orc.synthetic_rgbd(N, H, W, seed)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        for S in (1, 2, 5, 10):
            assert torch.equal(synthetic.synthetic_focus(a[1], S), orc.synthetic_focus(b[1], S))
    for ks in (11, 31):
        (Wa, ba), (Wb, bb) = synthetic.seeded_psfnet_weights(ks, 0), orc.seeded_psfnet_weights(ks, 0)
        assert all(torch.equal(x, y) for x, y in zip(Wa, Wb)) and all(torch.equal(x, y) for x, y in zip(ba, bb))
    sd = torch.load(os.path.join(GOLDEN, "rf50mm_PSFNet480x640_ks11.pkl"), map_location="cpu")
    (Wa, ba), (Wb, bb) = synthetic.split_state_dict(sd), orc.split_state_dict(sd)
    assert all(torch.equal(x, y) for x, y in zip(Wa, Wb)) and all(torch.equal(x, y) for x, y in zip(ba, bb))


def test_tile_row_partition_is_exact_and_balanced(pkg):
    """Every tile row is dealt exactly once, shares differ by at most one tile row, and no rank idles even when there
    are fewer (image, slice) items than ranks (c2: 5 items, c4: 10 items on 8 GPUs -- VERDICT r01 item 3)."""
    sh = pkg.sharding
    assert sh.TILE_ROW_H == pkg.native.lib.aadff_tile_row_height()
    for N, S, H in [(16, 5, 256), (1, 10, 1080), (1, 5, 512), (3, 7, 37), (1, 1, 8), (2, 3, 5)]:
        ty = sh.tile_rows_per_slice(H)
        for world in (1, 2, 4, 8):
            sizes, rows = [], []
            for r in range(world):
                R0, R1 = sh.tile_row_range(N, S, H, world, r)
                sizes.append(R1 - R0)
                for (n, s, h0, h1) in sh.local_runs(N, S, H, world, r):
                    assert 0 <= h0 < h1 <= H and h0 % sh.TILE_ROW_H == 0
                    rows += [(n, s, h) for h in range(h0, h1)]
                assert sh.flat_row(R1, H) - sh.flat_row(R0, H) == sum(h1 - h0 for (_, _, h0, h1) in sh.local_runs(N, S, H, world, r))
            assert rows == [(n, s, h) for n in range(N) for s in range(S) for h in range(H)]
            assert sum(sizes) == N * S * ty and max(sizes) - min(sizes) <= 1
            if N * S * ty >= world:
                assert min(sizes) >= 1
    # the BASELINE shapes on 8 GPUs: c4 and c2 are balanced to within one tile row (was 2,2,1,1,1,1,1,1 items / 3 idle GPUs)
    assert [sh.tile_row_range(1, 10, 1080, 8, r)[1] - sh.tile_row_range(1, 10, 1080, 8, r)[0] for r in range(8)] == [169, 169, 169, 169, 169, 169, 168, 168]
    assert {sh.tile_row_range(1, 5, 512, 8, r)[1] - sh.tile_row_range(1, 5, 512, 8, r)[0] for r in range(8)} == {40}


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
import aadff_b200
sh = aadff_b200.sharding
rank, world = int(sys.argv[1]), int(sys.argv[2])
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT={port!r}, RANK=str(rank), WORLD_SIZE=str(world))
dist.init_process_group("gloo", rank=rank, world_size=world)

class FakeLens:          # stands in for PSFNet.render_stack / render_stack_rows: deterministic, per pixel, CPU
    def render_stack(self, img, depth, foc):
        return img[:, :, None] * foc[:, None, :, None, None] + depth[:, :, None]
    def render_stack_rows(self, img, depth, foc, R0, R1):
        N, C, H, W = img.shape
        S = foc.shape[1]
        rows = self.render_stack(img, depth, foc).permute(0, 2, 3, 1, 4).reshape(N * S * H, C, W)
        return rows[sh.flat_row(R0, H):sh.flat_row(R1, H)].clone()

g = torch.Generator().manual_seed(0)
for (N, C, S, H, W) in [(3, 2, 7, 4, 5), (1, 3, 5, 37, 6), (2, 1, 1, 16, 3)]:      # H < 8, ragged H, H = 2 tile rows
    img, depth, foc = torch.rand(N, C, H, W, generator=g), torch.rand(N, 1, H, W, generator=g), torch.rand(N, S, generator=g)
    full, (R0, R1) = sh.render_stack_sharded(FakeLens(), img, depth, foc, rank, world)
    ref = FakeLens().render_stack(img, depth, foc)
    assert full.shape == ref.shape and torch.equal(full, ref), "gathered stack differs"
    local, _ = sh.render_stack_sharded(FakeLens(), img, depth, foc, rank, world, gather=False)
    assert local.shape[0] == sh.flat_row(R1, H) - sh.flat_row(R0, H)
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_sharded_render_gathers_to_single_rank_result_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=str(29500 + os.getpid() % 2000)))
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2"], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_bench_dump_outputs_whole_or_seeded_sample(tmp_path):
    """bench.py --dump-outputs: a stack within the budget is written whole, a larger one as the same seeded sample of
    values + flat indices on every run, all files together within the budget."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    out = torch.rand(2, 3, 5, 40, 56, generator=torch.Generator().manual_seed(1))
    bench.dump_output(out, str(tmp_path / "whole"), "render_stack", bench.DUMP_BYTES)
    whole = np.load(tmp_path / "whole" / "render_stack.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, out.numpy())
    budget = 40000
    for run in ("a", "b"):
        bench.dump_output(out, str(tmp_path / run), "render_stack", budget)
        assert sum(f.stat().st_size for f in (tmp_path / run).iterdir()) <= budget
    vals, idx = np.load(tmp_path / "a" / "render_stack.npy"), np.load(tmp_path / "a" / "render_stack_index.npy")
    assert vals.dtype == np.float32 and idx.dtype == np.float64 and len(vals) == len(idx) > 1000
    assert np.array_equal(vals, out.numpy().reshape(-1)[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "render_stack_index.npy"))


def test_bench_reference_arm_prints_contract_line():
    """`bench.py --impl reference` (the CPU arm) must emit one JSON line with the contract keys."""
    import json
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    line = json.loads(res.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "cpu_baseline", "e2e", "config"):
        assert key in line
    assert line["impl"] == "reference" and line["value"] > 0
    # the unmodified reference (baseline/_ref, baseline/make_ref.py) when present, else the oracle's port of it
    have_ref = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "deeplens", "psfnet.py"))
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    # both arms of bench.py must print the same metric string, or the driver cannot form the ratio (VERDICT r01)
    import re
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert len(re.findall(r'"metric":\s*METRIC', src)) >= 3 and src.count('"metric": "') == 0
    # ... and the reference arm must not load the product library
    res = subprocess.run([sys.executable, "-c", "import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', "
                          "'--workload', 'c1', '--steps', '1', '--warmup', '0']; runpy.run_path(%r, run_name='__main__'); "
                          "maps = open('/proc/self/maps').read(); assert 'libaadff' not in maps, 'reference arm mapped libaadff.so'; "
                          "assert 'aadff_native' not in sys.modules" % os.path.join(ROOT, "bench.py")],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
