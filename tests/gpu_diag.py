"""GPU bring-up diagnostics (not a pytest file): each stage runs in its own subprocess under a
hard timeout so that a hung kernel cannot take the whole box-call with it.

    python tests/gpu_diag.py [stage ...]        # default: all stages, log to gpurun_out/diag.log
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def stage_umma():
    import numpy as np
    import ctypes
    import aadff_b200
    nat = aadff_b200.native
    rng = np.random.default_rng(0)
    for K, N in [(32, 16), (64, 256), (256, 256), (256, 128), (256, 208)]:
        A = rng.standard_normal((128, K)).astype(np.float32)
        B = rng.standard_normal((N, K)).astype(np.float32)
        D = np.zeros((128, N), np.float32)
        rc = nat.lib.aadff_debug_umma_gemm(A.ctypes.data, B.ctypes.data, D.ctypes.data, K, N, 0)
        if rc:
            print(f"K={K} N={N}: rc={rc} {nat.lib.aadff_last_error().decode()}")
            continue
        ref = A.astype(np.float16).astype(np.float32) @ B.astype(np.float16).astype(np.float32).T
        err = np.abs(D - ref).max()
        print(f"K={K} N={N}: max|D-ref|={err:.3e}  (|ref|max={np.abs(ref).max():.2f})", flush=True)


def _lens(ks=11, mode="parity"):
    import torch
    import aadff_b200
    lens = aadff_b200.PSFNet(kernel_size=ks, device="cuda", mode=mode)
    if ks == 11:
        lens.load_net(os.path.join(ROOT, "tests/golden/rf50mm_PSFNet480x640_ks11.pkl"))
    return lens


def _check(name, out, ref):
    d = (out.cpu() - ref).abs()
    print(f"{name}: max-abs {float(d.max()):.3e}  mean-abs {float(d.mean()):.3e}", flush=True)


def stage_fp32():
    import numpy as np
    import torch
    from conftest import analytic_rgbd, load_golden
    lens = _lens(mode="fp32")
    g = load_golden("kat_a_pred.npz")
    _check("pred kat_a", lens.pred(torch.from_numpy(g["inp"]).cuda()), torch.from_numpy(g["psf"]))
    for N, H, W in [(1, 48, 64), (2, 64, 64)]:
        g = load_golden(f"kat_b_{N}x{H}x{W}.npz")
        img, dm = analytic_rgbd(N, H, W)
        out = lens.render(img.cuda(), -dm.cuda() * 1e3, torch.from_numpy(g["foc"]).cuda())
        _check(f"fp32 render kat_b {N}x{H}x{W}", out, torch.from_numpy(g["out"]))
    g = load_golden("kat_d_gather_0.npz")
    import aadff_b200
    out = aadff_b200.local_psf_render(torch.from_numpy(g["img"]).cuda(), torch.from_numpy(g["psf"]).cuda(), int(g["ks"]))
    _check("gather kat_d_0", out, torch.from_numpy(g["out"]))


def _tc(mode):
    import torch
    from conftest import analytic_rgbd, load_golden
    lens = _lens(mode=mode)
    for N, H, W in [(1, 48, 64), (2, 64, 64)]:
        g = load_golden(f"kat_b_{N}x{H}x{W}.npz")
        img, dm = analytic_rgbd(N, H, W)
        out = lens.render(img.cuda(), -dm.cuda() * 1e3, torch.from_numpy(g["foc"]).cuda())
        torch.cuda.synchronize()
        _check(f"{mode} render kat_b {N}x{H}x{W}", out, torch.from_numpy(g["out"]))
    g = load_golden("kat_e_stack_2x40x56.npz")
    out = lens.render_stack(torch.from_numpy(g["img"]).cuda(), -torch.from_numpy(g["depth_m"]).cuda() * 1e3,
                            -torch.from_numpy(g["foc_m"]).cuda() * 1e3)
    _check(f"{mode} stack kat_e", out, torch.from_numpy(g["out"]))


def stage_tc_parity():
    _tc("parity")


def stage_tc_fast():
    _tc("fast")
    _tc("mixed")
    _tc("econ")


def stage_econ():
    """econ mode with the calibrated fp16 weights vs plain rounding (debug flag 256), incl. a noise image at c2 size
    against the fp32 CUDA-core kernel."""
    import torch
    import aadff_b200
    from oracle import focal_stack_oracle as orc
    for flags in (0, 256):
        aadff_b200.native.lib.aadff_debug_set_flags(flags)
        print(f"--- econ, debug flags {flags} ({'plain fp16 rounding' if flags else 'calibrated rounding'})")
        _tc("econ")
        lens = _lens(mode="econ")
        gen = torch.Generator().manual_seed(5)
        img = torch.rand(1, 3, 512, 512, generator=gen).cuda()
        _, dm = orc.synthetic_rgbd(1, 512, 512, seed=77)
        dep = -dm.cuda() * 1e3
        foc = -orc.synthetic_focus(dm, 5).cuda() * 1e3
        out = lens.render_stack(img, dep, foc, mode="econ")
        ref = lens.render_stack(img, dep, foc, mode="fp32")
        par = lens.render_stack(img, dep, foc, mode="parity")
        print(f"noise image 5x512x512: econ vs fp32 max {float((out - ref).abs().max()):.3e} mean "
              f"{float((out - ref).abs().mean()):.3e}; parity vs fp32 max {float((par - ref).abs().max()):.3e}", flush=True)
    aadff_b200.native.lib.aadff_debug_set_flags(0)


def stage_eager_gpu():
    """The "before" number of SURVEY.md section 8d: the reference's operator sequence (11 x linear, replicate pad,
    unfold, C-fold PSF copy, multiply, sum -- deeplens/psfnet.py:424-441 + render_psf.py:96-107) as eager PyTorch on
    the same B200, fp32 with TF32 off, one slice per call like the reference's scripts."""
    import torch
    import torch.nn.functional as F
    from oracle import focal_stack_oracle as orc
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "rf50mm_PSFNet480x640_ks11.pkl"), map_location="cpu")
    Ws, bs = orc.split_state_dict(sd)
    Ws, bs = [w.cuda() for w in Ws], [b.cuda() for b in bs]
    ks = 11

    def render_eager(img, depth, foc):
        N, C, H, W = img.shape
        x, y = torch.meshgrid(torch.linspace(-1, 1, W, device="cuda"), torch.linspace(1, -1, H, device="cuda"), indexing="xy")
        z = ((depth.reshape(N, H, W) + 200.0) / (-19800.0)).clamp(0, 1)
        fz = ((foc.view(N, 1, 1) + 200.0) / (-19800.0)).clamp(0, 1).expand(N, H, W)
        h = torch.stack((x.expand(N, H, W), y.expand(N, H, W), z, fz), -1)
        for l, (Wl, bl) in enumerate(zip(Ws, bs)):
            h = F.linear(h, Wl, bl)
            h = torch.relu_(h) if l < len(Ws) - 1 else torch.sigmoid(h)
        psf = F.normalize(h, p=1, dim=-1)
        pad = F.pad(img, (5, 5, 5, 5), mode="replicate")
        cols = F.unfold(pad, (ks, ks)).view(N, C, ks * ks, H * W)
        taps = torch.stack(C * [psf.reshape(-1, ks, ks)], 1).view(N, H * W, C, ks * ks).permute(0, 2, 3, 1)
        return (cols * taps).sum(2).view(N, C, H, W)

    for name, (N, S, H, W) in (("c1", (1, 1, 480, 640)), ("c2", (1, 5, 512, 512)), ("c3", (16, 5, 256, 256))):
        img, dm = orc.synthetic_rgbd(N, H, W, seed=1234)
        foc = -orc.synthetic_focus(dm, max(S, 2)).cuda() * 1e3
        img, dep = img.cuda(), -dm.cuda() * 1e3
        lens = _lens(mode="parity")
        with torch.no_grad():
            ref0 = render_eager(img, dep, foc[:, 0].contiguous())
            ours0 = lens.render(img, dep, foc[:, 0].contiguous())
            err = float((ref0 - ours0).abs().max())
            for _ in range(2):
                for s in range(S):
                    render_eager(img, dep, foc[:, s].contiguous())
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            iters = 5
            e0.record()
            for _ in range(iters):
                out = torch.stack([render_eager(img, dep, foc[:, s].contiguous()) for s in range(S)], dim=2)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        print(f"eager PyTorch on B200, {name} {N}x{S}x{H}x{W} k11: {ms:.2f} ms per stack  "
              f"{N * S * H * W / ms / 1e3:.1f} Mpix*slices/s; peak mem {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB; "
              f"|eager - ours(parity)| max {err:.2e}", flush=True)


def stage_tc_ks31():
    import torch
    from conftest import load_golden
    from oracle import focal_stack_oracle as orc
    g = load_golden("kat_g_ks31_1x40x48.npz")
    Ws, bs = orc.seeded_psfnet_weights(31, seed=int(g["weight_seed"]))
    gen = torch.Generator().manual_seed(int(g["bias_seed"]))
    bs = [(torch.rand(b.shape, generator=gen) - 0.5) * 0.2 for b in bs]
    for mode in ("fp32", "parity", "fast"):
        lens = _lens(ks=31, mode=mode)
        sd = {}
        for l, (W, b) in enumerate(zip(Ws, bs)):
            sd[f"net.{2 * l}.weight"], sd[f"net.{2 * l}.bias"] = W, b
        lens.psfnet.load_state_dict(sd)
        out = lens.render(torch.from_numpy(g["img"]).cuda(), -torch.from_numpy(g["depth_m"]).cuda() * 1e3,
                          torch.from_numpy(g["foc"]).cuda())
        torch.cuda.synchronize()
        _check(f"{mode} ks31 kat_g", out, torch.from_numpy(g["out"]))


def stage_speed():
    import torch
    from oracle import focal_stack_oracle as orc
    for (N, S, H, W, ks, modes) in [(1, 5, 512, 512, 11, ("parity", "econ", "mixed", "fast", "fp32")),
                                    (16, 5, 256, 256, 11, ("parity", "fast")),
                                    (1, 2, 1080, 1920, 31, ("parity", "fast"))]:
        img, dm = orc.synthetic_rgbd(N, H, W, seed=1234)
        foc = -orc.synthetic_focus(dm, S).cuda() * 1e3
        img, dep = img.cuda(), -dm.cuda() * 1e3
        for mode in modes:
            lens = _lens(ks=ks, mode=mode)
            for _ in range(2):
                out = lens.render_stack(img, dep, foc)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            iters = 3 if mode == "fp32" else 10
            e0.record()
            for _ in range(iters):
                out = lens.render_stack(img, dep, foc)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            print(f"speed N{N} S{S} {H}x{W} ks{ks} {mode}: {ms:.3f} ms  {N * S * H * W / ms / 1e3:.1f} Mpix*slices/s",
                  flush=True)


def stage_rows():
    """Throughput of the stand-alone rows: local_psf_render (HBM-bound on the PSF read) and pred."""
    import torch
    import aadff_b200
    def timeit(fn, iters=10):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    for (N, H, W, ks) in [(1, 480, 640, 11), (4, 512, 512, 11), (16, 512, 512, 11), (4, 512, 512, 7), (1, 540, 960, 31)]:
        img = torch.rand(N, 3, H, W, device="cuda")
        psf = torch.rand(N, H, W, ks, ks, device="cuda")
        for flags in (0,):
            aadff_b200.native.lib.aadff_debug_set_flags(flags)
            ms = timeit(lambda: aadff_b200.local_psf_render(img, psf, ks))
            px = N * H * W
            gb = px * (ks * ks * 4 + 24) / 1e9
            print(f"gather N{N} {H}x{W} k{ks} flags={flags}: {ms:.3f} ms  {px / ms / 1e3:.1f} Mpix/s  {gb / ms * 1e3:.0f} GB/s",
                  flush=True)
        aadff_b200.native.lib.aadff_debug_set_flags(0)
    from deeplens.psfnet import ThinLens
    for (N, H, W, ks) in [(4, 512, 512, 11), (1, 1080, 1920, 31)]:
        tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=ks, sensor_size=[36.0, 24.0], sensor_res=(H, W)).to("cuda")
        img = torch.rand(N, 3, H, W, device="cuda")
        dep = -(300 + 5000 * torch.rand(N, 1, H, W, device="cuda"))
        foc = -(500 + 3000 * torch.rand(N, device="cuda"))
        ms = timeit(lambda: tl.render(img, dep, foc))
        print(f"thinlens N{N} {H}x{W} k{ks}: {ms:.3f} ms  {N * H * W / ms / 1e3:.1f} Mpix/s", flush=True)
    lens = _lens(mode="parity")
    inp = torch.rand(1 << 20, 4, device="cuda")
    ms = timeit(lambda: lens.pred(inp), iters=3)
    print(f"pred M=1Mi k11 (fp32 kernel): {ms:.3f} ms  {inp.shape[0] / ms / 1e3:.1f} Mprobes/s", flush=True)
    for mode in ("parity", "fast"):
        ms = timeit(lambda: lens.pred(inp, mode=mode), iters=5)
        print(f"pred M=1Mi k11 (tensor-core, {mode}): {ms:.3f} ms  {inp.shape[0] / ms / 1e3:.1f} Mprobes/s", flush=True)


def stage_rows2():
    """Round-2 rows: thin-lens with its bytes-based roofline, render_psf / render_psf_map (FFMA-bound), and the
    PSFNet fitting step (CUDA graph) against the same step in eager PyTorch on this GPU."""
    import torch
    import torch.nn as nn
    import aadff_b200
    from deeplens.psfnet import ThinLens
    from deeplens.render_psf import render_psf, render_psf_map
    def timeit(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    hbm = 6531.6
    for (N, H, W, ks) in [(4, 512, 512, 11), (16, 512, 512, 11), (16, 512, 512, 7), (1, 1080, 1920, 31)]:
        tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=ks, sensor_size=[36.0, 24.0], sensor_res=(H, W)).to("cuda")
        img = torch.rand(N, 3, H, W, device="cuda")
        dep = -(300 + 5000 * torch.rand(N, 1, H, W, device="cuda"))
        foc = -(500 + 3000 * torch.rand(N, device="cuda"))
        ms = timeit(lambda: tl.render(img, dep, foc))
        aadff_b200.native.lib.aadff_debug_set_flags(16)
        ms_no_tma = timeit(lambda: tl.render(img, dep, foc))
        aadff_b200.native.lib.aadff_debug_set_flags(0)
        print(f"  (halo by cp.async only, no TMA: {ms_no_tma:.3f} ms)")
        px = N * H * W
        gbs = px * 28 / ms / 1e6
        print(f"thinlens N{N} {H}x{W} k{ks}: {ms:.3f} ms  {px / ms / 1e3:.1f} Mpix/s  algorithmic 28 B/px -> {gbs:.0f} GB/s = "
              f"{gbs / hbm:.3f} of measured HBM peak; {px * ks * ks * 4 / ms / 1e9:.2f} T taps/s (per tap: FMUL + ISETP/FSEL + FADD + 3 FFMA + 3 LDS; issue-bound)", flush=True)
    for (B, C, H, W, ks, grid) in [(4, 3, 512, 512, 11, 1), (4, 3, 512, 512, 11, 8), (1, 3, 1080, 1920, 31, 4)]:
        img = torch.rand(B, C, H, W, device="cuda")
        pm = torch.rand(C, grid * ks, grid * ks, device="cuda")
        fn = (lambda: render_psf(img, pm)) if grid == 1 else (lambda: render_psf_map(img, pm, grid))
        ms = timeit(fn)
        fma = B * C * H * W * ks * ks
        print(f"psf_conv B{B} {H}x{W} k{ks} grid{grid}: {ms:.3f} ms  {B * C * H * W / ms / 1e3:.1f} Mpix*ch/s  {fma / ms / 1e9:.2f} TFMA/s "
              f"(fp32 FFMA peak 148 SM x 128 x 1.9 GHz = 36 TFMA/s)", flush=True)
    bgr = torch.randint(0, 255, (8, 1024, 1280, 3), dtype=torch.uint8, device="cuda")
    d16 = torch.randint(0, 8000, (8, 1024, 1280), dtype=torch.int16, device="cuda").view(torch.uint16)
    ms = timeit(lambda: aadff_b200.preprocess_rgbd(bgr, d16, (480, 640)))
    gb = (bgr.numel() + d16.numel() * 2 + 8 * 4 * 480 * 640 * 4) / 1e9
    print(f"preprocess_rgbd 8 x 1024x1280 -> 480x640 (image + depth): {ms:.3f} ms  {8 / ms:.1f} images/ms  {gb / ms * 1e3:.0f} GB/s of "
          f"algorithmic traffic (5 B per input pixel + 16 B per output pixel)", flush=True)
    # fitting step: bs = 128 as in the reference (psfnet.py:79)
    ks, bs = 11, 128
    lens = aadff_b200.PSFNet(kernel_size=ks, device="cuda")
    lin = [m for m in lens.psfnet.net if isinstance(m, nn.Linear)]
    tr = aadff_b200.native.NativeTrainer([l.weight.detach().cpu().numpy() for l in lin], [l.bias.detach().cpu().numpy() for l in lin], bs, 0)
    inp = torch.rand(bs, 4, device="cuda")
    tgt = torch.rand(bs, ks * ks, device="cuda")
    tgt = tgt / tgt.sum(1, keepdim=True)
    ms = timeit(lambda: aadff_b200.native.check(aadff_b200.native.lib.aadff_trainer_step(tr.handle, inp.data_ptr(), tgt.data_ptr(), 1e-4, None,
                                                                                    torch.cuda.current_stream().cuda_stream)), iters=200)
    mods = []
    dims = [4, 64, 256] + [256] * 8 + [ks * ks]
    for a, b in zip(dims[:-2], dims[1:-1]):
        mods += [nn.Linear(a, b), nn.ReLU(inplace=True)]
    net = nn.Sequential(*mods, nn.Linear(dims[-2], dims[-1]), nn.Sigmoid()).cuda()
    opt = torch.optim.AdamW(net.parameters(), 1e-4)
    def eager():
        pred = torch.nn.functional.normalize(net(inp), p=1, dim=-1)
        opt.zero_grad()
        nn.MSELoss()(pred, tgt).backward()
        opt.step()
    ms_e = timeit(eager, iters=50)
    print(f"train step bs={bs} k{ks}: CUDA-graph trainer {ms * 1e3:.1f} us/step, eager PyTorch (reference operators, same GPU) "
          f"{ms_e * 1e3:.1f} us/step -> {ms_e / ms:.1f}x", flush=True)


STAGES = {k[6:]: v for k, v in list(globals().items()) if k.startswith("stage_")}

if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--run":
        STAGES[sys.argv[2]]()
        sys.exit(0)
    names = sys.argv[1:] or ["umma", "fp32", "tc_parity", "tc_fast", "tc_ks31", "speed", "rows", "econ"]
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    log = open(os.path.join(ROOT, "gpurun_out", "diag.log"), "a")
    for name in names:
        t0 = time.time()
        try:
            res = subprocess.run([sys.executable, os.path.abspath(__file__), "--run", name], capture_output=True,
                                 text=True, timeout=int(os.environ.get("DIAG_TIMEOUT", "150")))
            txt = f"=== {name} (rc={res.returncode}, {time.time() - t0:.1f}s)\n{res.stdout}{res.stderr[-3000:]}\n"
        except subprocess.TimeoutExpired as ex:
            txt = f"=== {name} TIMEOUT after {time.time() - t0:.1f}s\n{ex.stdout or ''}\n{ex.stderr or ''}\n"
        print(txt, flush=True)
        log.write(txt)
        log.flush()
