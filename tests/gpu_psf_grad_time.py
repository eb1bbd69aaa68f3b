"""Timing of the local_psf_render / render_psf_map backward kernels against their forwards.  Not a pytest file.

    python tests/gpu_psf_grad_time.py [out.txt]        (default out: profiles/r04_psf_grad_time.txt)

local_psf_render: the forward, dimg and dP launches through the C ABI, each timed alone (CUDA events, median of
LAUNCHES, a 256 MB write evicting L2 before every launch), with algorithmic bytes over time as a fraction of the HBM
data-sheet peak (7.7 TB/s).  Every one of the three moves N H W (4 ks^2 + 8 C) bytes: the PSF tensor (or its gradient)
once, the image and grad_out once.  Then the same backward through eager torch autograd of the reference's unfold
formulation (deeplens/render_psf.py:76-107), where it fits in memory.  render_psf_map: forward and full backward
(dimg + both dK stages) time at 1x3x1080x1920."""
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402

HBM_PEAK = 7.7e12
LAUNCHES = 15
LOCAL = [("c1", 1, 3, 480, 640, 11), ("b16", 16, 3, 512, 512, 11), ("b16", 16, 3, 512, 512, 15),
         ("4k", 1, 3, 1080, 1920, 31)]


def timed(fn, flush, n=LAUNCHES):
    ts = []
    for _ in range(n + 2):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts[2:])


def ref_unfold(img, psf, ks):
    """deeplens/render_psf.py:76-107: replicate pad + unfold + multiply + sum."""
    N, C, H, W = img.shape
    r = (ks - 1) // 2
    unf = F.unfold(F.pad(img, (r, r, r, r), mode="replicate"), ks).view(N, C, ks * ks, H * W)
    return (unf * psf.reshape(N, 1, H * W, ks * ks).transpose(2, 3)).sum(2).view(N, C, H, W)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04_psf_grad_time.txt")
    lib = aadff_b200.native.lib
    check = aadff_b200.native.check
    from deeplens.render_psf import render_psf_map
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    st = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    lines = []
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    lines.append(f"# GPU (name, power limit, max SM clock): {smi}")
    lines.append(f"# median of {LAUNCHES} launches, L2 flushed before each; frac = algorithmic bytes / time / 7.7 TB/s")
    lines.append("# local_psf_render       ks   fwd ms (frac)    dimg ms (frac)   dP ms (frac)     fwd+bwd/fwd"
                 "   eager autograd bwd ms   eager/ours bwd")
    for name, N, C, H, W, ks in LOCAL:
        torch.manual_seed(0)
        img = torch.rand(N, C, H, W, device="cuda")
        psf = torch.rand(N, H, W, ks, ks, device="cuda")
        g = torch.randn(N, C, H, W, device="cuda")
        out, gi, gp = torch.empty_like(img), torch.empty_like(img), torch.empty_like(psf)
        fwd = lambda: check(lib.aadff_local_psf_render_f32(img.data_ptr(), psf.data_ptr(), out.data_ptr(),  # noqa: E731
                                                           N, C, H, W, ks, st()))
        bimg = lambda: check(lib.aadff_local_psf_render_backward_f32(  # noqa: E731
            img.data_ptr(), psf.data_ptr(), g.data_ptr(), gi.data_ptr(), None, N, C, H, W, ks, st()))
        bpsf = lambda: check(lib.aadff_local_psf_render_backward_f32(  # noqa: E731
            img.data_ptr(), psf.data_ptr(), g.data_ptr(), None, gp.data_ptr(), N, C, H, W, ks, st()))
        nbytes = N * H * W * (4 * ks * ks + 8 * C)
        t = [timed(f, flush) for f in (fwd, bimg, bpsf)]
        frac = [nbytes / (x * 1e-3) / HBM_PEAK for x in t]
        eager = "n/a"
        ratio = ""
        try:
            a, b = img.clone().requires_grad_(True), psf.clone().requires_grad_(True)

            def eager_bwd():
                a.grad = b.grad = None
                o = ref_unfold(a, b, ks)
                o.backward(g)

            def eager_fwd():
                with torch.no_grad():
                    ref_unfold(a, b, ks)
            te = timed(eager_bwd, flush, 5) - timed(eager_fwd, flush, 5)
            eager = f"{te:.3f}"
            ratio = f"{te / (t[1] + t[2]):.2f}x"
            del a, b
        except torch.cuda.OutOfMemoryError:
            eager = "out of memory"
        torch.cuda.empty_cache()
        lines.append(f"{name:>4} {N}x{C}x{H}x{W:<6} {ks:>4}   {t[0]:7.3f} ({frac[0]:.2f})  {t[1]:7.3f} ({frac[1]:.2f})"
                     f"  {t[2]:7.3f} ({frac[2]:.2f})   {(t[0] + t[1] + t[2]) / t[0]:5.2f}        {eager:>10}"
                     f"       {ratio}")
        print(lines[-1], flush=True)
        del img, psf, g, out, gi, gp
        torch.cuda.empty_cache()

    lines.append("# render_psf_map 1x3x1080x1920   grid  ks   fwd ms    bwd ms (dimg + dK)")
    for grid in (1, 8):
        for ks in (11, 31):
            torch.manual_seed(0)
            img = torch.rand(1, 3, 1080, 1920, device="cuda", requires_grad=True)
            pm = torch.rand(3, grid * ks, grid * ks, device="cuda", requires_grad=True)
            g = torch.randn(1, 3, 1080, 1920, device="cuda")

            def f_fwd():
                with torch.no_grad():
                    render_psf_map(img, pm, grid)

            def f_all():
                img.grad = pm.grad = None
                render_psf_map(img, pm, grid).backward(g)
            tf = timed(f_fwd, flush)
            tb = timed(f_all, flush) - tf
            lines.append(f"{'':31} {grid:>4} {ks:>3}  {tf:7.3f}  {tb:8.3f}")
            print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
