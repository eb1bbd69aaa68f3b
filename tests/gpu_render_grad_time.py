"""Timing of the differentiable focal-stack render (render_stack(differentiable=True)) against the hand-built eager
chain lens.psfnet(probes) -> local_psf_render -> backward().  Not a pytest file.

    python tests/gpu_render_grad_time.py [out.json]        (default out: profiles/r08_render_grad_time.json)

Workloads: c2 (5 images x 3 x 512^2, 1 slice each, k = 11, rf50mm), 1 x 3 x 480 x 640 with S = 5 (k = 11, rf50mm) and
1 x 3 x 1080 x 1920 with S = 1 (k = 31, seeded network).  For each, CUDA events over REPS runs after warm-up:
  - forward alone (no grad);
  - forward + backward with only the image requiring grad;
  - forward + backward with every gradient (image, depth, focus distances, weights, biases);
  - peak device memory of the all-gradient step;
and the same through the hand-built chain in mode fp32 (the chain's PSFs come from the fp32 MLP).  Every time is given as
median, min and max.  The image and upstream gradient of every workload fit the 126 MB L2 (31 / 22 / 50 MB), so they
are read from there after the first pass; the hand chain's stored PSF tensors (1.2 GB to 8 GB) do not.  Per workload also
the workspace that
aadff_render_stack_backward_work_bytes returns, and the device time per kernel of one image-only backward in parity mode
(torch.profiler, the forward outside the profiled window).  The card's name and power limit are read in the same run."""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402
from oracle import focal_stack_oracle as orc  # noqa: E402
from oracle import train_oracle as tor  # noqa: E402

CKPT = os.path.join(ROOT, "tests", "golden", "rf50mm_PSFNet480x640_ks11.pkl")
REPS = 10


def timed(fn, reps=REPS):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return {"median": statistics.median(ts), "min": min(ts), "max": max(ts), "reps": reps}


def kernel_times(lens, img, depth, foc, G):
    """Device time per kernel (ms, summed over launches) of one image-only backward."""
    x = img.clone().requires_grad_(True)
    for p in lens.psfnet.parameters():
        p.requires_grad_(False)
    out = lens.render_stack(x, depth, foc, differentiable=True)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out.backward(G)
        torch.cuda.synchronize()
    res = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            res[e.key[:90]] = t / 1e3
    return dict(sorted(res.items(), key=lambda kv: -kv[1]))


def peak(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def lens_for(ks, mode):
    lens = aadff_b200.PSFNet(kernel_size=ks, device="cuda", mode=mode)
    if ks == 11:
        lens.load_net(CKPT)
    else:
        gen = torch.Generator().manual_seed(0)
        Ws, bs = tor.kaiming_net([4, 64, 256] + [256] * 8 + [ks * ks], gen, bias_scale=0.1)
        with torch.no_grad():
            for lin, W, b in zip(lens.psfnet.linear_layers(), Ws, bs):
                lin.weight.copy_(torch.as_tensor(W))
                lin.bias.copy_(torch.as_tensor(b))
    return lens


def workload(N, S, H, W):
    img, depth_m = orc.synthetic_rgbd(N, H, W, seed=1)
    foc_m = orc.synthetic_focus(depth_m, S)
    return img.cuda(), (-depth_m * 1e3).cuda(), (-foc_m * 1e3).cuda()


def step_ours(lens, img, depth, foc, G, full):
    x = img.clone().requires_grad_(True)
    d = depth.clone().requires_grad_(full)
    f = foc.clone().requires_grad_(full)
    for p in lens.psfnet.parameters():
        p.requires_grad_(full)
        p.grad = None
    lens.render_stack(x, d, f, differentiable=True).backward(G)


def step_hand(lens, img, depth, foc, G, full):
    N, C, H, W = img.shape
    ks = lens.kernel_size
    x = img.clone().requires_grad_(True)
    d = depth.clone().requires_grad_(full)
    f = foc.clone().requires_grad_(full)
    for p in lens.psfnet.parameters():
        p.requires_grad_(full)
        p.grad = None
    xs = torch.from_numpy(orc.linspace_f32(-1.0, 1.0, W)).cuda().view(1, 1, W).expand(N, H, W)
    ys = torch.from_numpy(orc.linspace_f32(1.0, -1.0, H)).cuda().view(1, H, 1).expand(N, H, W)
    z = torch.clamp((d[:, 0] - lens.d_min) / (lens.d_max - lens.d_min), 0, 1)
    outs = []
    for s in range(foc.shape[1]):
        fz = torch.clamp((f[:, s] - lens.d_min) / (lens.d_max - lens.d_min), 0, 1).view(N, 1, 1).expand(N, H, W)
        psf = lens.psfnet(torch.stack((xs, ys, z, fz), -1))
        outs.append(aadff_b200.local_psf_render(x, psf.view(N, H, W, ks, ks), ks))
    torch.stack(outs, 2).backward(G)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r08_render_grad_time.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "rows": []}
    for name, (N, S, H, W, ks) in {"c2_5x3x512x512_k11": (5, 1, 512, 512, 11),
                                   "1x3x480x640_S5_k11": (1, 5, 480, 640, 11),
                                   "1x3x1080x1920_S1_k31": (1, 1, 1080, 1920, 31)}.items():
        img, depth, foc = workload(N, S, H, W)
        G = torch.randn(N, 3, S, H, W, device="cuda")
        row = {"workload": name}
        for mode in ("parity", "fp32"):
            lens = lens_for(ks, mode)
            with torch.no_grad():
                row[f"{mode}_forward_ms"] = timed(lambda: lens.render_stack(img, depth, foc))
            row[f"{mode}_fwd_bwd_img_ms"] = timed(lambda: step_ours(lens, img, depth, foc, G, False))
            row[f"{mode}_fwd_bwd_all_ms"] = timed(lambda: step_ours(lens, img, depth, foc, G, True), reps=5)
            row[f"{mode}_peak_all_mib"] = peak(lambda: step_ours(lens, img, depth, foc, G, True))
            if mode == "parity":
                row["work_bytes"] = int(aadff_b200.native.lib.aadff_render_stack_backward_work_bytes(
                    lens.native().handle, H, W))
                row["parity_bwd_img_kernels_ms"] = kernel_times(lens, img, depth, foc, G)
        lens = lens_for(ks, "fp32")
        row["hand_fwd_bwd_img_ms"] = timed(lambda: step_hand(lens, img, depth, foc, G, False), reps=5)
        row["hand_fwd_bwd_all_ms"] = timed(lambda: step_hand(lens, img, depth, foc, G, True), reps=5)
        row["hand_peak_all_mib"] = peak(lambda: step_hand(lens, img, depth, foc, G, True))
        print(json.dumps(row), flush=True)
        res["rows"].append(row)
        del lens
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
