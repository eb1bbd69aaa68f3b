"""Timing of the differentiable PSFNet MLP (lens.psfnet under autograd) against eager PyTorch autograd.  Not a pytest file.

    python tests/gpu_psfnet_grad_time.py [out.json]        (default out: profiles/r07_psfnet_grad_time.json)

With the rf50mm network at M = 128, 16 384 and 307 200 probes (CUDA events, median of REPS after warm-up; the
activations of the larger sizes exceed L2 on their own):
  - forward alone (lens.psfnet(x) without grad: mlp_fp32_kernel);
  - forward + backward for every gradient (probes and parameters);
  - the backward alone (aadff_psfnet_backward_f32 through the C ABI), with its FLOPs from the shapes: the recompute
    (the forward's 2 M sum K N) plus dA and dW (2 M sum K N each; the first layer has no dA but a dX);
  - the same nn.Sequential under eager torch autograd in fp32, TF32 off.
Then the wall time per step of a 128-probe torch.optim.AdamW loop through lens.psfnet, which rebuilds the packed handle
after every update (a device->host copy of the weights and a new upload), beside train_psfnet's native step.
The card's name and power limit are read in the same run."""
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402
from oracle import focal_stack_oracle as orc  # noqa: E402

CKPT = os.path.join(ROOT, "tests", "golden", "rf50mm_PSFNet480x640_ks11.pkl")
REPS = 10


def timed(fn, reps=REPS):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_psfnet_grad_time.json")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    lens = aadff_b200.PSFNet(kernel_size=11, device="cuda")
    lens.load_net(CKPT)
    Ws, bs = orc.split_state_dict(torch.load(CKPT, map_location="cpu"))
    dims = [4] + [w.shape[0] for w in Ws]
    mods = []
    for l, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        mods += [nn.Linear(a, b), nn.ReLU(inplace=True) if l < len(Ws) - 1 else nn.Sigmoid()]
    seq = nn.Sequential(*mods).cuda()
    with torch.no_grad():
        for lin, W, b in zip([m for m in seq if isinstance(m, nn.Linear)], Ws, bs):
            lin.weight.copy_(W)
            lin.bias.copy_(b)
    lib, nat = aadff_b200.native.lib, lens.native()
    params = list(lens.psfnet.parameters())
    res = {"gpu": smi, "network": "rf50mm, 11 layers, ks 11", "sizes": {}}
    flops_fwd_per_probe = 2 * sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    for M in (128, 16384, 307200):
        x = torch.rand(M, 4, device="cuda")
        g = torch.randn(M, 121, device="cuda")
        xg = x.clone().requires_grad_(True)

        def fwd():
            with torch.no_grad():
                lens.psfnet(x)

        def fwd_bwd():
            torch.autograd.grad(lens.psfnet(xg), params + [xg], g)

        def eager():
            p = seq(xg)
            p = p / p.abs().sum(-1, keepdim=True).clamp_min(1e-12)
            torch.autograd.grad(p, list(seq.parameters()) + [xg], g)

        gw = [torch.empty_like(p) for p in params]
        gx = torch.empty_like(x)
        c_f32p = aadff_b200.native.ctypes.POINTER(aadff_b200.native.ctypes.c_float)
        cast = lambda t: aadff_b200.native.ctypes.cast(aadff_b200.native.ctypes.c_void_p(t.data_ptr()), c_f32p)
        wp = (c_f32p * len(Ws))(*[cast(t) for t in gw[0::2]])
        bp = (c_f32p * len(Ws))(*[cast(t) for t in gw[1::2]])
        wb = lib.aadff_psfnet_backward_work_bytes(nat.handle, M)
        work = torch.empty(wb, dtype=torch.uint8, device="cuda")

        def bwd():
            aadff_b200.native.check(lib.aadff_psfnet_backward_f32(
                nat.handle, x.data_ptr(), g.data_ptr(), gx.data_ptr(), wp, bp, work.data_ptr(), wb, M,
                torch.cuda.current_stream().cuda_stream))

        t_f, t_fb, t_b, t_e = timed(fwd), timed(fwd_bwd), timed(bwd), timed(eager)
        flops_b = 3 * M * flops_fwd_per_probe      # recompute + dA (dX for layer 0) + dW
        res["sizes"][str(M)] = {"forward_ms": t_f, "forward_backward_ms": t_fb, "backward_ms": t_b,
                                "eager_autograd_fp32_forward_backward_ms": t_e, "backward_flops": flops_b,
                                "backward_tflops": flops_b / (t_b * 1e-3) / 1e12, "workspace_bytes": int(wb)}
        print(M, res["sizes"][str(M)], flush=True)

    # 128-probe AdamW loop through lens.psfnet (each update rebuilds the packed handle)
    opt = torch.optim.AdamW(lens.psfnet.parameters(), lr=1e-6)
    x = torch.rand(128, 4, device="cuda")
    t = torch.rand(128, 121, device="cuda")
    t = t / t.sum(1, keepdim=True)

    def step():
        opt.zero_grad()
        nn.MSELoss()(lens.psfnet(x), t).backward()
        opt.step()

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    n = 100
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    torch.cuda.synchronize()
    res["adamw_loop_128_ms_per_step"] = (time.perf_counter() - t0) / n * 1e3
    t0 = time.perf_counter()
    for _ in range(n):
        lens.refresh()
        lens.native()
    torch.cuda.synchronize()
    res["handle_rebuild_ms"] = (time.perf_counter() - t0) / n * 1e3
    # train_psfnet's native step at the same batch
    Wc = [l.weight.detach().cpu().numpy() for l in lens.psfnet.linear_layers()]
    bc = [l.bias.detach().cpu().numpy() for l in lens.psfnet.linear_layers()]
    tr = aadff_b200.native.NativeTrainer(Wc, bc, 128, 0)
    st = torch.cuda.current_stream().cuda_stream

    def native_step():
        lib.aadff_trainer_step(tr.handle, x.data_ptr(), t.data_ptr(), 1e-6, None, st)

    for _ in range(5):
        native_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        native_step()
    torch.cuda.synchronize()
    res["train_psfnet_native_step_ms"] = (time.perf_counter() - t0) / n * 1e3
    tr.close()
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
