#!/usr/bin/env python
"""Benchmark of the fused PSFNet + PSF-render focal-stack synthesis path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c2|c3|c4|c1|c5b8..c5b64] [--mode parity|econ8|econ|fast|mixed|fp32] [--c5]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic RGB-D: the whole focal stack
[N,3,S,H,W] of the workload, in ONE kernel launch.  Metric: Mpix*slices/s = N*S*H*W / t / 1e6
(SURVEY.md section 8d).  Default workload c2 = BASELINE.json configs[1]: 5-slice focal stack at
512x512, rf50mm checkpoint, k = 11.  Default mode econ8 = the fastest arithmetic whose worst case over ANY [0,1] image is
certified under north_star's 1e-4 (three fp16 hi/lo MMA terms for L1-L7, two for L8, L9 and the head; DESIGN.md section 5);
`other_modes` carries parity (three terms everywhere, the library's default), econ, mixed and fast.

Under torchrun (N > 1) the headline `value` is weak scaling -- every rank renders its own stack of
the workload's shape, no data-path collective, time = max over ranks -- and the same line carries
`strong`: BASELINE configs 2 and 3 (c3, c4) rendered ONCE across all ranks through
sharding.render_stack_sharded (tile-row partition), checked bit-for-bit against the single-GPU stack.

`--impl reference` runs the UNMODIFIED reference (baseline/_ref, see baseline/make_ref.py) through its own
public API, PSFNet.render, on the host CPU: same metric, workload and inputs; nothing of this repo's
product is imported by that arm.  Prints ONE JSON line (rank 0).

`--dump-outputs DIR` writes the focal stack of the last timed step as DIR/render_stack.npy (float32, [N,3,S,H,W]) so
that two builds run with the same arguments (hence the same seeded inputs) can be compared element for element.  A
stack larger than 64 MB is replaced by a fixed, seeded sample of its elements: render_stack.npy holds the values and
render_stack_index.npy (float64) their flat indices.  Under torchrun every rank writes render_stack_rank<r>*.npy of
its own stack within 64 MB / ranks.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "focal-stack Mpix*slices/s (fused PSFNet+PSF render)"     # the same string on both arms
UNIT = "Mpix*slices/s"
WORKLOADS = {  # name: (N, S, H, W, ks, description)
    "c1": (1, 1, 480, 640, 11, "0_warm_up.py: one 480x640 slice, rf50mm ckpt, k=11"),
    "c2": (1, 5, 512, 512, 11, "AiFNet config: 5-slice focal stack at 512x512, rf50mm ckpt, k=11"),
    "c3": (16, 5, 256, 256, 11, "DFVNet config: batch 16 x 5 slices at 256x256, rf50mm ckpt, k=11"),
    "c4": (1, 10, 1080, 1920, 31, "large render: 10 slices at 1920x1080, k=31, seeded random PSFNet"),
    # BASELINE configs[4] (AiF training step, batch sweep): these time the focal-stack simulation of one training
    # batch; the whole step (simulation + AiFNet forward/backward/Adam) is measured by --c5 (key `c5_training_step`)
    "c5b8": (8, 5, 512, 512, 11, "AiF training batch: 8 x 5 slices at 512x512 (simulation half of the step), k=11"),
    "c5b16": (16, 5, 512, 512, 11, "AiF training batch: 16 x 5 slices at 512x512 (simulation half of the step), k=11"),
    "c5b32": (32, 5, 512, 512, 11, "AiF training batch: 32 x 5 slices at 512x512 (simulation half of the step), k=11"),
    "c5b64": (64, 5, 512, 512, 11, "AiF training batch: 64 x 5 slices at 512x512 (simulation half of the step), k=11"),
}
CKPT = os.path.join(ROOT, "tests", "golden", "rf50mm_PSFNet480x640_ks11.pkl")
DTYPES = {"parity": "f32 via fp16 hi/lo split (3 tcgen05 terms, f32 accumulate)",
          "mixed": "fp16 split for 3 layers then single fp16 term (f32 accumulate)",
          "econ": "fp16 hi/lo split, 3 terms (early layers) / 2 terms on calibrated fp16 weights (late layers, head), f32 accumulate",
          "econ8": "fp16 hi/lo split, 3 terms for L1-L7, 2 terms on calibrated fp16 weights for L8, L9 and the head (worst case over any image 7.5e-5), f32 accumulate",
          "fast": "f16 operands, f32 accumulate", "fp32": "f32"}


# what the parity tests hold each mode to (tests/test_gpu_parity.py) and its worst case over any [0,1] image on the
# shipped checkpoint (half the L1 distance between the mode's PSFs and the fp32 PSFs over 2^20 probes, profiles/r02b_cert_econ8.txt)
MODE_ACCURACY = {
    "parity": "max-abs vs the reference's goldens 1.1e-5 (c2) / 9.1e-6 (c3) / 1.3e-6 (c4), tested at 2e-5; worst case over any image 5.6e-5; bar 1e-4",
    "econ8": "max-abs vs the reference's goldens 2.1e-5 (c2) / 2.6e-5 (c3) / 1.7e-6 (c4), tested at 4e-5; worst case over any image 7.5e-5 "
             "(asserted < 1e-4 in test_econ8_mode_certified_between_parity_and_econ); bar 1e-4",
    "econ": "max-abs vs the reference's goldens 3.1e-5 / 3.4e-5 / 2.2e-6, tested at 6e-5; worst case over a hand-built image 2.0e-4 (not certified)",
    "mixed": "2.2e-4 on the goldens (reduced precision)", "fast": "6e-3 max / 6e-5 mean on the goldens (reduced precision)",
    "fp32": "1.3e-6 on the goldens (CUDA cores, operation-exact)"}


DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs: all files of all ranks together


def dump_output(out, path, name, budget):
    """out -> path/<name>.npy (float32).  Over `budget` bytes: a sample of elements at seeded random flat indices
    (sorted, repeats possible), written with those indices as path/<name>_index.npy (float64, exact below 2^53)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = out.detach()
    room = budget - 4096                                   # .npy headers
    if out.numel() * 4 > room:
        idx = torch.randint(out.numel(), (room // (4 + 8),), generator=torch.Generator().manual_seed(0)).sort().values
        np.save(os.path.join(path, f"{name}_index.npy"), idx.double().numpy())
        out = out.reshape(-1)[idx.to(out.device)]
    np.save(os.path.join(path, f"{name}.npy"), out.float().cpu().numpy())


def flops_per_pixel(ks):
    return 2 * (4 * 64 + 64 * 256 + 8 * 256 * 256 + 256 * ks * ks)


def load_peaks():
    """(burst bf16 TFLOP/s, sustained bf16 TFLOP/s, HBM GB/s, source)"""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]), float(p.get("bf16_tflops_sustained", 0.0)), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1590.0, 1400.0, 6650.0, "fallback"


def mma_terms(mode, n_groups=10):
    """fp16 MMA terms per tensor-core group L1..L9 + head (layer 0 runs on CUDA cores)."""
    import aadff_b200
    first = aadff_b200.native.econ_first_group()
    return {"parity": [3] * 10, "fast": [1] * 10, "mixed": [3, 3, 3] + [1] * 7,
            "econ": [3] * first + [2] * (10 - first), "econ8": [3] * 7 + [2] * 3, "fp32": [0] * 10}[mode]


def executed_mma_flops_per_pixel(ks, mode):
    """MMA FLOPs the kernel really issues per pixel*slice: layers L1..L10 on tensor cores, head padded to a
    multiple of 16 columns, times the number of fp16 terms per layer, plus one K=16 bias-slab MMA per hidden layer."""
    head = (ks * ks + 15) // 16 * 16
    per_layer = [64 * 256] + [256 * 256] * 8 + [256 * head]
    terms = mma_terms(mode)
    bias_slabs = 0 if mode == "fp32" else 9 * 16 * 256
    return 2 * (sum(t * m for t, m in zip(terms, per_layer)) + bias_slabs), \
        sum(t * m for t, m in zip(terms, per_layer)) / sum(per_layer)


def ncu_traffic(workload, mode):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the fused kernel, from the committed
    `ncu --set full` captures (profiles/ncu_traffic.json, written by tests/gpu_ncu_summary.py); None if that
    workload/mode was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        e = t.get(f"{workload}/{mode}")
        return (e["bytes"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------------------ inputs
def _generators(product):
    """Seeded synthetic RGB-D / focus / weight generators.  The product arm uses the product package's copy, the
    reference arm the checker's copy (tests/test_host_cpu.py asserts that both give identical tensors), so that
    the reference arm imports nothing of the product."""
    if product:
        from aadff_b200 import synthetic as g
    else:
        from oracle import focal_stack_oracle as g
    return g


def weights_for(ks, product=True):
    g = _generators(product)
    if ks == 11:
        return g.split_state_dict(torch.load(CKPT, map_location="cpu"))
    return g.seeded_psfnet_weights(ks, seed=0)


def state_dict_for(ks, product=True):
    Ws, bs = weights_for(ks, product)
    sd = {}
    for l, (Wl, bl) in enumerate(zip(Ws, bs)):
        sd[f"net.{2 * l}.weight"], sd[f"net.{2 * l}.bias"] = Wl, bl
    return sd


def make_inputs(name, rank, product=True):
    g = _generators(product)
    N, S, H, W, ks, _ = WORKLOADS[name]
    img, depth_m = g.synthetic_rgbd(N, H, W, seed=1234 + 17 * rank)
    foc_m = g.synthetic_focus(depth_m, S)
    return img, -depth_m * 1e3, -foc_m * 1e3


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(rows)}


# ------------------------------------------------------------------------------------------------ reference arm
def reference_sample(name):
    """The bounded sample of the workload one reference step renders: ONE slice of ONE image (the reference has no
    cross-slice or cross-image reuse, 2_aber_aware_dff_aif.py:108-114, so per-slice cost is the whole cost); for
    k = 31 the frame is cropped to 270x480 (the reference's unfold of a full 1080p frame needs 3 x 24 GB)."""
    N, S, H, W, ks, _ = WORKLOADS[name]
    img, depth, foc = make_inputs(name, 0, product=False)
    hh, ww = (270, 480) if ks > 15 else (H, W)
    return (img[:1, :, :hh, :ww].contiguous(), depth[:1, :, :hh, :ww].contiguous(), foc[:1, 0].contiguous(), hh, ww)


def reference_renderer(name, device):
    """-> (render(img, depth, foc) callable, kind).  kind "reference": the unmodified reference's PSFNet.render from
    baseline/_ref; "port": the oracle's restatement of its operator sequence (only if baseline/_ref is absent)."""
    N, S, H, W, ks, _ = WORKLOADS[name]
    from baseline import ref_import
    if ref_import.available():
        # (PSFNet.render never reads sensor_res; the ray-traced constructor asserts the lens aspect ratio, so 1080p is not accepted)
        lens = ref_import.make_lens(ks, (H, W) if H * 4 == W * 3 or H == W else (480, 640), device, state_dict_for(ks, product=False))
        return (lambda img, depth, foc: lens.render(img, depth, foc)), "reference"
    from oracle import focal_stack_oracle as orc
    Ws, bs = weights_for(ks, product=False)
    Ws, bs = [w.to(device) for w in Ws], [b.to(device) for b in bs]
    return (lambda img, depth, foc: orc.render_reference_ops(Ws, bs, img, depth, foc, ks)), "port"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, S, H, W, ks, desc = WORKLOADS[args.workload]
    if args.ref_device == "cuda":
        return run_reference_eager_gpu(args)
    torch.set_num_threads(os.cpu_count() or 1)
    render, kind = reference_renderer(args.workload, "cpu")
    img, depth, foc, hh, ww = reference_sample(args.workload)
    what = "the unmodified reference's PSFNet.render (baseline/_ref)" if kind == "reference" else "oracle port of the reference's operator sequence"
    sample = f"each step = 1 slice of 1 image, {hh}x{ww}, k={ks}, {what}, fp32, host CPU"
    with torch.no_grad():
        for _ in range(args.warmup):
            render(img, depth, foc)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            render(img, depth, foc)
        dt = time.perf_counter() - t0
    value = hh * ww * args.steps / dt / 1e6
    cores = torch.get_num_threads()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}", "device": "host CPU", "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def run_reference_eager_gpu(args):
    """The "before" number: the reference's own eager-PyTorch path on this B200 (fp32, TF32 off), slice loop +
    torch.stack exactly as 2_aber_aware_dff_aif.py:108-114.  Spawned by the product arm as a subprocess."""
    if args.c5:
        return c5_training_step_reference(args)
    N, S, H, W, ks, desc = WORKLOADS[args.workload]
    torch.backends.cuda.matmul.allow_tf32 = False
    render, kind = reference_renderer(args.workload, "cuda")
    img, depth, foc = (t.cuda() for t in make_inputs(args.workload, 0, product=False))

    def step():
        return torch.stack([render(img, depth, foc[:, i]) for i in range(S)], dim=2)
    with torch.no_grad():
        for _ in range(max(1, args.warmup)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"impl": "reference", "device": "cuda", "kind": kind, "metric": METRIC, "unit": UNIT,
                      "value": N * S * H * W / (ms * 1e-3) / 1e6, "ms_per_step": ms, "steps": args.steps,
                      "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30, "checksum": float(out.double().sum())}))


def c5_training_step_reference(args):
    """BASELINE config 5 the way the reference does it (2_aber_aware_dff_aif.py:93-126): select_focus_dist + eager
    PSFNet.render slice loop + torch.stack + empty_cache, then AiFDepthNet forward/backward/Adam -- all reference
    code from baseline/_ref, on the GPU.  One JSON line: per batch size step / simulation time."""
    import importlib.util
    from baseline import ref_import
    torch.backends.cuda.matmul.allow_tf32 = False
    S, H, W = 5, 512, 512
    dev = torch.device("cuda")
    lens = ref_import.make_lens(11, (H, W), "cuda", state_dict_for(11, product=False))
    AiF = ref_import.load_aifnet()
    spec = importlib.util.spec_from_file_location("ref_dff_utils", os.path.join(ref_import.REF_ROOT, "dff", "utils.py"))
    dff_utils = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(dff_utils)
    out = {}
    for B in [int(b) for b in args.c5.split(",")]:
        try:
            torch.manual_seed(0)
            net = AiF.AiFDepthNet(n_stack=S).to(dev)
            net.train()
            opt = torch.optim.Adam(net.parameters(), lr=1e-4)
            aif_args = {"device": dev, "task": "D_FS", "stack_num": S}
            aif, depth = _generators(False).synthetic_rgbd(B, H, W, seed=99)
            aif, depth = aif.to(dev), depth.to(dev)

            def step():
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                with torch.no_grad():
                    focus_dists = dff_utils.select_focus_dist(depth, S, mode="linear")
                    focal_stack = []
                    for i in range(S):
                        focal_stack.append(lens.render(aif, depth=-depth * 1e3, foc_dist=-focus_dists[:, i] * 1e3))
                    focal_stack = torch.stack(focal_stack, dim=2)
                torch.cuda.empty_cache()
                e[1].record()
                losses, _ = net({"stack_rgb_img": focal_stack, "focus_position": focus_dists, "depth": depth, "AiF_img": aif}, aif_args)
                opt.zero_grad()
                losses["total"].mean().backward()
                opt.step()
                e[2].record()
                return e
            step()
            torch.cuda.synchronize()
            evs = [step() for _ in range(2)]
            torch.cuda.synchronize()
            sim = statistics.mean(a.elapsed_time(b) for a, b, _ in evs)
            tot = statistics.mean(a.elapsed_time(c) for a, _, c in evs)
            out[f"B{B}"] = {"step_ms": tot, "simulation_ms": sim, "simulation_share": sim / tot,
                            "simulation_Mpix_slices_per_s": B * S * H * W / (sim * 1e-3) / 1e6,
                            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
            del net, opt
        except torch.cuda.OutOfMemoryError:
            out[f"B{B}"] = {"error": "CUDA out of memory (reference eager path)"}
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
    print(json.dumps({"impl": "reference", "device": "cuda", "c5_training_step": out}))


def spawn_reference(workload, steps, warmup, device="cpu", timeout=600, c5=""):
    """Run `bench.py --impl reference` in a child process (the reference's `deeplens` and the product's shadow
    `deeplens` cannot live in one interpreter) and return its JSON line, or {"error": ...}."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload,
           "--steps", str(steps), "--warmup", str(warmup), "--ref-device", device] + (["--c5", c5] if c5 else [])
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        return json.loads(res.stdout.strip().splitlines()[-1])
    except Exception as e:            # noqa: BLE001 -- a missing baseline must not lose the product's own line
        return {"error": f"{type(e).__name__}: {e}"[:300]}


# ------------------------------------------------------------------------------------------------ product arm
def make_lens(aadff_b200, ks, H, W, local, mode):
    lens = aadff_b200.PSFNet(kernel_size=ks, sensor_res=(H, W), device=f"cuda:{local}", mode=mode)
    lens.psfnet.load_state_dict(state_dict_for(ks))
    return lens


def strong_scaling(aadff_b200, dist, name, mode, local, rank, world, steps, flush):
    """One stack of BASELINE config `name` rendered once across all ranks: tile-row partition, one launch per rank,
    no collective in the timed region; afterwards the shares are all-gathered and compared bit for bit with the
    stack every rank renders alone."""
    N, S, H, W, ks, desc = WORKLOADS[name]
    lens = make_lens(aadff_b200, ks, H, W, local, mode)
    img, dep, foc = (t.cuda() for t in make_inputs(name, 0))          # the same stack on every rank
    sh = aadff_b200.sharding

    def timed(fn):
        for _ in range(2):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        evs = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs) / steps], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)
    ms_single = timed(lambda: lens.render_stack(img, dep, foc, mode=mode))        # every GPU alone (max over ranks)
    ms_sharded = timed(lambda: sh.render_stack_sharded(lens, img, dep, foc, rank, world, gather=False, mode=mode))
    full, (R0, R1) = sh.render_stack_sharded(lens, img, dep, foc, rank, world, gather=True, mode=mode)
    equal = torch.tensor([int(torch.equal(full, lens.render_stack(img, dep, foc, mode=mode)))], device="cuda")
    dist.all_reduce(equal, op=dist.ReduceOp.MIN)
    units = N * S * H * W
    return {"workload": f"{name}: {desc}", "value": units / (ms_sharded * 1e-3) / 1e6, "unit": UNIT,
            "ms_per_stack": ms_sharded, "single_gpu_value": units / (ms_single * 1e-3) / 1e6,
            "single_gpu_ms": ms_single, "speedup": ms_single / ms_sharded, "eff": ms_single / ms_sharded / world,
            "bit_equal_to_single_gpu": bool(int(equal)), "steps": steps,
            "partition": f"{N * S * sh.tile_rows_per_slice(H)} tile rows (8 image rows each) in {world} contiguous runs, "
                         f"one launch per rank; rank 0 renders tile rows [{R0},{R1})"}


def c5_training_step(aadff_b200, lens, batches, n_steps=3):
    """BASELINE config 5: one training step of 2_aber_aware_dff_aif.py:93-126 -- focal-stack simulation feeding the
    reference's AiFDepthNet (dff/AiFNet.py, used as is from baseline/_ref), forward + backward + Adam -- with the
    simulation done by PSFNet.simulate_focal_stack (select_focus + ONE fused launch)."""
    from baseline import ref_import
    if not ref_import.available():
        return {"unavailable": "baseline/_ref missing"}
    AiF = ref_import.load_aifnet()
    S, H, W = 5, 512, 512
    out = {}
    dev = torch.device("cuda")
    for B in batches:
        try:
            torch.manual_seed(0)
            net = AiF.AiFDepthNet(n_stack=S).to(dev)
            net.train()
            opt = torch.optim.Adam(net.parameters(), lr=1e-4)
            aif_args = {"device": dev, "task": "D_FS", "stack_num": S}
            img, depth_m = _generators(True).synthetic_rgbd(B, H, W, seed=99)
            img, depth_m = img.to(dev), depth_m.to(dev)

            def step():
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                stack, focus = lens.simulate_focal_stack(img, depth_m, S)
                e[1].record()
                losses, _ = net({"stack_rgb_img": stack, "focus_position": focus, "depth": depth_m, "AiF_img": img}, aif_args)
                opt.zero_grad()
                losses["total"].mean().backward()
                opt.step()
                e[2].record()
                return e
            step()
            torch.cuda.synchronize()
            evs = [step() for _ in range(n_steps)]
            torch.cuda.synchronize()
            sim = statistics.mean(a.elapsed_time(b) for a, b, _ in evs)
            tot = statistics.mean(a.elapsed_time(c) for a, _, c in evs)
            out[f"B{B}"] = {"step_ms": tot, "simulation_ms": sim, "simulation_share": sim / tot,
                            "simulation_Mpix_slices_per_s": B * S * H * W / (sim * 1e-3) / 1e6,
                            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
            del net, opt
            torch.cuda.empty_cache()
        except torch.cuda.OutOfMemoryError:
            out[f"B{B}"] = {"error": "CUDA out of memory in AiFDepthNet forward/backward"}
            torch.cuda.empty_cache()
    return out


def secondary_kernels(aadff_b200, flush, peak_hbm):
    """The HBM-bound kernels of the path's neighbours, one line each (median of 7 launches, L2 flushed before each):
    local_psf_render alone on a PSF tensor in HBM (algorithmic bytes = 4 k^2 + 24 per pixel at C = 3) and the fused
    thin-lens render (28 B per pixel: far from HBM-bound, reported in Gpix/s)."""
    import torch
    ThinLens = aadff_b200.ThinLens

    def median_ms(fn):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(7):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    res = {}
    g = torch.Generator(device="cuda").manual_seed(11)
    for ks, n in ((11, 16), (31, 4)):
        img = torch.rand(n, 3, 512, 512, device="cuda", generator=g)
        psf = torch.rand(n, 512, 512, ks, ks, device="cuda", generator=g)
        ms = median_ms(lambda: aadff_b200.local_psf_render(img, psf, ks))
        gbs = n * 512 * 512 * (4 * ks * ks + 24) / ms / 1e6
        res[f"local_psf_render_k{ks}"] = {
            "shape": [n, 3, 512, 512], "ms": ms, "Gpix_per_s": n * 512 * 512 / ms / 1e6,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm},
            "kernel": "local_psf_strip_kernel" if ks <= 15 else "local_psf_coalesced_kernel"}
        del img, psf
    tl = ThinLens(foc_len=50.0, fnum=1.8, kernel_size=11, sensor_size=[36.0, 24.0], sensor_res=(512, 512)).to("cuda")
    img = torch.rand(16, 3, 512, 512, device="cuda", generator=g)
    dep = -(300 + 5000 * torch.rand(16, 1, 512, 512, device="cuda", generator=g))
    foc = -(500 + 3000 * torch.rand(16, device="cuda", generator=g))
    ms = median_ms(lambda: tl.render(img, dep, foc))
    res["thinlens_render_k11"] = {"shape": [16, 3, 512, 512], "ms": ms, "Gpix_per_s": 16 * 512 * 512 / ms / 1e6,
                                  "T_taps_per_s": 16 * 512 * 512 * 121 / ms / 1e9, "bound": "issue (FFMA + LDS per tap)",
                                  "kernel": "thinlens_render2_kernel"}
    return res


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    import aadff_b200
    nat = aadff_b200.native

    N, S, H, W, ks, desc = WORKLOADS[args.workload]
    lens = make_lens(aadff_b200, ks, H, W, local, args.mode)
    img_h, dep_h, foc_h = make_inputs(args.workload, rank)
    img, dep, foc = img_h.cuda(), dep_h.cuda(), foc_h.cuda()
    units = N * S * H * W                               # pixel*slices per step per rank
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value"): CUDA events around every step, L2 flushed between
    def timed(mode, steps, warmup):
        for _ in range(warmup):
            out = lens.render_stack(img, dep, foc, mode=mode)
        barrier()
        evs = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = lens.render_stack(img, dep, foc, mode=mode)
            e1.record()
            evs.append((e0, e1))
        barrier()
        return [a.elapsed_time(b) for a, b in evs], out

    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = nat.lib.aadff_launch_count()
    t_wall0 = time.perf_counter()
    times, out = timed(args.mode, args.steps, args.warmup)
    t_wall1 = time.perf_counter()
    launches = nat.lib.aadff_launch_count() - launches0 - args.warmup
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs:
        dump_output(out, args.dump_outputs, "render_stack" if world == 1 else f"render_stack_rank{rank}",
                    DUMP_BYTES // world)
    total_ms = torch.tensor([sum(times)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)
    value = units * world * args.steps / (total_ms * 1e-3) / 1e6

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D + kernel + D2H per step
    img_p, dep_p, foc_p = img_h.contiguous().pin_memory(), dep_h.reshape(N, H, W).contiguous().pin_memory(), \
        foc_h.contiguous().pin_memory()
    out_p = torch.empty(N, 3, S, H, W).pin_memory()
    h = lens.native().handle

    def host_call():
        nat.check(nat.lib.aadff_render_stack_host_f32(h, img_p.data_ptr(), dep_p.data_ptr(), foc_p.data_ptr(),
                                                      out_p.data_ptr(), N, 3, S, H, W, float(lens.d_min),
                                                      float(lens.d_max), nat.MODES[args.mode]))
    for _ in range(max(1, args.warmup)):
        host_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_call()
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = units * world * args.steps / float(e2e_s) / 1e6
    same = float((out_p.cuda() - out).abs().max())

    # ---- verification gather (outside every timed region)
    checksum = out.double().sum().reshape(1)
    if world > 1:
        sums = [torch.zeros_like(checksum) for _ in range(world)]
        dist.all_gather(sums, checksum)
        checksum = torch.stack(sums).sum().reshape(1)

    # ---- strong scaling of the sharded BASELINE configs (torchrun only)
    strong = {}
    if world > 1 and not args.no_strong:
        for name in ("c3", "c4"):
            strong[name] = strong_scaling(aadff_b200, dist, name, args.mode, local, rank, world, max(5, args.steps // 2), flush)

    extra = {}
    if rank == 0 and world == 1 and not args.no_extra:
        for mode in [m for m in ("parity", "econ8", "econ", "fast", "mixed") if m != args.mode]:
            tt, _ = timed(mode, max(3, args.steps // 2), 2)
            extra[mode] = {"value": units / (statistics.mean(tt) * 1e-3) / 1e6, "unit": UNIT, "dtype": DTYPES[mode]}
    secondary = {}
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            secondary = secondary_kernels(aadff_b200, flush, load_peaks()[2])
        except Exception as e:                                   # never lose the headline line over a side measurement
            secondary = {"error": repr(e)}

    if rank == 0:
        peak_tf, peak_tf_sus, peak_hbm, peak_src = load_peaks()
        ms_kernel = statistics.mean(times)
        achieved = flops_per_pixel(ks) * units / (ms_kernel * 1e-3) / 1e12
        exec_flops, avg_terms = executed_mma_flops_per_pixel(ks, args.mode)
        executed = exec_flops * units / (ms_kernel * 1e-3) / 1e12
        traffic, traffic_src = ncu_traffic(args.workload, args.mode)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPES[args.mode],
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "mode": args.mode, "mode_accuracy": MODE_ACCURACY.get(args.mode), "per_gpu_shape": [N, 3, S, H, W],
                       "kernel_size": ks, "l2": "flushed (256 MiB fill) before every timed step",
                       "parallelism": f"replicated PSFNet, {world} independent stack(s), no collective on the path"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": (img_p.numel() + dep_p.numel() + foc_p.numel()) * 4,
                    "d2h_bytes_per_step": out_p.numel() * 4, "api": "aadff_render_stack_host_f32 (pinned host buffers)",
                    "launches_per_step": S, "launch_shape": "one launch per focal slice (the D2H copy of slice s "
                    "overlaps the kernel of slice s+1); `value` times one launch for the whole stack",
                    "max_abs_vs_device_path": same},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": f"{peak_src} bf16 burst",
                         "executed_mma_tflops": executed, "executed_frac_of_burst_peak": executed / peak_tf,
                         "executed_frac_of_sustained_peak": (executed / peak_tf_sus) if peak_tf_sus else None,
                         "avg_executed_terms": avg_terms, "frac_of_terms_ceiling": achieved / peak_tf * avg_terms if avg_terms else None,
                         "algorithmic_bytes_per_launch": int(units * (12 + 16 / S)),
                         "kernel": "fused_psfnet_render_kernel", "kernel_ms": ms_kernel,
                         "algorithmic_flops_per_pixel_slice": flops_per_pixel(ks),
                         "executed_mma_terms_per_group": mma_terms(args.mode)},
            "checksum": float(checksum),
        }
        if strong:
            line["strong"] = strong
        if extra:
            line["other_modes"] = extra
        if secondary:
            line["secondary_kernels"] = secondary
        if world == 1 and not args.no_cpu:
            del flush
            torch.cuda.empty_cache()
            # the "before" number on the same GPU: the reference's eager path (child process, baseline/_ref)
            if not args.no_eager and args.workload in ("c1", "c2", "c3"):
                r = spawn_reference(args.workload, 3, 1, device="cuda")
                line["gpu_eager_baseline"] = r if "error" in r else {
                    "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "kind": r["kind"],
                    "peak_mem_gb": r["peak_mem_gb"], "what": "reference PSFNet.render slice loop + torch.stack, eager "
                    "PyTorch fp32 (TF32 off) on the same GPU, device-resident inputs"}
            # the reference's CPU path on this box's host cores (child process)
            r = spawn_reference(args.workload, max(2, int(args.cpu_seconds // 2)), 1, device="cpu")
            line["cpu_baseline"] = r["cpu_baseline"] if "cpu_baseline" in r else {"error": r.get("error", "no line")}
        if world == 1 and args.c5:
            ours = c5_training_step(aadff_b200, make_lens(aadff_b200, 11, 512, 512, local, args.mode),
                                    [int(b) for b in args.c5.split(",")])
            torch.cuda.empty_cache()
            ref = spawn_reference("c2", 1, 0, device="cuda", timeout=1500, c5=args.c5)
            line["c5_training_step"] = {
                "what": "2_aber_aware_dff_aif.py:93-126 at 5 x 512 x 512 per image: focal-stack simulation + the reference's "
                        "AiFDepthNet (random init) forward/backward/Adam; `reference` = all reference code, eager, same GPU",
                "ours": ours, "reference": ref.get("c5_training_step", ref)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="econ8", choices=["parity", "econ8", "econ", "fast", "mixed", "fp32"],
                    help="econ8 (default) = the fastest mode whose worst case over ANY [0,1] image is certified under the 1e-4 bar; "
                         "parity = three MMA terms everywhere (the library's default)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-eager", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--c5", default="", help="comma-separated batch sizes of the end-to-end AiF training step, e.g. 8,16,32,64")
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"], help="reference arm only (cuda = eager baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the focal stack of the last timed step to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
