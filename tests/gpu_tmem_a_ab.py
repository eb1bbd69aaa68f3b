"""A/B timing of the fused render kernel: A operands in tensor memory (default) against the shared-memory-operand path
(debug flag 1 << 20), alternated in one process.  Not a pytest file.

    python tests/gpu_tmem_a_ab.py [out.txt] [--rounds R]     (default out: profiles/r03_tmem_a_ab.txt)

Every timed launch follows a 256 MB write that evicts L2 (the inputs are re-read from HBM, as in a training loop), and
each leg starts after a short idle so that neither path inherits the other's clock state.  Reports per-workload
medians of the per-launch device time (CUDA events) and the ratio new / old, plus whether the outputs are identical."""
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402
from oracle import focal_stack_oracle as orc  # noqa: E402

SMEM_A = 1 << 20
WORKLOADS = [("c1", 1, 1, 480, 640), ("c2", 1, 5, 512, 512), ("c3", 16, 5, 256, 256), ("c5b16", 16, 5, 512, 512)]
LAUNCHES = 10          # timed launches per leg


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_path = args[0] if args else os.path.join(ROOT, "profiles", "r03_tmem_a_ab.txt")
    rounds = int(sys.argv[sys.argv.index("--rounds") + 1]) if "--rounds" in sys.argv else 5
    nat = aadff_b200.native
    lens = aadff_b200.PSFNet(kernel_size=11, device="cuda")
    lens.load_net(os.path.join(ROOT, "tests/golden/rf50mm_PSFNet480x640_ks11.pkl"))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    lines = []
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines.append(f"# GPU (name, power limit, max SM clock, SM clock at start): {smi}")
    lines.append(f"# {rounds} rounds x {LAUNCHES} launches per leg, L2 flushed before every launch; median ms per launch")
    lines.append("# workload mode       tmem-A ms   smem-A ms   smem/tmem  identical")
    for mode in ("econ8", "parity"):
        for (name, N, S, H, W) in WORKLOADS:
            img, dm = orc.synthetic_rgbd(N, H, W, seed=1234)
            foc = (-orc.synthetic_focus(dm, S) * 1e3).cuda()
            img, dep = img.cuda(), -dm.cuda() * 1e3
            out = torch.empty(N, 3, S, H, W, device="cuda")
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(LAUNCHES)]

            def leg(flags):
                nat.lib.aadff_debug_set_flags(flags)
                try:
                    r = lens.render_stack(img, dep, foc, mode=mode)          # warm-up (and the output to compare)
                    torch.cuda.synchronize()
                    time.sleep(0.2)
                    for e0, e1 in ev:
                        flush.zero_()
                        e0.record()
                        lens.render_stack(img, dep, foc, mode=mode)
                        e1.record()
                    torch.cuda.synchronize()
                finally:
                    nat.lib.aadff_debug_set_flags(0)
                return [e0.elapsed_time(e1) for e0, e1 in ev], r

            t_new, t_old = [], []
            same = True
            for rd in range(rounds):
                order = (0, SMEM_A) if rd % 2 == 0 else (SMEM_A, 0)
                for flags in order:
                    ts, r = leg(flags)
                    (t_new if flags == 0 else t_old).extend(ts)
                    if flags == 0:
                        out.copy_(r)
                    else:
                        same &= bool(torch.equal(out, r))
            mn, mo = statistics.median(t_new), statistics.median(t_old)
            line = f"  {name:7s}  {mode:8s}  {mn:9.4f}   {mo:9.4f}   {mo / mn:8.3f}   {same}"
            print(line, flush=True)
            lines.append(line)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
