"""Timeline trace of CTA 0 of the fused kernel (debug aid, not a pytest file).

    python tests/gpu_trace.py [mode] [ks]      -> gpurun_out/trace_<mode>.txt
Prints, per role, (delta-cycles, event) for the second tile the CTA processes (steady state).
Event codes are defined next to TcTrace in csrc/fused_tc_kernel.cuh."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aadff_b200  # noqa: E402
from oracle import focal_stack_oracle as orc  # noqa: E402

NAMES = {0x1: "slab_issue g", 0x2: "mma_group_start g", 0x3: "mma_wait_A j", 0x4: "mma_got_A j", 0x5: "mma_wait_W kc",
         0x6: "mma_got_W kc", 0x7: "mma_group_issued g", 0x8: "tile_start", 0x9: "L0_done", 0xA: "epi_wait_acc g",
         0xB: "epi_got_acc g", 0xC: "epi_chunk_done j", 0xD: "gather_done"}


def main():
    mode = sys.argv[1] if len(sys.argv) > 1 else "parity"
    ks = int(sys.argv[2]) if len(sys.argv) > 2 else 11
    nat = aadff_b200.native
    n = nat.lib.aadff_debug_trace_entries()
    lens = aadff_b200.PSFNet(kernel_size=ks, device="cuda", mode=mode)
    if ks == 11:
        lens.load_net(os.path.join(ROOT, "tests/golden/rf50mm_PSFNet480x640_ks11.pkl"))
    img, dm = orc.synthetic_rgbd(1, 512, 512, seed=1234)
    foc = -orc.synthetic_focus(dm, 5).cuda() * 1e3
    img, dep = img.cuda(), -dm.cuda() * 1e3
    lens.render_stack(img, dep, foc)
    buf = torch.zeros(4 * n, dtype=torch.int64, device="cuda")
    nat.lib.aadff_debug_set_trace(buf.data_ptr())
    lens.render_stack(img, dep, foc)
    torch.cuda.synchronize()
    nat.lib.aadff_debug_set_trace(None)
    t = buf.cpu().view(4, n)
    ep = t[2]
    starts = [int(v) & 0xFFFFFFFFFF for v in ep.tolist() if (int(v) >> 48) == 0x8 >> 0 and v != 0 and ((int(v) >> 40) & 0xF00) == 0x800]
    t0, t1 = starts[1], starts[2]          # second tile of this CTA
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", f"trace_{mode}_ks{ks}.txt"), "w") as f:
        f.write(f"# mode={mode} ks={ks}; cycles relative to the start of CTA 0's 2nd tile; tile length {t1 - t0} cycles\n")
        for role, name in enumerate(["producer", "mma", "epi_e0", "epi_e7"]):
            f.write(f"## {name}\n")
            prev = None
            for v in t[role].tolist():
                v = int(v)
                if v == 0:
                    continue
                code, clk = v >> 40, v & 0xFFFFFFFFFF
                if clk < t0 - 3000 or clk > t1 + 1000:
                    continue
                f.write(f"{clk - t0:8d} {'' if prev is None else clk - prev:>7}  {NAMES.get(code >> 8, hex(code))} {code & 0xFF}\n")
                prev = clk
    print(open(os.path.join(ROOT, "gpurun_out", f"trace_{mode}_ks{ks}.txt")).read()[:200])


if __name__ == "__main__":
    main()
