"""CPU tests of oracle/tc_arith_oracle.py, the float64 emulation of the fused tensor-core kernel's per-mode
arithmetic that tests/test_gpu_fused_vs_f64.py compares the kernel with."""
import os
import re

import pytest
import torch

from oracle import focal_stack_oracle as orc
from oracle import tc_arith_oracle as tao

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def noise_inputs(N, S, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(N, 3, H, W, generator=g)
    depth = -(200 + 19800 * torch.rand(N, 1, H, W, generator=g))
    foc = -(200 + 19800 * torch.rand(N, S, generator=g))
    return img, depth, foc


# DESIGN.md section 5, by layer name: which layers of the reference network (L1..L9 hidden, then the head) take two
# terms, or one.  Groups of a network with h hidden layers: L1 .. L(h+1), then the head blocks.
DESIGN_TABLE = {
    "parity": lambda layer: 3,
    "fast": lambda layer: 1,
    "econ": lambda layer: 3 if layer <= 4 else 2,           # 3 terms for L1-L4; 2 for L5-L9 and the head
    "econ8": lambda layer: 3 if layer <= 7 else 2,          # 3 terms for L1-L7; 2 for L8, L9 and the head
    "mixed": lambda layer: 3 if layer <= 3 else 1,          # 3 terms for L1-L3, then 1
}


@pytest.mark.parametrize("mode", sorted(DESIGN_TABLE))
def test_term_pattern_restates_the_mode_table(mode):
    for h in range(0, 9):
        for nb in range(1, 5):
            # group g holds layer g + 1; head block b is group h + 1 + b, so it takes the rule of "layer" h + 2 + b
            # (a shallower net reaches its reduced region, if at all, in the head)
            layers = list(range(1, h + 2)) + [h + 2 + b for b in range(nb)]
            want = [DESIGN_TABLE[mode](layer) for layer in layers]
            got = tao.term_pattern(mode, h, nb)
            assert got == want, (mode, h, nb, got, want)
    assert tao.term_pattern("econ8", 8, 1) == [3] * 7 + [2] * 3           # the reference network: L8, L9, head
    assert tao.term_pattern("econ8", 5, 2) == [3] * 7 + [2]                 # head block 0 three terms, block 1 two
    assert tao.term_pattern("econ", 2, 2) == [3] * 4 + [2]
    assert tao.term_pattern("mixed", 1, 2) == [3, 3, 3, 1]
    assert tao.term_pattern("econ8", 2, 4) == [3] * 7                       # nothing reduced: parity


def test_term_pattern_first_groups_match_the_kernel_constants():
    """The emulation's first reduced groups are the kernel's (fused_tc_kernel.cuh)."""
    with open(os.path.join(ROOT, "aberration-aware-depth-from-focus_b200", "csrc", "fused_tc_kernel.cuh")) as f:
        src = f.read()
    const = {k: int(v) for k, v in re.findall(r"constexpr int TC_(\w+)_FIRST_GROUP = (\d+);", src)}
    assert const == {"MIXED": tao.MODE_PATTERN["mixed"][0], "ECON": tao.MODE_PATTERN["econ"][0],
                     "ECON8": tao.MODE_PATTERN["econ8"][0]}


@pytest.mark.parametrize("ks,blocks", [(1, [16]), (11, [128]), (13, [176]), (15, [240]), (17, [256, 48]),
                                       (21, [256, 192]), (23, [256, 256, 32]), (27, [256, 256, 224]),
                                       (31, [256, 256, 256, 208])])
def test_head_blocks(ks, blocks):
    assert tao.head_blocks(ks) == blocks


def test_fp16_roundings():
    x = torch.tensor([0.0, 1.0, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 1.0 - 2.0 ** -12, 3.0 * 2.0 ** -25,
                      65504.0, 2.0 ** -14 * 1.5 + 2.0 ** -26], dtype=torch.float64)
    assert tao.fp16_rz(x).tolist() == [0.0, 1.0, 1.0, 1.0 + 2.0 ** -10, 1.0 - 2.0 ** -11, 2.0 ** -24, 65504.0,
                                       2.0 ** -14 * 1.5]
    assert tao.fp16_rn(x)[2:4].tolist() == [1.0, 1.0 + 2.0 ** -9]               # ties to even


def _activations(Ws, bs, o):
    a, out = o.double(), []
    for W, b in zip(Ws[:-1], bs[:-1]):
        a = torch.relu(a @ W.double().T + b.double())
        out.append(tao.f32(a))
    return torch.cat([x.reshape(-1) for x in out])


def test_fp16_split_keeps_the_activation():
    """On seeded nets the fp16 (hi, lo) split holds an activation a to within 2^-22 |a| (round-to-nearest hi, layer 0)
    or 2^-21 |a| (round-toward-zero hi, the hidden layers), down to a floor of 2^-25 where lo is subnormal."""
    Ws, bs = tao.seeded_net(11, 8, 1)
    o = torch.rand(4096, 4, generator=torch.Generator().manual_seed(2))
    o[:, :2] = o[:, :2] * 2 - 1
    a = _activations(Ws, bs, o)
    a = a[(a >= 2.0 ** -14) & (a <= 65504)]                 # normal fp16 range
    assert a.numel() > 100000
    hi, lo = tao.split_rn(a)
    assert bool(((a - hi - lo).abs() <= torch.maximum(2.0 ** -22 * a, torch.full_like(a, 2.0 ** -25))).all())
    big = a >= 2.0 ** -3                                       # lo is a normal fp16 number
    assert bool(((a - hi - lo).abs()[big] <= 2.0 ** -22 * a[big]).all())
    hi, lo = tao.split_relu_rz(a)
    assert bool((hi <= a).all())
    assert bool(((a - hi - lo).abs() <= torch.maximum(2.0 ** -21 * a, torch.full_like(a, 2.0 ** -25))).all())


@pytest.fixture(scope="module")
def small_case():
    img, depth, foc = noise_inputs(1, 2, 12, 20, seed=4)
    return img, depth, foc


@pytest.mark.parametrize("net", ["rf50mm", "seeded"])
def test_three_term_emulation_matches_float64_truth(net, small_case, rf50mm_weights):
    """SURVEY.md section 7.3 measured the fp16 3-term arithmetic with layer 0 in fp32 at 1.2e-6 .. 6e-6 of the fp32
    reference on the rf50mm checkpoint; against float64 the emulation must stay within 1e-6."""
    Ws, bs = rf50mm_weights if net == "rf50mm" else tao.seeded_net(11, 8, 5)
    img, depth, foc = small_case
    truth = tao.render_truth(Ws, bs, img, depth, foc, 11)
    ref64 = orc.render_stack(Ws, bs, img, depth, foc, 11, dtype=torch.float64)
    assert float((truth - ref64).abs().max()) == 0.0                         # the oracle itself, rearranged
    emu = tao.render_emulated(Ws, bs, img, depth, foc, 11, tao.term_pattern("parity", 8, 1))
    err = float((emu - truth).abs().max())
    assert err < 1e-6, err


@pytest.mark.parametrize("drop", ["hh", "lh", "hl"])
def test_dropping_any_term_changes_the_result(drop, small_case):
    """Each of the three terms carries weight: without it the render moves by far more than the 3-term emulation's
    distance from the truth."""
    Ws, bs = tao.seeded_net(11, 8, 5)
    img, depth, foc = small_case
    truth = tao.render_truth(Ws, bs, img, depth, foc, 11)
    three = tao.render_emulated(Ws, bs, img, depth, foc, 11, [3] * 10)
    base = float((three - truth).abs().max())
    terms = [tuple(t for t in ("hh", "lh", "hl") if t != drop)] * 10
    moved = float((tao.render_emulated(Ws, bs, img, depth, foc, 11, terms) - three).abs().max())
    assert moved > 1e-6 and moved > 50 * base, (drop, moved, base)
    # dropped in one layer only (L2), the change is still visible
    one = [3] * 10
    one[1] = terms[0]
    moved1 = float((tao.render_emulated(Ws, bs, img, depth, foc, 11, one) - three).abs().max())
    assert moved1 > 10 * base, (drop, moved1, base)


def test_pred_emulated_is_normalised_and_matches_mlp_forward():
    Ws, bs = tao.seeded_net(7, 2, 6)
    probes = torch.rand(500, 4, generator=torch.Generator().manual_seed(7))
    probes[:, :2] = probes[:, :2] * 2 - 1
    psf = tao.pred_emulated(Ws, bs, probes, tao.term_pattern("parity", 2, 1))
    assert psf.shape == (500, 7, 7)
    assert float((psf.sum((-1, -2)) - 1).abs().max()) < 1e-12
    ref = orc.mlp_forward(Ws, bs, probes, torch.float64).reshape(-1, 7, 7)
    assert float((psf - ref).abs().max()) < 1e-6
