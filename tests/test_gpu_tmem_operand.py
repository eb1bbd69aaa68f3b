"""Fused render kernel with its A operands in tensor memory (fused_tc_kernel.cuh, TA) against the shared-memory-operand
kernel (debug flag 1 << 20 keeps a launch on it).  Both evaluate the same fp16 products in the same order and gather in
the same tap order, so the stacks must be bit-identical."""
import pytest
import torch

from oracle import focal_stack_oracle as orc

SMEM_A = 1 << 20

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


def make_lens(pkg, ks, hidden_layers):
    from deeplens.psfnet_arch import MLP
    l = pkg.PSFNet(kernel_size=ks, device="cuda")
    torch.manual_seed(50 + ks + hidden_layers)
    l.psfnet = MLP(in_features=4, out_features=ks * ks, hidden_features=256, hidden_layers=hidden_layers).to("cuda")
    l.psfnet._evaluator = l._mlp_eval
    l._native = None
    gen = torch.Generator().manual_seed(11 + ks + hidden_layers)
    with torch.no_grad():
        for lin in l.psfnet.linear_layers():
            lin.bias.copy_(((torch.rand(lin.bias.shape, generator=gen) - 0.5) * 0.2).cuda())
    return l


def inputs(N, C, S, H, W, seed):
    img, dm = orc.synthetic_rgbd(N, H, W, seed=seed)
    if C == 1:
        img = img[:, :1]
    elif C == 4:
        img = torch.cat([img, 0.5 * img[:, :1]], 1)
    foc = -orc.synthetic_focus(dm, S) * 1e3
    return img.contiguous().cuda(), -dm.cuda() * 1e3, foc.cuda()


def both(pkg, fn):
    new = fn()
    pkg.native.lib.aadff_debug_set_flags(SMEM_A)
    try:
        old = fn()
    finally:
        pkg.native.lib.aadff_debug_set_flags(0)
    torch.cuda.synchronize()
    return new, old


# one tile; ragged edges with an odd tile count; C = 1 / 4; several tiles per CTA (the gather of a tile runs during the
# next tile, the last one after the tile loop)
SHAPES = [(1, 3, 1, 8, 16), (1, 3, 3, 37, 50), (2, 1, 2, 24, 40), (1, 4, 3, 29, 61), (1, 3, 5, 256, 256)]


@pytest.mark.parametrize("ks,hidden_layers", [(11, 8), (13, 8), (15, 8), (11, 2), (11, 5), (11, 0)])
@pytest.mark.parametrize("mode", ["parity", "econ8", "econ"])
def test_tmem_operand_path_bit_identical(pkg, ks, hidden_layers, mode):
    """ks <= 13 with at least two hidden groups takes the tensor-memory path; ks = 15 (one head block of N = 240, more
    than the 192 columns the path leaves for the head) and the single-hidden-group net fall back to the shared-memory
    path, so the comparison is trivially equal there.  tests/test_gpu_fused_vs_f64.py compares both paths with float64."""
    lens = make_lens(pkg, ks, hidden_layers)
    for i, (N, C, S, H, W) in enumerate(SHAPES):
        img, dep, foc = inputs(N, C, S, H, W, seed=20 + i)
        new, old = both(pkg, lambda: lens.render_stack(img, dep, foc, mode=mode))
        assert torch.isfinite(new).all()
        assert torch.equal(new, old), (ks, hidden_layers, mode, (N, C, S, H, W), float((new - old).abs().max()))


@pytest.mark.parametrize("mode", ["parity", "econ8"])
def test_tmem_operand_path_tile_row_ranges(pkg, mode):
    lens = make_lens(pkg, 11, 8)
    img, dep, foc = inputs(2, 3, 3, 45, 70, seed=33)
    rows_total = 2 * 3 * ((45 + 7) // 8)
    for (r0, r1) in [(0, rows_total), (1, 4), (5, rows_total - 2), (7, 8)]:
        new, old = both(pkg, lambda: lens.render_stack_rows(img, dep, foc, r0, r1, mode=mode))
        assert torch.equal(new, old), (mode, r0, r1)
