"""Float64 emulation of the fused tensor-core kernel's declared arithmetic (fused_tc_kernel.cuh).

TEST INFRASTRUCTURE ONLY, like the rest of ``oracle/``: nothing in the product package imports it.

``focal_stack_oracle.render_stack(..., dtype=torch.float64)`` is what the network *means*.  This module gives what
each mode of the tensor-core kernel *computes*: the same network with its operands split into fp16 parts and only the
MMA terms the mode declares, so that a test can tell "the kernel ran its own pattern" from "the kernel ran a
neighbouring pattern", which the accuracy bounds alone cannot.  Everything is restated from the kernel's comments and
DESIGN.md section 5, not imported from the C++:

* layer groups: one per hidden MMA layer (L1 .. L(h+1) for ``MLP(..., hidden_layers=h)``), then one per <= 256-column
  block of the head, whose k*k outputs are padded to a multiple of 16;
* mode -> (first reduced group, terms): parity none, fast (0, 1), econ (4, 2), econ8 (7, 2), mixed (3, 1); groups
  before ``first`` take three terms.  When ``first`` is not below the number of groups nothing is reduced and the
  network runs as in parity mode;
* terms of a K-step: 3 = Ah*Wh + Al*Wh + Ah*Wl, 2 = Ah*Wh + Al*Wh, 1 = Ah*Wh, where W = Wh + Wl is the fp16 split of
  the fp32 weight (round to nearest both times) and A = Ah + Al that of the activation;
* layer 0 (4 -> 64) runs in fp32 FMAs; its output is split with round-to-nearest.  A hidden layer's output is split
  with hi = round-toward-zero(relu(a)), lo = rn(relu(a - hi)) when its consumer reads lo parts, else hi = rn(relu(a));
* a hidden group's accumulator starts at fp16(b) + fp16(b - fp16(b)) (the bias slab);
* head: sigmoid as 1 / (1 + 2^(z * fp32(-log2 e) + b')) with b' = fp32(-log2 e * b), L1 normalised with
  max(sum, 1e-12), then the replicate-border k x k gather.

Sums over K are taken in float64; the kernel accumulates in fp32, so the two agree to fp32-accumulation level, not bit
for bit.  The econ / econ8 weights are the library's *calibrated* fp16 roundings, which are not exposed; the
emulation of those modes is the plain-rounding variant the library runs under debug flag 256.
"""
from __future__ import annotations

import math
from typing import Sequence

import torch

from oracle import focal_stack_oracle as orc

MAX_GROUPS = 16
MODE_PATTERN = {            # mode -> (first reduced group, terms of the reduced groups)
    "parity": (MAX_GROUPS, 3),
    "fast": (0, 1),
    "econ": (4, 2),
    "econ8": (7, 2),
    "mixed": (3, 1),
}
TERMS = {3: ("hh", "lh", "hl"), 2: ("hh", "lh"), 1: ("hh",)}     # h/l of (activation, weight)
NEG_LOG2E_F32 = float(torch.tensor(-1.4426950408889634, dtype=torch.float32))


def head_blocks(ks: int) -> list[int]:
    """MMA N of each head block: k*k outputs padded to a multiple of 16, cut into blocks of <= 256 columns."""
    pad = (ks * ks + 15) // 16 * 16
    return [min(256, pad - 256 * b) for b in range((pad + 255) // 256)]


def pattern_terms(first: int, terms: int, n_groups: int) -> list[int]:
    """Terms of each group for 'groups from `first` on take `terms`, the groups before three'."""
    if first >= n_groups:
        return [3] * n_groups
    return [3 if g < first else terms for g in range(n_groups)]


def term_pattern(mode: str, hidden_layers: int, n_head_blocks: int) -> list[int]:
    """MMA terms of each layer group of ``MLP(..., hidden_layers)`` with `n_head_blocks` head blocks in `mode`
    (one of MODE_PATTERN; fp32 mode has no tensor-core groups)."""
    first, terms = MODE_PATTERN[mode]
    return pattern_terms(first, terms, hidden_layers + 1 + n_head_blocks)


def seeded_net(ks: int, hidden_layers: int, seed: int):
    """Kaiming-uniform MLP(4, ks^2, 256, hidden_layers) (the reference's initialiser) with biases in [-0.1, 0.1]:
    the random networks the emulation is tested on, on the host and against the kernel."""
    g = torch.Generator().manual_seed(seed)
    dims = [4, 64, 256] + [256] * hidden_layers + [ks * ks]
    Ws, bs = [], []
    for fin, fout in zip(dims[:-1], dims[1:]):
        Ws.append((torch.rand(fout, fin, generator=g) * 2 - 1) * math.sqrt(6.0 / fin))
        bs.append((torch.rand(fout, generator=g) - 0.5) * 0.2)
    return Ws, bs


# ----------------------------------------------------------------------------------------------- roundings
def f32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(torch.float64)


def fp16_rn(x: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even to fp16 (x holds fp32 values), returned as float64."""
    return x.to(torch.float32).to(torch.float16).to(torch.float64)


def fp16_rz(x: torch.Tensor) -> torch.Tensor:
    """Round toward zero to fp16 (x holds fp32 values inside the fp16 range), returned as float64."""
    x = x.to(torch.float64)
    _, e = torch.frexp(x)                                   # |x| in [2^(e-1), 2^e)
    ulp = torch.exp2(torch.clamp(e - 11, min=-24).to(torch.float64))
    return torch.trunc(x / ulp) * ulp


def split_rn(a: torch.Tensor):
    """(hi, lo) with hi = rn(a), lo = rn(a - hi): the weight split (pack_group) and layer 0's activation split."""
    hi = fp16_rn(a)
    return hi, fp16_rn(f32(a) - hi)


def split_relu_rz(a: torch.Tensor):
    """(hi, lo) of relu(a) with hi = rz(relu(a)), lo = rn(relu(a - hi)): a hidden layer's output for a consumer that
    reads lo parts (epi_group8 / epi_ta16)."""
    a = f32(a)
    hi = fp16_rz(torch.relu(a))
    return hi, fp16_rn(torch.relu(a - hi))


# ----------------------------------------------------------------------------------------------- forward pass
def _term_set(t) -> tuple:
    return TERMS[t] if isinstance(t, int) else tuple(t)


def _mma(Ah, Al, W, term_set):
    Wh, Wl = split_rn(W)
    parts = {"hh": (Ah, Wh), "lh": (Al, Wh), "hl": (Ah, Wl), "ll": (Al, Wl)}
    acc = 0.0
    for name in term_set:
        a, w = parts[name]
        acc = acc + a @ w.T
    return acc


def mlp_emulated(Ws: Sequence[torch.Tensor], bs: Sequence[torch.Tensor], o: torch.Tensor, terms) -> torch.Tensor:
    """[M,4] fp32 network inputs -> [M,k*k] L1-normalised PSFs as the kernel's arithmetic gives them.

    `terms`: one entry per layer group (term_pattern's output); an entry is 1, 2, 3 or a tuple of the term names
    'hh', 'lh', 'hl' (activation part, weight part) to take a term out of a pattern."""
    dev = o.device
    Ws = [W.to(dev, torch.float64) for W in Ws]
    bs = [b.to(dev, torch.float64) for b in bs]
    n_hidden = len(Ws) - 2
    kk = Ws[-1].shape[0]
    blocks = []
    t0 = 0
    while t0 < kk:
        blocks.append((t0, min(t0 + 256, kk)))
        t0 += 256
    assert len(terms) == n_hidden + len(blocks), (len(terms), n_hidden, len(blocks))
    sets = [_term_set(t) for t in terms]
    # layer 0: fp32 FMAs in the order b + w.x*x + w.y*y + w.z*z + w.w*fz, ReLU
    o = o.to(torch.float64)
    a = bs[0].expand(o.shape[0], -1).clone()
    for k in range(4):
        a = f32(a + Ws[0][:, k] * o[:, k:k + 1])         # the float64 product is exact, one rounding = the FMA's
    a = torch.relu(a)
    Ah, Al = split_rn(a)
    if "lh" not in sets[0]:
        Al = torch.zeros_like(Al)
    for g in range(n_hidden):
        bh, bl = split_rn(bs[g + 1])
        acc = f32(bh + bl + _mma(Ah, Al, Ws[g + 1], sets[g]))
        if "lh" in sets[g + 1]:
            Ah, Al = split_relu_rz(acc)
        else:
            Ah, Al = fp16_rn(torch.relu(acc)), torch.zeros_like(acc)
    z = torch.cat([f32(_mma(Ah, Al, Ws[-1][t0:t1], sets[n_hidden + i])) for i, (t0, t1) in enumerate(blocks)], dim=1)
    b_head = f32(NEG_LOG2E_F32 * f32(bs[-1]))
    sg = 1.0 / (1.0 + torch.exp2(f32(z * NEG_LOG2E_F32 + b_head)))
    return sg / sg.sum(-1, keepdim=True).clamp_min(1e-12)


def pred_emulated(Ws, bs, probes: torch.Tensor, terms) -> torch.Tensor:
    """PSFNet.pred in the kernel's arithmetic: probes [M,4] (fp32) -> [M,ks,ks] float64."""
    ks = math.isqrt(Ws[-1].shape[0])
    return mlp_emulated(Ws, bs, probes.to(torch.float32), terms).reshape(-1, ks, ks)


def stack_inputs(depth: torch.Tensor, foc: torch.Tensor, device=None) -> torch.Tensor:
    """Network inputs of a focal stack, [N,S,H,W,4] fp32 (focal_stack_oracle.model_input per slice)."""
    S = foc.shape[1]
    o = torch.stack([orc.model_input(depth.reshape(depth.shape[0], *depth.shape[-2:]).cpu(), foc[:, s].cpu())
                     for s in range(S)], dim=1)
    return o.to(device) if device is not None else o


def render_emulated(Ws, bs, img: torch.Tensor, depth: torch.Tensor, foc: torch.Tensor, ks: int, terms) -> torch.Tensor:
    """render_stack [N,C,S,H,W] (float64) in the kernel's arithmetic, on img's device."""
    o = stack_inputs(depth, foc, img.device)
    N, S, H, W, _ = o.shape
    psf = mlp_emulated(Ws, bs, o.reshape(-1, 4), terms).reshape(N, S, H, W, ks * ks)
    return _gather_stack(img, psf, ks)


def render_truth(Ws, bs, img: torch.Tensor, depth: torch.Tensor, foc: torch.Tensor, ks: int) -> torch.Tensor:
    """focal_stack_oracle's float64 render_stack evaluated on img's device: the same torch operations
    (mlp_forward, local_psf_render), with the network inputs built on the host as the oracle builds them."""
    o = stack_inputs(depth, foc, img.device)
    N, S, H, W, _ = o.shape
    dev = img.device
    psf = orc.mlp_forward([w.to(dev) for w in Ws], [b.to(dev) for b in bs], o, torch.float64)
    return _gather_stack(img, psf.reshape(N, S, H, W, ks * ks), ks)


def _gather_stack(img, psf, ks):
    S = psf.shape[1]
    img = img.to(torch.float64)
    return torch.stack([orc.local_psf_render(img, psf[:, s], ks) for s in range(S)], dim=2)
