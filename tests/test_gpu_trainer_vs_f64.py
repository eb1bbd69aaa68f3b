"""The PSFNet fitting step on the device (csrc/train_kernels.cuh, aadff_trainer_* in csrc/aadff_api.cu) against
float64, step by step, at every kernel size, several batch and network shapes, and several AdamW settings.

Every step reads the device parameters P_before, steps, then reads the gradients G, the parameters P_after and the
predicted PSFs p, and checks
- the loss and p against the float64 forward at P_before (oracle/train_oracle.py: step_f64);
- every dW and db against float64 autograd at P_before, and that a gradient which is exactly 0 in float64 (a unit that
  is dead for the whole batch, or ks 1) is exactly 0 on the device;
- P_after, element by element, against torch's AdamW update in float64 (adamw_f64) of P_before with the device's own
  G of this and every earlier step, the moments carried across steps in float64.
Comparing every step from the device's own P_before and G keeps the parameter check free of Adam's normalisation of
small, noisy gradients, so it can be tight: the tolerance is in units of ulp(P) + 1e-6 lr.  Probes come from the
oracle's sampler, which redraws probes whose float64 forward sits next to a ReLU kink or the 1e-12 clamp of the L1
normalisation (there fp32 and float64 may take different branches).  Observed errors per case, and which tests
catch four deliberate library mutations: profiles/NOTES_r06_trainer_vs_f64.md.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import train_oracle as tro

pytestmark = pytest.mark.gpu

# Tolerances; the largest errors a B200 showed over two runs of all cases are in brackets.
LOSS_TOL = 2e-6          # relative, times sqrt(batch / 128) above 128 probes [6.7e-7 at 128, 9.1e-7 at 1000]: the loss
                         # is an atomicAdd of one fp32 term per probe in any order (two orders differed by 5.4e-7 at 129)
P_TOL = 2e-6             # of the largest p of the batch [1.03e-6, after a step at lr 1e-2]
GRAD_TOL = 1e-5          # of the tensor's largest |float64 gradient| [2.3e-6]
PARAM_TOL = 3.0          # in units of ulp(float64 reference) + 1e-6 * lr [1.52]


def ref_dims(kk):
    """MLP(4, kk, 256, 8) of PSFNet (psfnet.py:58): 4 -> 64 -> 256 x 9 -> kk."""
    return [4, 64] + [256] * 9 + [kk]


@pytest.fixture(scope="module")
def pkg():
    import aadff_b200
    return aadff_b200


class StepChecker:
    """One trainer, stepped on the default stream and checked against the oracle after every step."""

    def __init__(self, pkg, Ws, bs, batch, betas=(0.9, 0.999), eps=1e-8, wd=1e-2, seed=0):
        self.nat = pkg.native
        self.trainer = self.nat.NativeTrainer(Ws, bs, batch, 0, betas, eps, wd)
        self.batch, self.kk, self.L = batch, Ws[-1].shape[0], len(Ws)
        self.betas, self.eps, self.wd = betas, eps, wd
        self.gen = torch.Generator().manual_seed(seed)
        self.loss_dev = torch.zeros(1, device="cuda")
        self.steps = self.redrawn = 0
        self.worst = dict(loss=0.0, p=0.0, grad=0.0, param=0.0)
        Wd, bd = self.trainer.read(0)
        assert all(np.array_equal(a, b) for a, b in zip(Wd + bd, list(Ws) + list(bs)))    # the upload is exact
        self.m = tro.zero_moments(Wd + bd)
        self.v = tro.zero_moments(Wd + bd)

    def pred(self):
        out = np.empty((self.batch, self.kk), np.float32)
        c_f32p = ctypes.POINTER(ctypes.c_float)
        self.nat.check(self.nat.lib.aadff_trainer_read(self.trainer.handle, 2, (c_f32p * 1)(out.ctypes.data_as(c_f32p)),
                                                       None, None))
        return out

    def step(self, lr):
        Wb, bb = self.trainer.read(0)
        inp, n = tro.sample_probes(Wb, bb, self.batch, self.gen)
        tgt = tro.random_targets(self.batch, self.kk, self.gen)
        self.redrawn += n
        inp_d, tgt_d = torch.from_numpy(inp).cuda(), torch.from_numpy(tgt).cuda()
        self.nat.check(self.nat.lib.aadff_trainer_step(self.trainer.handle, inp_d.data_ptr(), tgt_d.data_ptr(), lr,
                                                       self.loss_dev.data_ptr(), None))
        Gw, Gb = self.trainer.read(1)
        Wa, ba = self.trainer.read(0)
        p = self.pred()
        loss = float(self.loss_dev)
        self.steps += 1
        k = self.steps
        loss64, p64, dW64, db64 = tro.step_f64(Wb, bb, inp, tgt)

        e_loss = abs(loss - loss64) / loss64 if loss64 > 0 else (0.0 if loss == 0 else math.inf)
        assert e_loss <= LOSS_TOL * max(1.0, math.sqrt(self.batch / 128)), f"step {k}: loss {loss!r} vs {loss64!r}"
        e_p = float(np.abs(p - p64).max() / p64.max())
        assert e_p <= P_TOL, f"step {k}: p off by {e_p:.2e} of max p"
        e_g = 0.0
        for l, (g, r) in enumerate(zip(Gw + Gb, dW64 + db64)):
            name = f"{'dW' if l < self.L else 'db'}[{l % self.L}]"
            assert np.all(g[r == 0] == 0), f"step {k}: {name} is not 0 where the float64 gradient is exactly 0"
            scale = np.abs(r).max()
            e = float(np.abs(g - r).max() / scale) if scale > 0 else 0.0
            assert e <= GRAD_TOL, f"step {k}: {name} off by {e:.2e} of its max |ref| {scale:.2e}"
            e_g = max(e_g, e)
        P_ref = tro.adamw_f64(Wb + bb, Gw + Gb, self.m, self.v, k, lr, self.betas, self.eps, self.wd)
        e_par = 0.0
        for l, (a, r) in enumerate(zip(Wa + ba, P_ref)):
            unit = np.spacing(np.abs(r).astype(np.float32)).astype(np.float64) + 1e-6 * lr
            e = float((np.abs(a - r) / unit).max())
            assert e <= PARAM_TOL, (f"step {k}: parameter tensor {l} off by {e:.1f} (ulp + 1e-6 lr) against AdamW in "
                                    f"float64 (lr {lr}, betas {self.betas}, eps {self.eps}, wd {self.wd})")
            e_par = max(e_par, e)
        for key, e in zip(("loss", "p", "grad", "param"), (e_loss, e_p, e_g, e_par)):
            self.worst[key] = max(self.worst[key], e)
        return dict(P_before=Wb + bb, P_after=Wa + ba, G=Gw + Gb, inp=inp)

    def report(self, label):
        w = self.worst
        print(f"\n[trainer vs f64] {label}: {self.steps} steps, batch {self.batch}, {self.redrawn} probes redrawn; "
              f"loss {w['loss']:.2e} rel, p {w['p']:.2e} of max p, grad {w['grad']:.2e} of max |ref|, "
              f"param {w['param']:.2f} (ulp + 1e-6 lr)")

    def close(self):
        self.trainer.close()


def run_case(pkg, label, dims, batch, lrs, seed, bias_scale=0.1, **adamw):
    gen = torch.Generator().manual_seed(seed)
    Ws, bs = tro.kaiming_net(dims, gen, bias_scale)
    chk = StepChecker(pkg, Ws, bs, batch, seed=seed, **adamw)
    try:
        for lr in lrs:
            chk.step(lr)
        chk.report(label)
    finally:
        chk.close()


@pytest.mark.parametrize("ks", [1, 3, 5, 11, 13, 17, 31])
def test_every_kernel_size(pkg, ks):
    """kk from 1 to 961: up to 31 taps per lane in the head kernel, ragged N tiles of the head GEMM and ragged M tiles
    of its dW."""
    run_case(pkg, f"ks {ks}", ref_dims(ks * ks), 128, [1e-3] * 3, seed=ks)


@pytest.mark.parametrize("batch", [1, 7, 32, 33, 129, 1000])
def test_every_batch_size(pkg, batch):
    """Ragged M tiles in the forward and dX GEMMs and a ragged K in dW = dZ^T X (batch % 32 != 0); one probe."""
    run_case(pkg, f"ks 11, batch {batch}", ref_dims(121), batch, [1e-3] * 3, seed=100 + batch)


NETS = {
    "one layer": lambda kk: [4, kk],                              # no hidden layer, no dX chain
    "narrow": lambda kk: [4, 8, 8, kk],
    "ragged": lambda kk: [4, 40, 136, 200, kk],                   # partial K and N tiles in all three GEMM orientations
    "16 layers": lambda kk: [4, 64] + [128] * 14 + [kk],          # MAX_LAYERS
}


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("ks", [5, 17])
def test_network_shapes(pkg, ks, net):
    run_case(pkg, f"ks {ks}, {net}", NETS[net](ks * ks), 33, [1e-3] * 3, seed=7 * ks + len(net))


def test_from_scratch_start_has_exactly_zero_gradients_for_dead_units(pkg):
    """The reference's initialiser (kaiming-uniform weights, zero biases): units dead for the whole batch get gradients
    that are exactly 0, on the device as in float64 (StepChecker checks every such element)."""
    gen = torch.Generator().manual_seed(11)
    Ws, bs = tro.kaiming_net(ref_dims(121), gen)
    chk = StepChecker(pkg, Ws, bs, 128, seed=11)
    try:
        for _ in range(3):
            out = chk.step(1e-3)
            pre, _, _ = tro.forward_f64(out["P_before"][:chk.L], out["P_before"][chk.L:], out["inp"])
            dead = sum(int(((z <= 0).all(0)).sum()) for z in pre)
            assert dead > 0, "no unit is dead for the whole batch: the case tests nothing"
            n_zero = sum(int((g == 0).sum()) for g in out["G"])
            assert n_zero > 0
        chk.report(f"ks 11 from scratch ({dead} dead units, {n_zero} zero gradients in the last step)")
    finally:
        chk.close()


def test_ks1_gradients_are_zero_and_only_decay_moves(pkg):
    """ks 1: p = s / s = 1 whatever the network, so the loss and every gradient are exactly 0 and AdamW only decays:
    P_after = P_before (1 - lr wd), with lr wd = 2^-10 exact in fp32, to 1 ulp."""
    gen = torch.Generator().manual_seed(1)
    lr, wd = 2.0 ** -7, 2.0 ** -3
    Ws, bs = tro.kaiming_net(ref_dims(1), gen, 0.1)
    chk = StepChecker(pkg, Ws, bs, 128, wd=wd, seed=1)
    try:
        for _ in range(3):
            out = chk.step(lr)
            assert float(chk.loss_dev) == 0.0
            assert all(np.all(g == 0) for g in out["G"])
            for a, b in zip(out["P_after"], out["P_before"]):
                ref = b.astype(np.float64) * (1 - lr * wd)
                assert np.all(np.abs(a - ref) <= np.spacing(np.abs(ref).astype(np.float32)))
        chk.report("ks 1, lr 2^-7, wd 2^-3")
    finally:
        chk.close()


def test_normalisation_clamp_both_sides(pkg):
    """A saturated head at ks 3 (head biases near -31): probes on both sides of S = 1e-12, so train_head_kernel takes
    both the normalised branch and the clamped one (no normalisation gradient)."""
    gen = torch.Generator().manual_seed(3)
    Ws, bs = tro.kaiming_net([4, 32, 32, 9], gen, 0.1)
    bs = tro.saturate_head(Ws, bs, gen)
    chk = StepChecker(pkg, Ws, bs, 128, seed=3)
    try:
        for _ in range(3):
            out = chk.step(1e-4)
            _, S, _ = tro.forward_f64(out["P_before"][:chk.L], out["P_before"][chk.L:], out["inp"])
            below = int((S < tro.NORMALIZE_EPS).sum())
            assert 0 < below < chk.batch, f"{below} of {chk.batch} probes below the clamp"
        chk.report(f"ks 3, saturated head (bias {float(bs[-1].mean()):.1f}, {below} of 128 probes below the clamp)")
    finally:
        chk.close()


def test_adamw_strong_decay(pkg):
    """lr 1e-2, wd 0.1: decay moves a weight by 1e-3 |w|, about a thousand times the parameter tolerance."""
    run_case(pkg, "ks 5, lr 1e-2, wd 0.1", ref_dims(25), 128, [1e-2] * 3, seed=21, wd=0.1)


def test_adamw_eps_and_betas(pkg):
    run_case(pkg, "ks 5, eps 1e-3, betas (0.8, 0.99)", ref_dims(25), 128, [1e-3] * 5, seed=22, eps=1e-3,
             betas=(0.8, 0.99))


def test_adamw_zero_lr_step_advances_moments_only(pkg):
    """A step at lr 0 leaves the parameters bit-identical but advances the moments and the step count: the next step's
    parameters are checked against AdamW whose moments include the lr-0 step."""
    gen = torch.Generator().manual_seed(23)
    Ws, bs = tro.kaiming_net(ref_dims(25), gen, 0.1)
    chk = StepChecker(pkg, Ws, bs, 33, seed=23)
    try:
        out = chk.step(0.0)
        assert all(np.array_equal(a, b) for a, b in zip(out["P_after"], out["P_before"]))
        chk.step(1e-3)
        chk.step(1e-3)
        chk.report("ks 5, lr 0 then 1e-3")
    finally:
        chk.close()


def test_adamw_long_cosine_schedule(pkg):
    """200 steps of CosineAnnealingLR from 1e-2 on a small net: bias correction at high step counts."""
    n = 200
    lrs = [0.5 * 1e-2 * (1 + math.cos(math.pi * i / n)) for i in range(n)]
    run_case(pkg, "ks 3, [4, 16, 24, 9], 200 cosine steps from lr 1e-2", [4, 16, 24, 9], 33, lrs, seed=24)


def test_two_trainers_on_two_streams_are_bit_identical(pkg):
    """Two trainers from the same parameters, stepped interleaved on two streams with the same inputs, and a third
    stepped alone on the default stream: bit-identical parameters and gradients after 10 steps (nothing is shared
    between trainers, and the graph's dW / db side branches do not race).  The loss is an atomicAdd over probes, so it
    is only compared to LOSS_TOL."""
    nat = pkg.native
    gen = torch.Generator().manual_seed(31)
    Ws, bs = tro.kaiming_net(ref_dims(121), gen, 0.1)
    steps, batch = 10, 129
    inps = [torch.from_numpy(tro.draw_probes(batch, gen)).cuda() for _ in range(steps)]
    tgts = [torch.from_numpy(tro.random_targets(batch, 121, gen)).cuda() for _ in range(steps)]
    trainers = [nat.NativeTrainer(Ws, bs, batch, 0) for _ in range(3)]
    losses = torch.zeros(3, steps, device="cuda")
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    try:
        for s in streams:
            s.wait_stream(torch.cuda.current_stream())
        for i in range(steps):
            for j, s in enumerate(streams):
                nat.check(nat.lib.aadff_trainer_step(trainers[j].handle, inps[i].data_ptr(), tgts[i].data_ptr(), 1e-3,
                                                     losses[j, i].data_ptr(), s.cuda_stream))
        for i in range(steps):
            nat.check(nat.lib.aadff_trainer_step(trainers[2].handle, inps[i].data_ptr(), tgts[i].data_ptr(), 1e-3,
                                                 losses[2, i].data_ptr(), None))
        streams_of = [streams[0].cuda_stream, streams[1].cuda_stream, None]
        P = [t.read(0, st) for t, st in zip(trainers, streams_of)]
        G = [t.read(1, st) for t, st in zip(trainers, streams_of)]
        torch.cuda.synchronize()
        for j in (1, 2):
            for a, b in zip(P[0][0] + P[0][1], P[j][0] + P[j][1]):
                assert np.array_equal(a, b), f"trainer {j}: parameters differ"
            for a, b in zip(G[0][0] + G[0][1], G[j][0] + G[j][1]):
                assert np.array_equal(a, b), f"trainer {j}: gradients differ"
        assert not np.array_equal(P[0][0][0], Ws[0])                       # the steps did move the parameters
        rel = ((losses - losses[0]).abs() / losses[0]).max()
        assert float(rel) <= LOSS_TOL
        print(f"\n[trainer vs f64] two streams: bit-identical after {steps} steps, loss spread {float(rel):.1e}")
    finally:
        for t in trainers:
            t.close()


def test_train_psfnet_lr_schedule_and_psf_size(pkg, monkeypatch):
    """PSFNet.train_psfnet hands aadff_trainer_step the lr of CosineAnnealingLR(T_max=iters) over iters + 1 steps,
    and refuses, before any step, PSFs whose size is not kernel_size^2."""
    nat = pkg.native
    lrs = []
    step = nat.lib.aadff_trainer_step

    def recording_step(handle, inp, tgt, lr, loss, stream):
        lrs.append(lr)
        return step(handle, inp, tgt, lr, loss, stream)

    monkeypatch.setattr(nat.lib, "aadff_trainer_step", recording_step)
    ks, iters, lr0, bs = 5, 12, 3e-3, 16

    def data(bs, spp, taps=ks * ks):
        x = torch.rand(bs, 4, device="cuda")
        x[:, :2] = x[:, :2] * 2 - 1
        t = torch.rand(bs, taps, device="cuda") + 1e-3
        return x, t / t.sum(1, keepdim=True)

    lens = pkg.PSFNet(kernel_size=ks, device="cuda")
    lens.train_psfnet(iters=iters, bs=bs, lr=lr0, evaluate_every=4, data=data, save=False)
    opt = torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=lr0)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=iters)
    ref = []
    for _ in range(iters + 1):
        ref.append(opt.param_groups[0]["lr"])
        opt.step()
        sched.step()
    assert len(lrs) == iters + 1
    for i, (a, b) in enumerate(zip(lrs, ref)):
        assert abs(a - b) <= 1e-12 * max(abs(b), 1e-12 * lr0), (i, a, b)
    for taps in ((ks - 2) ** 2, (ks + 2) ** 2):
        lrs.clear()
        with pytest.raises(ValueError, match="kernel_size"):
            lens.train_psfnet(iters=iters, bs=bs, lr=lr0, data=lambda bs, spp: data(bs, spp, taps), save=False)
        assert lrs == []
