"""PSFNet / ThinLens host wrappers (mirror of the reference's deeplens/psfnet.py:14-76, 375-454, 489-570).

Same constructor, attributes and method signatures as the reference so that 0_warm_up.py,
dff/factory.get_lens and the 2_aber_aware_dff_* training loops run unchanged; ``render`` and
``pred`` dispatch through the C ABI (include/aadff.h) into the sm_100a kernels.

The module has a name of its own (it is re-exported as ``deeplens.psfnet`` by the shadow package next to
it) so that it can never be confused with a reference ``deeplens`` that is already imported; and every
method below reads the lens through duck typing only (``kernel_size``, ``psfnet.net``, ``d_min``,
``d_max``), so that ``aadff_install.install()`` can graft the same functions onto the reference's own
``PSFNet`` / ``ThinLens`` classes.

Differences from the reference, all deliberate (DESIGN.md):
  * the ray-traced lens model behind ``Lensgroup`` is out of scope: ``filename`` is recorded, not
    parsed, and ``analysis()`` only logs;
  * ``load_net`` passes ``map_location`` (the reference's bare torch.load fails on a box whose
    device differs from the one the checkpoint was saved on);
  * an input of unsupported rank raises instead of silently returning None;
  * ``render_stack`` renders all focal slices of a batch in one launch, writing [B,C,S,H,W]
    (AiFNet layout) or [B,S,C,H,W] (DFVNet layout) directly.
"""
import logging
import os

import numpy as np
import torch
import torch.nn as nn

import aadff_native as _nat
from aadff_arch import MLP, initialize_weights
from aadff_render import local_psf_render  # noqa: F401  (the reference's psfnet module exports it too)

DMIN = 200     # [mm]
DMAX = 20000   # [mm]


def _device_index(device) -> int:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"aadff-b200 runs on CUDA (sm_100a) only, got device '{device}'; there is no CPU path")
    return dev.index if dev.index is not None else torch.cuda.current_device()


def _linear_layers(net):
    """The nn.Linear modules of an MLP container (ours or the reference's: both keep them in ``.net``)."""
    return [m for m in net.net if isinstance(m, nn.Linear)]


class PSFNet(nn.Module):
    def __init__(self, filename=None, model_name='mlp', kernel_size=11, sensor_res=(512, 512), device='cuda',
                 mode=None):
        super().__init__()
        self.filename = filename
        self.sensor_res = sensor_res
        self.device = device
        self.in_features = 4
        self.kernel_size = kernel_size
        self.model_name = model_name
        self.mode = mode or os.environ.get("AADFF_MODE", "parity")
        self.d_max = -DMAX
        self.d_min = -DMIN
        self.foc_d_arr = np.array([-500, -600, -700, -800, -900, -1000, -1250, -1500, -1750, -2000,
                                   -2500, -3000, -4000, -5000, -6000, -8000, -10000, -12000, -15000, -20000])
        self.foc_z_arr = (self.foc_d_arr - self.d_min) / (self.d_max - self.d_min)
        self._native = None
        self._native_sig = None
        self.init_net()

    # ------------------------------------------------------------------ network
    def init_net(self):
        ks = self.kernel_size
        if self.model_name == 'mlp':
            self.psfnet = MLP(in_features=4, out_features=ks ** 2, hidden_features=256, hidden_layers=8)
        elif self.model_name in ('mlpconv', 'siren'):
            raise NotImplementedError(f"'{self.model_name}' is not on the focal-stack synthesis path")
        else:
            raise Exception('Unsupported PSF network architecture.')
        self.psfnet.apply(initialize_weights)
        self.psfnet.to(self.device)
        self.psfnet._evaluator = self._mlp_eval
        self._native = None

    def load_net(self, net_path):
        """Load pretrained network (state_dict with keys net.{0,2,...}.{weight,bias})."""
        self.psfnet.load_state_dict(torch.load(net_path, map_location=self.device))
        self._native = None

    def _signature(self):
        return tuple((p.data_ptr(), p._version) for p in self.psfnet.parameters())

    def native(self) -> "_nat.NativePSFNet":
        """The pre-packed device copy of the weights; rebuilt when the parameters change
        (in-place edits through ``.data`` do not bump ``_version``: call ``refresh()`` after those)."""
        sig = PSFNet._signature(self)
        if getattr(self, "_native", None) is None or sig != getattr(self, "_native_sig", None):
            layers = _linear_layers(self.psfnet)
            idx = _device_index(layers[0].weight.device)
            ws = [l.weight.detach().float().cpu().numpy() for l in layers]
            bs = [l.bias.detach().float().cpu().numpy() for l in layers]
            if getattr(self, "_native", None) is not None:
                self._native.close()
            self._native = _nat.NativePSFNet(ws, bs, self.kernel_size, idx)
            self._native_sig = sig
        return self._native

    def refresh(self):
        """Drop the packed device copy of the weights (it is rebuilt on the next call)."""
        self._native = None

    def analysis(self, *args, **kwargs):
        logging.info("PSFNet.analysis(): lens plots/ray tracing are outside the synthesis path; skipped.")

    # ------------------------------------------------------------------ inference
    def _mlp_eval(self, inp, mode="fp32"):
        nat = PSFNet.native(self)
        kk = self.kernel_size ** 2
        flat = inp.detach().reshape(-1, 4).to(f"cuda:{nat.device_index}", torch.float32).contiguous()
        out = torch.empty(flat.shape[0], kk, device=flat.device, dtype=torch.float32)
        if flat.shape[0] == 0:
            return out.reshape(*inp.shape[:-1], kk)
        with torch.cuda.device(flat.device):
            _nat.check(_nat.lib.aadff_psfnet_pred_tc_f32(nat.handle, flat.data_ptr(), out.data_ptr(), flat.shape[0],
                                                         _nat.MODES[mode], torch.cuda.current_stream().cuda_stream))
        return out.reshape(*inp.shape[:-1], kk)

    @torch.no_grad()
    def pred(self, inp, mode=None):
        """inp [...,4] = (x, y, z, foc_z) -> psf [..., ks, ks].  mode=None: fp32 CUDA-core kernel (operation for
        operation with the reference); 'parity' / 'econ8' / 'econ' / 'mixed' / 'fast': the tensor-core kernel (~30x faster)."""
        psf = PSFNet._mlp_eval(self, inp, "fp32" if mode is None else mode)
        return psf.reshape(*psf.shape[:-1], self.kernel_size, self.kernel_size)

    def _launch(self, img, depth, foc, out_ptr, strides, mode, rows=None):
        nat = PSFNet.native(self)
        N, C, H, W = img.shape
        S = foc.shape[1]
        if N * C * S * H * W == 0:      # empty batch: nothing to launch (data_ptr() of an empty tensor is NULL)
            return
        arr = (_nat.ctypes.c_int64 * 5)(*strides)
        m = _nat.MODES[mode or getattr(self, "mode", None) or os.environ.get("AADFF_MODE", "parity")]
        with torch.cuda.device(img.device):
            st = torch.cuda.current_stream().cuda_stream
            if rows is None:
                _nat.check(_nat.lib.aadff_render_stack_f32(
                    nat.handle, img.data_ptr(), depth.data_ptr(), foc.data_ptr(), out_ptr, arr,
                    N, C, S, H, W, float(self.d_min), float(self.d_max), m, st))
            else:
                _nat.check(_nat.lib.aadff_render_stack_rows_f32(
                    nat.handle, img.data_ptr(), depth.data_ptr(), foc.data_ptr(), out_ptr, arr,
                    N, C, S, H, W, float(self.d_min), float(self.d_max), m, int(rows[0]), int(rows[1]), st))

    def _prep(self, img, depth):
        nat = PSFNet.native(self)
        dev = torch.device(f"cuda:{nat.device_index}")
        img = img.detach().to(dev, torch.float32).contiguous()
        N, C, H, W = img.shape
        depth = depth.detach().to(dev, torch.float32).reshape(N, H, W).contiguous()
        return img, depth, dev

    @torch.no_grad()
    def render(self, img, depth, foc_dist, mode=None):
        """Render image with aif image and depth map.

        img [N,C,H,W], depth [N,1,H,W] (mm, negative), foc_dist [N] (mm, negative) -> [N,C,H,W];
        or img [C,H,W], depth [H,W], scalar foc_dist -> [1,C,H,W].
        """
        if img.dim() == 3:
            img = img.unsqueeze(0)
            depth = depth.reshape(1, *depth.shape[-2:])
            foc_dist = torch.as_tensor([float(foc_dist)], dtype=torch.float32)
        elif img.dim() != 4:
            raise ValueError(f"render expects a [N,C,H,W] or [C,H,W] image, got shape {tuple(img.shape)}")
        img, depth, dev = PSFNet._prep(self, img, depth)
        N, C, H, W = img.shape
        foc = torch.as_tensor(foc_dist).detach().to(dev, torch.float32).reshape(N, 1).contiguous()
        out = torch.empty_like(img)
        PSFNet._launch(self, img, depth, foc, out.data_ptr(), (C * H * W, H * W, 0, W, 1), mode)
        return out

    @torch.no_grad()
    def render_stack(self, img, depth, foc_dists, layout="BCSHW", mode=None):
        """All S focal slices in one launch: foc_dists [N,S] (mm, negative) -> [N,C,S,H,W]
        (== torch.stack([render(img, depth, foc_dists[:, s]) for s], dim=2)), or [N,S,C,H,W]."""
        if img.dim() != 4:
            raise ValueError("render_stack expects a [N,C,H,W] image")
        img, depth, dev = PSFNet._prep(self, img, depth)
        N, C, H, W = img.shape
        foc = foc_dists.detach().to(dev, torch.float32).reshape(N, -1).contiguous()
        S = foc.shape[1]
        if layout == "BCSHW":
            out = torch.empty(N, C, S, H, W, device=dev, dtype=torch.float32)
            strides = (C * S * H * W, S * H * W, H * W, W, 1)
        elif layout == "BSCHW":
            out = torch.empty(N, S, C, H, W, device=dev, dtype=torch.float32)
            strides = (S * C * H * W, H * W, C * H * W, W, 1)
        else:
            raise ValueError("layout must be 'BCSHW' or 'BSCHW'")
        PSFNet._launch(self, img, depth, foc, out.data_ptr(), strides, mode)
        return out

    @torch.no_grad()
    def render_stack_rows(self, img, depth, foc_dists, tile_row_begin, tile_row_end, mode=None):
        """One contiguous run of tile rows (8 image rows each) of the flattened (image, slice, row) stack -- the
        unit of the multi-GPU partition (sharding.py).  Returns the rows in [flat_rows, C, W] layout, where
        flat row = (n*S + s)*H + h; bit-identical to the same rows of ``render_stack``."""
        img, depth, dev = PSFNet._prep(self, img, depth)
        N, C, H, W = img.shape
        foc = foc_dists.detach().to(dev, torch.float32).reshape(N, -1).contiguous()
        S = foc.shape[1]
        th = _nat.lib.aadff_tile_row_height()
        ty = -(-H // th)
        fr = [(R // ty) * H + min((R % ty) * th, H) for R in (int(tile_row_begin), int(tile_row_end))]
        out = torch.empty(fr[1] - fr[0], C, W, device=dev, dtype=torch.float32)
        # element strides of a virtual [N,S,H,C,W] tensor whose flat row fr[0] sits at out[0]
        strides = (S * H * C * W, W, H * C * W, C * W, 1)
        if out.numel():
            PSFNet._launch(self, img, depth, foc, out.data_ptr() - fr[0] * C * W * 4, strides, mode,
                           rows=(tile_row_begin, tile_row_end))
        return out

    @torch.no_grad()
    def simulate_focal_stack(self, aif, depth_m, n_stack, layout="BCSHW", mode=None, check=False):
        """The focal-stack simulation block of the training scripts (2_aber_aware_dff_aif.py:101-114) in one
        call with no host synchronisation: focus distances from `select_focus_dist(depth_m, n_stack, 'linear')`
        (metres, device-side reductions), then ONE fused launch for all slices.
        aif [B,C,H,W] in [0,1], depth_m [B,1,H,W] metres (0 = invalid) -> (stack [B,C,S,H,W], focus_dists [B,S] m).

        An image without a single valid depth gets NaN focus distances (the reference raises on it and its
        training loop skips such batches, 2_aber_aware_dff_aif.py:103-105); its slices are then meaningless.
        ``check=True`` raises for such a batch (this costs a device->host synchronisation); without it test
        ``torch.isnan(focus_dists).any(1)`` whenever convenient."""
        from aadff_focus import select_focus_dist
        focus_dists = select_focus_dist(depth_m, n_stack, mode='linear')
        if check and bool(torch.isnan(focus_dists).any()):
            raise ValueError("simulate_focal_stack: an image of the batch has no valid (> 0) depth")
        stack = PSFNet.render_stack(self, aif, -depth_m * 1e3, -focus_dists * 1e3, layout=layout, mode=mode)
        return stack, focus_dists

    # ------------------------------------------------------------------ fitting (SURVEY.md 8f, row f3)
    def train_psfnet(self, iters=10000, bs=128, lr=1e-4, spp=2048, evaluate_every=1000, result_dir='./results/temp',
                     data=None, save=True):
        """Fit the PSF representation network (mirror of deeplens/psfnet.py:79-132).  The optimisation --
        psfnet(inp), nn.MSELoss, backward, AdamW with CosineAnnealingLR(T_max=iters) -- runs on the device as one
        CUDA-graph replay per iteration (csrc/train_kernels.cuh).  The training targets are ray-traced PSFs
        (get_training_data, psfnet.py:135-170) and stay with the reference: ``data(bs=, spp=)`` must return
        ``(inp [bs,4], psf [bs,ks*ks])``; by default ``self.get_training_data`` is used, which exists when these
        methods are grafted onto the reference's PSFNet (aadff_install.install()).  Returns the list of losses
        recorded every ``evaluate_every`` iterations (the reference plots PSFs there)."""
        import math
        data = data or getattr(self, "get_training_data", None)
        if data is None:
            raise NotImplementedError("train_psfnet needs `data`: ray-traced training targets come from the reference "
                                      "(PSFNet.get_training_data); this build does not contain the ray tracer")
        layers = _linear_layers(self.psfnet)
        idx = _device_index(layers[0].weight.device)
        dev = torch.device(f"cuda:{idx}")
        trainer = _nat.NativeTrainer([l.weight.detach().float().cpu().numpy() for l in layers],
                                     [l.bias.detach().float().cpu().numpy() for l in layers], bs, idx)
        loss_dev = torch.zeros(1, device=dev)
        history = []
        try:
            with torch.cuda.device(dev):
                for i in range(iters + 1):
                    inp, psf = data(bs=bs, spp=spp)
                    inp = inp.detach().to(dev, torch.float32).reshape(bs, 4).contiguous()
                    psf = psf.detach().to(dev, torch.float32).reshape(bs, -1).contiguous()
                    if psf.shape[-1] != self.kernel_size ** 2:      # the step reads bs * ks^2 target values
                        raise ValueError(f"train_psfnet: data returned PSFs of {psf.shape[-1]} taps per probe; "
                                         f"kernel_size {self.kernel_size} needs {self.kernel_size ** 2}")
                    lr_i = 0.5 * lr * (1.0 + math.cos(math.pi * i / iters)) if iters > 0 else lr   # CosineAnnealingLR, eta_min 0
                    _nat.check(_nat.lib.aadff_trainer_step(trainer.handle, inp.data_ptr(), psf.data_ptr(), lr_i,
                                                           loss_dev.data_ptr(), torch.cuda.current_stream().cuda_stream))
                    if (i + 1) % evaluate_every == 0:
                        history.append((i + 1, float(loss_dev)))
                ws, bs_ = trainer.read(0, torch.cuda.current_stream().cuda_stream)
            with torch.no_grad():
                for l, w, b in zip(layers, ws, bs_):
                    l.weight.copy_(torch.from_numpy(w))
                    l.bias.copy_(torch.from_numpy(b))
            self._native = None
        finally:
            trainer.close()
        if save:
            os.makedirs(result_dir, exist_ok=True)
            torch.save(self.psfnet.state_dict(), f'{result_dir}/PSFNet_{getattr(self, "model_name", "mlp")}.pkl')
        return history

    # ------------------------------------------------------------------ utils
    def depth2z(self, depth):
        z = (depth - self.d_min) / (self.d_max - self.d_min)
        return torch.clamp(z, min=0, max=1)

    def z2depth(self, z):
        return z * (self.d_max - self.d_min) + self.d_min


# names install() grafts onto the reference's PSFNet (everything render/pred need, nothing the ray tracer owns)
PSFNET_GRAFT = ("native", "refresh", "_mlp_eval", "pred", "_launch", "_prep", "render", "render_stack",
                "render_stack_rows", "simulate_focal_stack", "train_psfnet")


class ThinLens(nn.Module):
    """Thin-lens baseline (mirror of deeplens/psfnet.py:489-570): clipped-Gaussian PSF from the
    circle of confusion, rendered with the same per-pixel gather kernel."""

    def __init__(self, foc_len, fnum, kernel_size, sensor_size, sensor_res, device='cpu'):
        super().__init__()
        self.d_max = DMAX
        self.d_min = DMIN
        self.kernel_size = kernel_size
        self.foc_len = foc_len
        self.fnum = fnum
        self.sensor_size = sensor_size
        self.sensor_res = sensor_res
        self.ps = self.sensor_size[0] / self.sensor_res[0]
        self.device = device

    def to(self, device):
        self.device = device
        return self

    def coc(self, depth, foc_dist):
        if (depth < 0).any():
            depth = -depth
            foc_dist = -foc_dist
        depth = torch.clamp(depth, self.d_min, self.d_max)
        coc = self.foc_len / self.fnum * torch.abs(depth - foc_dist) / depth * self.foc_len / (foc_dist - self.foc_len)
        return torch.clamp(coc / self.ps, min=0.1)

    @torch.no_grad()
    def render(self, img, depth, foc_dist):
        """img [N,C,H,W], depth [N,1,H,W], foc_dist [N] -> [N,C,H,W] (fused CUDA kernel: coc -> clipped
        Gaussian PSF -> gather; the PSF tensor of the reference is never materialised).  The reference's
        data-dependent sign convention (`if (depth < 0).any()`, psfnet.py:504) is decided on the device:
        no host synchronisation, CUDA-graph capturable."""
        if img.dim() != 4:
            raise ValueError("ThinLens.render expects a [N,C,H,W] image")
        if not img.is_cuda:
            raise RuntimeError("ThinLens.render: CUDA tensors required (no CPU fallback in this build)")
        N, C, H, W = img.shape
        img = img.detach().contiguous().float()
        dep = depth.detach().to(img.device, torch.float32).reshape(N, H, W).contiguous()
        foc = torch.as_tensor(foc_dist).detach().to(img.device, torch.float32).reshape(N).contiguous()
        out = torch.empty_like(img)
        if out.numel() == 0:
            return out
        flag = torch.empty(1, dtype=torch.uint8, device=img.device)
        with torch.cuda.device(img.device):
            st = torch.cuda.current_stream().cuda_stream
            _nat.check(_nat.lib.aadff_any_negative_f32(dep.data_ptr(), dep.numel(), flag.data_ptr(), st))
            _nat.check(_nat.lib.aadff_thinlens_render_f32(
                img.data_ptr(), dep.data_ptr(), foc.data_ptr(), out.data_ptr(), N, C, H, W, int(self.kernel_size),
                float(self.foc_len), float(self.fnum), float(self.ps), float(self.d_min), float(self.d_max), 0,
                flag.data_ptr(), st))
        return out

    @torch.no_grad()
    def psf(self, depth, foc_dist):
        """The per-pixel thin-lens PSFs [N,H,W,ks,ks] as the reference builds them (psfnet.py:549-566); kept
        for inspection / for callers that want to feed local_psf_render themselves."""
        ks = self.kernel_size
        device = depth.device
        N, _, H, W = depth.shape
        foc = foc_dist.to(device).view(N, 1, 1, 1).expand(N, 1, H, W)
        lin = torch.linspace(-ks / 2 + 1 / 2, ks / 2 - 1 / 2, ks)
        x, y = torch.meshgrid(lin, torch.linspace(ks / 2 - 1 / 2, -ks / 2 + 1 / 2, ks), indexing='xy')
        x, y = x.to(device), y.to(device)
        radius = (ThinLens.coc(self, depth, foc).squeeze(1) / 2)[..., None, None]
        r2 = x ** 2 + y ** 2
        psf = torch.exp(-r2 / 2 / radius ** 2) / (2 * np.pi * radius ** 2)
        psf = psf * (r2 < radius ** 2)
        return psf / psf.sum((-1, -2), keepdim=True)


THINLENS_GRAFT = ("render",)
