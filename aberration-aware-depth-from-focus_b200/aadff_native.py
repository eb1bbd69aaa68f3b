"""ctypes binding of libaadff.so (C ABI in include/aadff.h) + the in-tree build recipe.

This is the only way the Python host layer reaches the GPU: there is no PyTorch-eager or CPU
fallback behind it.  If the shared library is missing and cannot be built, importing this
module raises -- loudly -- instead of degrading.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("AADFF_LIB_PATH") or os.path.join(_HERE, "libaadff.so")   # override: experiments only
HEADER = os.path.join(_REPO, "include", "aadff.h")

MODE_PARITY, MODE_FAST, MODE_FP32, MODE_MIXED, MODE_ECON, MODE_ECON8 = 0, 1, 2, 3, 4, 5
MODES = {"parity": MODE_PARITY, "fast": MODE_FAST, "fp32": MODE_FP32, "mixed": MODE_MIXED, "econ": MODE_ECON,
         "econ8": MODE_ECON8}

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + [HEADER]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/aadff_api.cu -> libaadff.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if not force and os.path.exists(LIB_PATH):
        newest = max(os.path.getmtime(s) for s in _sources())
        if os.path.getmtime(LIB_PATH) >= newest:
            return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("libaadff.so is not built and nvcc was not found; cannot build the CUDA extension")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH, os.path.join(CSRC, "aadff_api.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


def _header_symbols():
    import re
    with open(HEADER) as f:
        return sorted(set(re.findall(r"\b(aadff_[a-z0-9_]+)\s*\(", f.read())))


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        build()
    lib = ctypes.CDLL(LIB_PATH)
    if any(not hasattr(lib, name) for name in _header_symbols()):     # stale binary: rebuild once
        import _ctypes
        _ctypes.dlclose(lib._handle)
        build(force=True)
        lib = ctypes.CDLL(LIB_PATH)
    c_f32p = ctypes.POINTER(ctypes.c_float)
    lib.aadff_version.restype = ctypes.c_int
    lib.aadff_last_error.restype = ctypes.c_char_p
    lib.aadff_launch_count.restype = ctypes.c_int64
    lib.aadff_psfnet_create.argtypes = [ctypes.POINTER(c_f32p), ctypes.POINTER(c_f32p),
                                        ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.POINTER(ctypes.c_void_p)]
    lib.aadff_psfnet_destroy.argtypes = [ctypes.c_void_p]
    lib.aadff_render_stack_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)] + [ctypes.c_int] * 5 + \
                                          [ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_void_p]
    lib.aadff_render_stack_rows_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)] + [ctypes.c_int] * 5 + \
                                               [ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_int64,
                                                ctypes.c_int64, ctypes.c_void_p]
    lib.aadff_tile_row_height.restype = ctypes.c_int
    lib.aadff_econ_first_group.restype = ctypes.c_int
    lib.aadff_render_psf_map_f32.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + \
                                            [ctypes.POINTER(ctypes.c_int)] * 2 + [ctypes.c_void_p]
    lib.aadff_trainer_create.argtypes = [ctypes.POINTER(c_f32p), ctypes.POINTER(c_f32p), ctypes.POINTER(ctypes.c_int),
                                         ctypes.c_int, ctypes.c_int] + [ctypes.c_float] * 4 + \
                                        [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
    lib.aadff_trainer_step.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p,
                                       ctypes.c_void_p]
    lib.aadff_trainer_read.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(c_f32p), ctypes.POINTER(c_f32p),
                                       ctypes.c_void_p]
    lib.aadff_trainer_destroy.argtypes = [ctypes.c_void_p]
    lib.aadff_preprocess_rgbd_u8.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 5 + [ctypes.c_float, ctypes.c_int,
                                             ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.aadff_prepare_planes_u8.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3 + [ctypes.c_float, ctypes.c_void_p,
                                            ctypes.c_void_p, ctypes.c_void_p]
    lib.aadff_spline_affine_f32.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_void_p, ctypes.c_int,
                                            ctypes.c_void_p]
    lib.aadff_resize_planes_f32.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_int, ctypes.c_void_p]
    lib.aadff_any_negative_f32.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
    lib.aadff_render_stack_host_f32.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int] * 5 + \
                                               [ctypes.c_float, ctypes.c_float, ctypes.c_int]
    lib.aadff_psfnet_pred_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                          ctypes.c_void_p]
    lib.aadff_psfnet_pred_tc_f32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                             ctypes.c_int, ctypes.c_void_p]
    lib.aadff_local_psf_render_f32.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    lib.aadff_local_psf_render_backward_f32.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    lib.aadff_render_psf_map_backward_work_bytes.argtypes = [ctypes.c_int] * 6 + [ctypes.POINTER(ctypes.c_int)] * 2
    lib.aadff_render_psf_map_backward_work_bytes.restype = ctypes.c_int64
    lib.aadff_render_psf_map_backward_f32.argtypes = [ctypes.c_void_p] * 6 + [ctypes.c_int64] + [ctypes.c_int] * 6 + \
                                                     [ctypes.POINTER(ctypes.c_int)] * 2 + [ctypes.c_void_p]
    lib.aadff_debug_umma_gemm.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3
    lib.aadff_thinlens_render_f32.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int] * 5 + [ctypes.c_float] * 5 + \
                                             [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.aadff_debug_set_desc_swap.argtypes = [ctypes.c_int]
    lib.aadff_debug_econ_round.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                           ctypes.c_void_p]
    lib.aadff_debug_econ_round.restype = ctypes.c_int
    lib.aadff_select_focus_f32.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p,
                                           ctypes.c_void_p]
    for fn in ("aadff_psfnet_create", "aadff_psfnet_destroy", "aadff_render_stack_f32", "aadff_render_stack_rows_f32",
               "aadff_any_negative_f32", "aadff_render_psf_map_f32", "aadff_preprocess_rgbd_u8", "aadff_prepare_planes_u8",
               "aadff_spline_affine_f32", "aadff_resize_planes_f32", "aadff_trainer_create", "aadff_trainer_step",
               "aadff_trainer_read", "aadff_trainer_destroy",
               "aadff_render_stack_host_f32", "aadff_psfnet_pred_f32", "aadff_psfnet_pred_tc_f32", "aadff_local_psf_render_f32",
               "aadff_local_psf_render_backward_f32", "aadff_render_psf_map_backward_f32", "aadff_thinlens_render_f32", "aadff_select_focus_f32",
               "aadff_debug_umma_gemm", "aadff_debug_set_desc_swap"):
        getattr(lib, fn).restype = ctypes.c_int
    return lib


lib = _load()


class AadffError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        raise AadffError(f"libaadff error {rc}: {lib.aadff_last_error().decode()}")


def econ_first_group() -> int:
    """First tensor-core group (0 = L1) that AADFF_MODE_ECON runs with two MMA terms instead of three."""
    return int(lib.aadff_econ_first_group())


def exported_symbols():
    """Names declared in include/aadff.h (used by the CPU test that checks the library exports them)."""
    return _header_symbols()


class NativePSFNet:
    """Owns an aadff_psfnet_t: the pre-packed network on one device."""

    def __init__(self, weights, biases, ks: int, device_index: int):
        import numpy as np
        self._np = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        self._nb = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        n = len(self._np)
        dims = [self._np[0].shape[1]] + [w.shape[0] for w in self._np]
        c_f32p = ctypes.POINTER(ctypes.c_float)
        wp = (c_f32p * n)(*[w.ctypes.data_as(c_f32p) for w in self._np])
        bp = (c_f32p * n)(*[b.ctypes.data_as(c_f32p) for b in self._nb])
        dm = (ctypes.c_int * (n + 1))(*dims)
        self.handle = ctypes.c_void_p()
        self.ks = ks
        self.device_index = device_index
        check(lib.aadff_psfnet_create(wp, bp, dm, n, ks, device_index, ctypes.byref(self.handle)))
        self._np = self._nb = None

    def close(self):
        if getattr(self, "handle", None):
            lib.aadff_psfnet_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class NativeTrainer:
    """Owns an aadff_trainer_t: device parameters + AdamW state + one batch of activations (include/aadff.h)."""

    def __init__(self, weights, biases, batch: int, device_index: int, betas=(0.9, 0.999), eps=1e-8,
                 weight_decay=1e-2):
        import numpy as np
        self._np = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        self._nb = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        n = len(self._np)
        if n < 1 or len(self._nb) != n:
            raise ValueError(f"NativeTrainer: need as many biases as weights (>= 1), got {n} and {len(self._nb)}")
        self.dims = [self._np[0].shape[-1]] + [w.shape[0] for w in self._np]
        for l, (w, b) in enumerate(zip(self._np, self._nb)):
            # the library copies dims[l+1] * dims[l] weights and dims[l+1] biases of each layer from these buffers
            if w.shape != (self.dims[l + 1], self.dims[l]) or b.shape != (self.dims[l + 1],):
                raise ValueError(f"NativeTrainer: layer {l} has weight {tuple(w.shape)} and bias {tuple(b.shape)}; "
                                 f"expected ({self.dims[l + 1]}, {self.dims[l]}) and ({self.dims[l + 1]},)")
        self.batch, self.device_index = int(batch), device_index
        c_f32p = ctypes.POINTER(ctypes.c_float)
        wp = (c_f32p * n)(*[w.ctypes.data_as(c_f32p) for w in self._np])
        bp = (c_f32p * n)(*[b.ctypes.data_as(c_f32p) for b in self._nb])
        dm = (ctypes.c_int * (n + 1))(*self.dims)
        self.handle = ctypes.c_void_p()
        check(lib.aadff_trainer_create(wp, bp, dm, n, self.batch, betas[0], betas[1], eps, weight_decay, device_index,
                                       ctypes.byref(self.handle)))

    def read(self, which: int, stream=None):
        """which 0: parameters, 1: gradients of the last step -> (weights, biases) as numpy arrays."""
        import numpy as np
        n = len(self.dims) - 1
        ws = [np.empty((self.dims[l + 1], self.dims[l]), np.float32) for l in range(n)]
        bs = [np.empty((self.dims[l + 1],), np.float32) for l in range(n)]
        c_f32p = ctypes.POINTER(ctypes.c_float)
        wp = (c_f32p * n)(*[w.ctypes.data_as(c_f32p) for w in ws])
        bp = (c_f32p * n)(*[b.ctypes.data_as(c_f32p) for b in bs])
        check(lib.aadff_trainer_read(self.handle, which, wp, bp, stream))
        return ws, bs

    def close(self):
        if getattr(self, "handle", None):
            lib.aadff_trainer_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
