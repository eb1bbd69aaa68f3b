"""ctypes binding of libaadff.so (C ABI in include/aadff.h) + the in-tree build recipe.

This is the only way the Python host layer reaches the GPU: there is no PyTorch-eager or CPU
fallback behind it.  If the shared library is missing and cannot be built, importing this
module raises -- loudly -- instead of degrading.
"""
from __future__ import annotations

import ctypes
import os
import re
import shutil
import subprocess

import torch

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


# C types of include/aadff.h's scalar parameters and return values.  Every pointer or array parameter is c_void_p, which
# takes data_ptr() ints, None, ctypes arrays and byref(); a type outside this map fails the import instead of falling
# back to ctypes' default (a 32-bit int).
_CTYPES = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "float": ctypes.c_float, "double": ctypes.c_double,
           "const char*": ctypes.c_char_p, "aadff_psfnet_t": ctypes.c_void_p, "aadff_trainer_t": ctypes.c_void_p}


def _ctype(decl):
    t = " ".join(decl.replace("*", " * ").split()).replace(" *", "*")
    if t not in _CTYPES:
        raise TypeError(f"include/aadff.h: no ctypes mapping for C type '{t}'")
    return _CTYPES[t]


def _prototypes(text=None):
    """{name: (restype, argtypes)} of each prototype `ret aadff_name(params);` in include/aadff.h (or in `text`)."""
    if text is None:
        with open(HEADER) as f:
            text = f.read()
    text = re.sub(r"^\s*#.*$", "", re.sub(r"/\*.*?\*/", " ", text, flags=re.S), flags=re.M)
    protos = {}
    for ret, name, params in re.findall(r"(\w[\w\s*]*?)\s*\b(aadff_\w+)\s*\(([^()]*)\)\s*;", text):
        params = [p for p in params.split(",") if p.strip() not in ("", "void")]
        protos[name] = (_ctype(ret), [ctypes.c_void_p if "*" in p or "[" in p else _ctype(p.rsplit(None, 1)[0])
                                      for p in params])
    return protos


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        build()
    lib = ctypes.CDLL(LIB_PATH)
    protos = _prototypes()
    if any(not hasattr(lib, name) for name in protos):     # stale binary: rebuild once
        import _ctypes
        _ctypes.dlclose(lib._handle)
        build(force=True)
        lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in protos.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
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
    return sorted(_prototypes())


def call(fn_name: str, *args, device: torch.device) -> None:
    """lib.<fn_name>(*args, stream) on `device` with its current stream; raises AadffError on a non-zero return."""
    # by index: resolving the torch.device in both torch calls would cost more host time than the rest of this helper
    idx = device.index
    with torch.cuda.device(idx):
        check(getattr(lib, fn_name)(*args, torch.cuda.current_stream(idx).cuda_stream))


def workspace(nbytes: int, device) -> torch.Tensor:
    """The device workspace an aadff_*_work_bytes query asked for; a negative size is the query's refusal and raises.
    The caching allocator hands out blocks aligned to at least 256 bytes, as the render backward requires."""
    if nbytes < 0:
        check(nbytes)
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def f32_ptrs(seq):
    """Host array of float* for the C ABI's per-layer pointer arrays: one per tensor or numpy array, NULL for None.
    The caller keeps the arrays alive for the duration of the call."""
    return (ctypes.c_void_p * len(seq))(*[None if t is None else t.data_ptr() if torch.is_tensor(t) else t.ctypes.data
                                          for t in seq])


class NativePSFNet:
    """Owns an aadff_psfnet_t: the pre-packed network on one device."""

    def __init__(self, weights, biases, ks: int, device_index: int):
        import numpy as np
        ws = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        bs = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        n = len(ws)
        dims = [ws[0].shape[1]] + [w.shape[0] for w in ws]
        self.handle = ctypes.c_void_p()
        self.ks = ks
        self.n_layers = n
        self.device_index = device_index
        check(lib.aadff_psfnet_create(f32_ptrs(ws), f32_ptrs(bs), (ctypes.c_int * (n + 1))(*dims), n, ks, device_index,
                                      ctypes.byref(self.handle)))

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
        ws = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        bs = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        n = len(ws)
        if n < 1 or len(bs) != n:
            raise ValueError(f"NativeTrainer: need as many biases as weights (>= 1), got {n} and {len(bs)}")
        self.dims = [ws[0].shape[-1]] + [w.shape[0] for w in ws]
        for l, (w, b) in enumerate(zip(ws, bs)):
            # the library copies dims[l+1] * dims[l] weights and dims[l+1] biases of each layer from these buffers
            if w.shape != (self.dims[l + 1], self.dims[l]) or b.shape != (self.dims[l + 1],):
                raise ValueError(f"NativeTrainer: layer {l} has weight {tuple(w.shape)} and bias {tuple(b.shape)}; "
                                 f"expected ({self.dims[l + 1]}, {self.dims[l]}) and ({self.dims[l + 1]},)")
        self.batch, self.device_index = int(batch), device_index
        self.handle = ctypes.c_void_p()
        check(lib.aadff_trainer_create(f32_ptrs(ws), f32_ptrs(bs), (ctypes.c_int * (n + 1))(*self.dims), n, self.batch,
                                       betas[0], betas[1], eps, weight_decay, device_index, ctypes.byref(self.handle)))

    def read(self, which: int, stream=None):
        """which 0: parameters, 1: gradients of the last step -> (weights, biases) as numpy arrays."""
        import numpy as np
        n = len(self.dims) - 1
        ws = [np.empty((self.dims[l + 1], self.dims[l]), np.float32) for l in range(n)]
        bs = [np.empty((self.dims[l + 1],), np.float32) for l in range(n)]
        check(lib.aadff_trainer_read(self.handle, which, f32_ptrs(ws), f32_ptrs(bs), stream))
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
