"""ctypes binding of the C ABI declared in include/pcd_b200.h.

There is NO CPU fallback: if the shared library is missing, or a compute entry point is
called without a CUDA device, this module raises.  torch is used only for device memory,
streams and torch.distributed plumbing.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCD_LIB_PATH") or os.path.join(_HERE, "libpcd_b200.so")   # PCD_LIB_PATH: A/B-compare two builds on one box
CSRC = os.path.join(_HERE, "csrc")
SOURCES = ["api.cu", "api_latent.cu", "gemm_tc.cu", "gemm_simt.cu", "chamfer.cu", "emd.cu", "emd_exact.cu", "latent.cu", "latent_mk.cu", "chain_tc.cu", "folding.cu", "api_vae3d.cu", "vae3d.cu", "conv3d_tc.cu", "api_pointvae.cu"]

PRECISION = {"bf16": 0, "fp32": 1, "bf16x3": 2, "f16": 3, "f16mix": 4}
SCHED_ROW = 8


class PcdError(RuntimeError):
    pass


class _NamedTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int32), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 4)]


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
OBJ_DIR = os.path.join(_HERE, "build")      # git-ignored object cache: one .o per source, compiled in parallel


def nvcc_command(out_path: str = LIB_PATH):
    """The single-command form of the build (what a maintainer would type by hand)."""
    return ["nvcc"] + NVCC_FLAGS + ["-shared", "-o", out_path] + [os.path.join(CSRC, s) for s in SOURCES]


def build(force: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU): every source to its own object
    (only the stale ones, all of them in parallel), then one link."""
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if not f.endswith(".cu")] + \
              [os.path.join(_HERE, "..", "include", "pcd_b200.h")]
    hdr_time = max(os.path.getmtime(h) for h in headers)
    src_time = max(os.path.getmtime(os.path.join(CSRC, f)) for f in SOURCES)
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(hdr_time, src_time):
        return LIB_PATH         # e.g. on the GPU box: the prebuilt library travels, the object cache does not
    os.makedirs(OBJ_DIR, exist_ok=True)
    jobs, objs = [], []
    for src in SOURCES:
        sp, op = os.path.join(CSRC, src), os.path.join(OBJ_DIR, src[:-3] + ".o")
        objs.append(op)
        if force or not os.path.exists(op) or os.path.getmtime(op) < max(os.path.getmtime(sp), hdr_time):
            jobs.append((src, subprocess.Popen(["nvcc"] + NVCC_FLAGS + ["-c", "-o", op, sp])))
    failed = [src for src, pr in jobs if pr.wait() != 0]
    if failed:
        raise RuntimeError("nvcc failed for " + ", ".join(failed))
    if jobs or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(o) for o in objs):
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs, check=True)
    return LIB_PATH


_lib = None

_SIGNATURES = {
    "pcd_abi_version": (C.c_int, []),
    "pcd_last_error": (C.c_char_p, []),
    "pcd_launch_count": (C.c_int64, []),
    "pcd_denoiser_create": (C.c_int, [C.POINTER(_NamedTensor), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pcd_denoiser_destroy": (C.c_int, [C.c_void_p]),
    "pcd_denoiser_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                             C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_sample_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                  C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_sample_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                  C.c_uint64, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_sample_host_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                       C.c_uint64, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_philox_normal": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_denoiser_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "pcd_denoiser_tap": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "pcd_linear_bf16": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_latent_create": (C.c_int, [C.POINTER(_NamedTensor), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pcd_latent_destroy": (C.c_int, [C.c_void_p]),
    "pcd_latent_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pcd_latent_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                    C.c_int32, C.c_void_p]),
    "pcd_latent_sample_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                         C.c_int32, C.c_void_p]),
    "pcd_vae_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pcd_latent_philox_normal": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_vae3d_create": (C.c_int, [C.POINTER(_NamedTensor), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pcd_vae3d_destroy": (C.c_int, [C.c_void_p]),
    "pcd_vae3d_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pcd_vae3d_tap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "pcd_vae3d_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "pcd_vae3d_encoder_create": (C.c_int, [C.POINTER(_NamedTensor), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pcd_vae3d_encoder_destroy": (C.c_int, [C.c_void_p]),
    "pcd_vae3d_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pcd_vae3d_encoder_tap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "pcd_vae3d_encoder_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "pcd_point_encoder_create": (C.c_int, [C.POINTER(_NamedTensor), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "pcd_point_encoder_destroy": (C.c_int, [C.c_void_p]),
    "pcd_point_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "pcd_point_encoder_tap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "pcd_point_encoder_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "pcd_voxel_count": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "pcd_voxel_points": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "pcd_chamfer_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcd_chamfer_matrix": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                     C.c_void_p]),
    "pcd_sinkhorn_emd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_int32,
                                   C.c_float, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "pcd_emd_exact": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PcdError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype, fn.argtypes = res, args
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise PcdError(lib().pcd_last_error().decode("utf-8", "replace"))


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def launch_count() -> int:
    return int(lib().pcd_launch_count())


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise PcdError(f"{name} must be a CUDA tensor: the B200 path has no CPU fallback")


class Denoiser:
    """Owns the opaque pcd_denoiser handle built from a reference-layout state_dict."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device: torch.device, precision: str = "f16mix"):
        if precision not in PRECISION:
            raise ValueError(f"precision must be one of {sorted(PRECISION)}")
        if device.type != "cuda":
            raise PcdError("the B200 path needs a CUDA device; there is no CPU fallback")
        self.device = device
        self.precision = precision
        keep, arr = [], (_NamedTensor * len(state_dict))()
        for i, (k, v) in enumerate(state_dict.items()):
            v = v.detach()
            if v.dtype == torch.int64:
                t, code = v.cpu().contiguous(), 1
            else:
                t, code = v.to(device="cpu", dtype=torch.float32).contiguous(), 0
            keep.append(t)
            arr[i].name = k.encode()
            arr[i].data = t.data_ptr()
            arr[i].dtype = code
            arr[i].ndim = min(t.dim(), 4)
            for d in range(min(t.dim(), 4)):
                arr[i].shape[d] = t.shape[d]
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        check(lib().pcd_denoiser_create(arr, len(state_dict), PRECISION[precision], idx, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().pcd_denoiser_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def forward(self, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        _require_cuda(x, "x")
        x = x.to(torch.float32).contiguous()
        t = t.to(device=x.device, dtype=torch.float32).contiguous()
        B, N, _ = x.shape
        eps = torch.empty_like(x)
        if B == 0 or N == 0:           # empty batch / empty clouds: nothing to evaluate (the reference returns the empty tensor too)
            return eps
        check(lib().pcd_denoiser_forward(self._h, x.data_ptr(), t.data_ptr(), eps.data_ptr(), B, N, stream_ptr(x.device)))
        return eps

    def sample_(self, sched: torch.Tensor, x: torch.Tensor, noise: Optional[torch.Tensor] = None, seed: int = 0,
                sample_offset: int = 0) -> torch.Tensor:
        """Run the table-driven reverse loop in place on x [B,N,3] (CUDA fp32)."""
        _require_cuda(x, "x")
        assert x.dtype == torch.float32 and x.is_contiguous()
        sched = sched.to(device="cpu", dtype=torch.float32).contiguous()
        S = sched.shape[0]
        B, N, _ = x.shape
        if B == 0 or N == 0:           # the reference's loops run on empty tensors and return them
            return x
        # [S, 8]: one row per step shared by the batch; [S, B, 8]: one row per step AND sample ('linear' schedule quirk)
        rows = 1 if sched.dim() == 2 else sched.shape[1]
        assert sched.shape[-1] == SCHED_ROW and rows in (1, B)
        nptr = None
        if noise is not None:
            _require_cuda(noise, "noise")
            assert noise.dtype == torch.float32 and noise.is_contiguous() and tuple(noise.shape) == (S - 1, B, N, 3)
            nptr = noise.data_ptr()
        check(lib().pcd_sample_rows(self._h, sched.data_ptr(), S, rows, x.data_ptr(), nptr, seed, sample_offset, B, N,
                                    stream_ptr(x.device)))
        return x

    def sample_host(self, sched: torch.Tensor, x_T: torch.Tensor, out: torch.Tensor, seed: int = 0,
                    sample_offset: int = 0) -> torch.Tensor:
        """Host-buffer entry (H2D + loop + D2H + sync inside the call): the e2e path of bench.py."""
        assert not x_T.is_cuda and not out.is_cuda and x_T.dtype == torch.float32 and x_T.is_contiguous()
        sched = sched.to(device="cpu", dtype=torch.float32).contiguous()
        B, N, _ = x_T.shape
        rows = 1 if sched.dim() == 2 else sched.shape[1]       # [S, 8] shared by the batch, or [S, B, 8] one row per sample
        assert sched.shape[-1] == SCHED_ROW and rows in (1, B)
        check(lib().pcd_sample_host_rows(self._h, sched.data_ptr(), sched.shape[0], rows, x_T.data_ptr(), out.data_ptr(), None,
                                         seed, sample_offset, B, N, stream_ptr(self.device)))
        return out

    def profile(self, x: torch.Tensor, t: torch.Tensor):
        """One eager forward with CUDA events between launches -> [(name, ms, algorithmic_flops)]."""
        _require_cuda(x, "x")
        x = x.to(torch.float32).contiguous()
        t = t.to(device=x.device, dtype=torch.float32).contiguous()
        B, N, _ = x.shape
        eps = torch.empty_like(x)
        cap, stride = 64, 48
        ms = (C.c_float * cap)()
        fl = (C.c_double * cap)()
        names = C.create_string_buffer(cap * stride)
        n = C.c_int32(0)
        check(lib().pcd_denoiser_profile(self._h, x.data_ptr(), t.data_ptr(), eps.data_ptr(), B, N, ms, fl, names, stride,
                                         cap, C.byref(n), stream_ptr(x.device)))
        raw = names.raw
        return [(raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode(), float(ms[i]), float(fl[i])) for i in range(n.value)]

    def tap(self, name: str, shape) -> torch.Tensor:
        out = torch.empty(shape, dtype=torch.float32)
        check(lib().pcd_denoiser_tap(self._h, name.encode(), out.data_ptr(), out.numel()))
        return out


def philox_normal(seed: int, sample_offset: int, step: int, B: int, N: int, device) -> torch.Tensor:
    out = torch.empty(B, N, 3, device=device, dtype=torch.float32)
    check(lib().pcd_philox_normal(seed, sample_offset, step, out.data_ptr(), B, N, stream_ptr(out.device)))
    return out


def linear_bf16(a0: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, a1: Optional[torch.Tensor] = None,
                relu: bool = True) -> torch.Tensor:
    """out = relu?([a0|a1] @ w.T + bias) with bf16 operands on the tcgen05 kernel (one fused per-point layer)."""
    _require_cuda(a0, "a0")
    assert a0.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and bias.dtype == torch.float32
    a0, w, bias = a0.contiguous(), w.contiguous(), bias.contiguous()
    M, K0 = a0.shape
    K1 = 0
    if a1 is not None:
        a1 = a1.contiguous()
        K1 = a1.shape[1]
    Cout = w.shape[0]
    assert w.shape[1] == K0 + K1
    out = torch.empty(M, Cout, device=a0.device, dtype=torch.bfloat16)
    check(lib().pcd_linear_bf16(a0.data_ptr(), K0, a1.data_ptr() if a1 is not None else None, K1, w.data_ptr(),
                                bias.data_ptr(), out.data_ptr(), M, Cout, int(relu), stream_ptr(a0.device)))
    return out


def chamfer_pairs(x: torch.Tensor, y: torch.Tensor, scaling: float = 1e3, return_indices: bool = False):
    _require_cuda(x, "x")
    _require_cuda(y, "y")
    x = x.to(torch.float32).contiguous()
    y = y.to(torch.float32).contiguous()
    B, N, _ = x.shape
    M = y.shape[1]
    if B == 0:                         # batch mean of nothing: NaN, as in the reference (metrics.py:46)
        e = torch.empty(0, device=x.device, dtype=torch.float32)
        z = torch.empty(0, N, device=x.device, dtype=torch.int32), torch.empty(0, M, device=x.device, dtype=torch.int32)
        return (e, z[0], z[1]) if return_indices else e
    cd = torch.empty(B, device=x.device, dtype=torch.float32)
    ixy = iyx = None
    if return_indices:
        ixy = torch.empty(B, N, device=x.device, dtype=torch.int32)
        iyx = torch.empty(B, M, device=x.device, dtype=torch.int32)
    check(lib().pcd_chamfer_pairs(x.data_ptr(), y.data_ptr(), B, N, M, scaling, cd.data_ptr(),
                                  ixy.data_ptr() if return_indices else None,
                                  iyx.data_ptr() if return_indices else None, stream_ptr(x.device)))
    return (cd, ixy, iyx) if return_indices else cd


def chamfer_matrix(G: torch.Tensor, R: torch.Tensor, scaling: float = 1e3) -> torch.Tensor:
    _require_cuda(G, "G")
    _require_cuda(R, "R")
    G = G.to(torch.float32).contiguous()
    R = R.to(torch.float32).contiguous()
    assert G.shape[1] == R.shape[1], "all clouds must have the same number of points"
    out = torch.empty(G.shape[0], R.shape[0], device=G.device, dtype=torch.float32)
    check(lib().pcd_chamfer_matrix(G.data_ptr(), G.shape[0], R.data_ptr(), R.shape[0], G.shape[1], scaling,
                                   out.data_ptr(), stream_ptr(G.device)))
    return out


def sinkhorn_emd(x: torch.Tensor, y: torch.Tensor, epsilon: float = 1e-2, thresh: float = 1e-5, max_iter: int = 100,
                 scaling: float = 1.0):
    """Per-pair Sinkhorn EMD (reference metrics.py:94-158) -> (emd[B] on the device, iterations run)."""
    _require_cuda(x, "x")
    _require_cuda(y, "y")
    x = x.to(torch.float32).contiguous()
    y = y.to(torch.float32).contiguous()
    B, N, _ = x.shape
    assert y.shape[0] == B, "batch sizes must be the same"
    emd = torch.empty(B, device=x.device, dtype=torch.float32)
    iters = C.c_int32(0)
    check(lib().pcd_sinkhorn_emd(x.data_ptr(), y.data_ptr(), B, N, y.shape[1], epsilon, thresh, max_iter, scaling,
                                 emd.data_ptr(), C.byref(iters), stream_ptr(x.device)))
    return emd, int(iters.value)


def emd_exact(x: torch.Tensor, y: torch.Tensor, scaling: float = 1.0, return_assignment: bool = False):
    """Per-pair exact EMD (reference metrics.py:49-92) -> emd[B] on the device and, with return_assignment, the matched y index
    of every x as int32 [B, N] (-1: unmatched)."""
    _require_cuda(x, "x")
    _require_cuda(y, "y")
    x = x.to(torch.float32).contiguous()
    y = y.to(torch.float32).contiguous()
    B, N, _ = x.shape
    assert y.shape[0] == B, "batch sizes must be the same"
    emd = torch.empty(B, device=x.device, dtype=torch.float32)
    assign = torch.empty(B, N, device=x.device, dtype=torch.int32) if return_assignment else None
    if B > 0:
        check(lib().pcd_emd_exact(x.data_ptr(), y.data_ptr(), B, N, y.shape[1], scaling, emd.data_ptr(),
                                  assign.data_ptr() if return_assignment else None, stream_ptr(x.device)))
    return (emd, assign) if return_assignment else emd
