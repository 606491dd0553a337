"""ctypes binding of libtdb200.so (the C ABI declared in include/tdb200.h).

The product path has NO fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p

import torch

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libtdb200.so")
if os.environ.get("TDB200_LIB"):   # kernel-variant experiments: a differently compiled build of the same ABI (see profiles/r02_gemm_experiments.md, call 21)
    LIB_PATH = os.environ["TDB200_LIB"]

DTYPE_TAG = {torch.bfloat16: 0, torch.float16: 1}

_P, _I64, _F, _I = c_void_p, c_int64, c_float, c_int

# name -> argtypes (restype is int unless listed in _RESTYPES)
_PROTOS = {
    "tdb200_abi_version": [],
    "tdb200_last_error": [],
    "tdb200_quant_int8_block128": [_P, _I, _I64, _I64, _P, _P, _P],
    "tdb200_gelu_quant_int8_block128": [_P, _I, _I64, _I64, _P, _P, _P],
    "tdb200_gemm_w8a8": [_P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I64, _P],
    "tdb200_gemm_w8a8_ex": [_P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I64, _I, _P],
    "tdb200_gemm_w8a8_split": [_P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I64, _I64, _P],
    "tdb200_gemm_w8a8_quant_out": [_P, _P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I64, _I, _P],
    "tdb200_rms_norm_f32": [_P, _P, _P, _I64, _I64, _F, _P],
    "tdb200_layer_norm_f32": [_P, _P, _P, _P, _I64, _I64, _F, _P],
    "tdb200_rms_norm": [_P, _I, _P, _P, _I64, _I64, _F, _P],
    "tdb200_layer_norm": [_P, _I, _P, _P, _P, _I64, _I64, _F, _P],
    "tdb200_layer_norm_modulate": [_P, _I, _P, _P, _P, _I64, _I64, _F, _P],
    "tdb200_layer_norm_modulate_quant": [_P, _I, _P, _P, _P, _P, _P, _I64, _I64, _F, _P],
    "tdb200_gate_residual": [_P, _P, _P, _P, _I, _I64, _I64, _P],
    "tdb200_gate_residual_stats": [_P, _P, _P, _P, _P, _I, _I64, _I64, _F, _P],
    "tdb200_layer_norm_modulate_quant_stats": [_P, _I, _P, _P, _P, _P, _P, _I64, _I64, _P],
    "tdb200_rope_interleaved": [_P, _I, _P, _P, _I64, _I64, _I64, _P],
    "tdb200_rms_norm_rope": [_P, _I, _P, _P, _P, _I64, _I64, _I64, _F, _P],
    "tdb200_rms_norm_rope_table": [_P, _I, _P, _P, _P, _I64, _I64, _I64, _F, _P],
    "tdb200_sla_quant_qk": [_P, _P, _I, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P],
    "tdb200_sla_block_map": [_P, _P, _I, _I64, _I64, _I64, _I64, _I64, _I64, _P, _P, _P],
    "tdb200_sla_linear_moments": [_P, _P, _I, _I64, _I64, _I64, _I64, _P, _P, _P],
    "tdb200_sla_linear_moments_ex": [_P, _P, _I, _I64, _I64, _I64, _I64, _I, _P, _P, _P],
    "tdb200_sla_linear_moments_workspace": [_I64, _I64, _I64, _I64, ctypes.POINTER(c_int64)],
    "tdb200_sla_linear_moments_ws": [_P, _P, _I, _I64, _I64, _I64, _I64, _I, _P, _P, _P, _I64, _P],
    "tdb200_sla_attn_fwd": [_P, _P, _P, _P, _P, _P, _I, _P, _I64, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _F,
                            _P],
    "tdb200_sla_attn_fwd_kseq": [_P, _P, _P, _P, _P, _P, _I, _P, _I64, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _F,
                                 _P],
    "tdb200_sla_project_moments": [_P, _P, _I, _I64, _I64, _P, _P],
    "tdb200_sla_kmean_partial": [_P, _I, _I64, _I64, _I64, _I64, _P, _P],
    "tdb200_sla_kmean_final": [_P, _I64, _I64, _I64, _I64, _I64, _P, _P],
    "tdb200_sla_quant_k_seq": [_P, _P, _I, _I64, _I64, _I64, _I64, _P, _P, _P, _P],
    "tdb200_sla_attn_fwd_qk16": [_P, _P, _P, _I, _P, _I64, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _F, _P],
    "tdb200_sla_attn_fwd_v2": [_P, _P, _P, _P, _P, _P, _I, _P, _I64, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _F, _I,
                               _P],
    "tdb200_ltx_modulated_rms_norm_ada": [_P, _I, _P, _P, _I, _I, _I, _P, _I64, _I64, _I64, _I64, _F, _P],
    "tdb200_ltx_modulate_ada": [_P, _I, _P, _P, _I, _I, _I, _P, _I64, _I64, _I64, _I64, _P],
    "tdb200_ltx_gated_residual_ada": [_P, _P, _I, _P, _P, _I, _I, _P, _I64, _I64, _I64, _I64, _P],
    "tdb200_ltx_split_rope": [_P, _P, _P, _I, _P, _I64, _I64, _I64, _I64, _P],
    "tdb200_quant_int8_rowwise": [_P, _I, _I64, _I64, _P, _P, _P],
    "tdb200_gemm_w8a8_rowwise": [_P, _P, _P, _P, _P, _P, _I, _I64, _I64, _I64, _P],
    "tdb200_debug_set_attn_trace": [_P],
    "tdb200_selftest_umma_bf16": [_P, _P, _P, _P],
    "tdb200_selftest_tmem_read": [_I, _I, _I, _P, _P, _P],
    "tdb200_selftest_mufu": [_I, _I, _I, _P, _P, _P],
    "tdb200_selftest_softmax_exps": [_I, _I, _I, _P, _P, _P],
}
_RESTYPES = {"tdb200_last_error": c_char_p}

_lib = None


class Tdb200Error(RuntimeError):
    pass


def exported_names():
    return list(_PROTOS.keys())


def lib() -> ctypes.CDLL:
    """Load libtdb200.so (once).  Raises if it has not been built: there is no CPU or eager fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Tdb200Error(
                f"{LIB_PATH} not found. Build it with `python -m turbodiffusion_b200._build` "
                "(or __graft_entry__.build()). turbodiffusion_b200 has no fallback path.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, argtypes in _PROTOS.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, c_int)
        if handle.tdb200_abi_version() != 1:
            raise Tdb200Error("libtdb200.so ABI version mismatch")
        _lib = _DeviceGuarded(handle)
    return _lib


_CALL_DEVICE = None  # device index of the tensors of the call being assembled (set by stream_ptr)


class _DeviceGuarded:
    """The C side works on the CUDA runtime's *current* device (cudaGetDevice) with the stream handed in.  Every Python
    wrapper evaluates stream_ptr(tensor.device) while building its argument list; if that device is not the current one,
    the call is made under torch.cuda.device(...) so tensors on a non-current GPU work like they do for torch ops."""

    def __init__(self, handle):
        self._handle = handle
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            raw = getattr(self._handle, name)

            def fn(*args, _raw=raw):
                global _CALL_DEVICE
                dev, _CALL_DEVICE = _CALL_DEVICE, None
                if dev is not None and dev != torch.cuda.current_device():
                    with torch.cuda.device(dev):
                        return _raw(*args)
                return _raw(*args)

            self._cache[name] = fn
        return fn


LAUNCHES = 0  # kernels launched through the C ABI (each entry point documents how many it enqueues)
_KERNELS_PER_CALL = {"sla_quant_qk": 4, "layernorm_modulate_quant": 2, "sla_linear_moments": 2}  # upper bounds per entry point


def check(rc: int, what: str, launches: int = None) -> None:
    global LAUNCHES
    LAUNCHES += _KERNELS_PER_CALL.get(what, 1) if launches is None else launches
    if rc != 0:
        msg = lib().tdb200_last_error()
        raise Tdb200Error(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def stream_ptr(device=None) -> int:
    global _CALL_DEVICE
    if device is not None:
        dev = torch.device(device)
        _CALL_DEVICE = dev.index if dev.index is not None else torch.cuda.current_device()
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t):
    return 0 if t is None else t.data_ptr()


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise Tdb200Error("turbodiffusion_b200 ops take CUDA tensors only (no CPU fallback)")
