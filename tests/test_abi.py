"""CPU checks of the drop-in boundary: libtdb200.so loads and exports exactly what include/tdb200.h declares."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tdb200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tdb200_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def libpath():
    from turbodiffusion_b200 import _build
    return _build.build()


def test_header_declares_the_hot_path():
    names = _declared()
    for required in ("tdb200_quant_int8_block128", "tdb200_gemm_w8a8", "tdb200_rms_norm", "tdb200_layer_norm",
                     "tdb200_layer_norm_modulate_quant", "tdb200_gate_residual", "tdb200_rope_interleaved",
                     "tdb200_sla_block_map", "tdb200_sla_quant_qk", "tdb200_sla_linear_moments", "tdb200_sla_attn_fwd"):
        assert required in names


def test_library_exports_every_declared_symbol(libpath):
    out = subprocess.run(["nm", "-D", "--defined-only", libpath], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r" T (tdb200_[a-z0-9_]+)", out)))
    assert exported == _declared()


def test_ctypes_binding_matches_header(libpath):
    from turbodiffusion_b200 import _lib
    assert sorted(_lib.exported_names()) == _declared()
    lib = _lib.lib()  # raises if any prototype names a missing symbol
    assert lib.tdb200_abi_version() == 1
    assert lib.tdb200_last_error() is not None


def test_no_torch_types_in_the_abi():
    src = open(HEADER).read()
    assert "torch" not in src.replace("PyTorch", "") or "at::" not in src
    assert "at::Tensor" not in src and "torch::" not in src


def test_errors_are_codes_not_exits(libpath):
    """Argument validation happens before any CUDA call, so it can be exercised without a GPU."""
    from turbodiffusion_b200 import _lib
    lib = _lib.lib()
    rc = lib.tdb200_quant_int8_block128(None, 0, 4, 8, None, None, None)
    assert rc == -1 and b"null" in lib.tdb200_last_error()
    rc = lib.tdb200_gemm_w8a8(ctypes.c_void_p(16), ctypes.c_void_p(16), ctypes.c_void_p(16), ctypes.c_void_p(16), None,
                              ctypes.c_void_p(16), 0, 128, 128, 100, None)
    assert rc == -2 and b"multiple of 128" in lib.tdb200_last_error()


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "turbodiffusion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "td_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def _p(v=4096):
    return ctypes.c_void_p(v)          # non-null, 16-byte aligned, never dereferenced: validation runs before any CUDA call


def test_argument_validation_of_every_kernel_family(libpath):
    """Every entry point checks pointers / shapes / dtypes first and reports through the return code + tdb200_last_error
    (never exit(), never a crash), so the contract can be exercised on a machine without a GPU."""
    from turbodiffusion_b200 import _lib
    lib = _lib.lib()
    INVALID, UNSUPPORTED, WORKSPACE = -1, -2, -5
    cases = [
        ("quant null", lambda: lib.tdb200_quant_int8_block128(None, 0, 128, 128, _p(), _p(), None), INVALID, b"null"),
        ("gemm k%128", lambda: lib.tdb200_gemm_w8a8(_p(), _p(), _p(), _p(), None, _p(), 0, 128, 128, 100, None), UNSUPPORTED, b"128"),
        ("gemm n%8", lambda: lib.tdb200_gemm_w8a8(_p(), _p(), _p(), _p(), None, _p(), 0, 128, 100, 128, None), UNSUPPORTED, b"multiple of 8"),
        ("gemm misaligned", lambda: lib.tdb200_gemm_w8a8(_p(4100), _p(), _p(), _p(), None, _p(), 0, 128, 128, 128, None), INVALID, b"aligned"),
        ("gemm epilogue", lambda: lib.tdb200_gemm_w8a8_ex(_p(), _p(), _p(), _p(), None, _p(), 0, 128, 128, 128, 9, None), INVALID, b"epilogue"),
        ("rowwise null", lambda: lib.tdb200_gemm_w8a8_rowwise(_p(), _p(), _p(), _p(), None, None, 0, 128, 128, 128, None), INVALID, b"null"),
        ("rowquant k%8", lambda: lib.tdb200_quant_int8_rowwise(_p(), 0, 4, 12, _p(), _p(), None), INVALID, b"shape"),
        ("sla prep head dim", lambda: lib.tdb200_sla_quant_qk(_p(), _p(), 0, 1, 256, 256, 2, 96, _p(), _p(), _p(), _p(), _p(), _p(), _p(), None),
         UNSUPPORTED, b"head dim"),
        ("block map topk", lambda: lib.tdb200_sla_block_map(_p(), _p(), 0, 1, 2, 4, 8, 128, 9, _p(), _p(), None), INVALID, b"topk"),
        ("moments head dim", lambda: lib.tdb200_sla_linear_moments(_p(), _p(), 0, 1, 256, 2, 96, _p(), _p(), None), UNSUPPORTED, b"head dim"),
        ("moments feature map", lambda: lib.tdb200_sla_linear_moments_ex(_p(), _p(), 0, 1, 256, 2, 64, 7, _p(), _p(), None), INVALID, b"feature"),
        ("moments ws too small", lambda: lib.tdb200_sla_linear_moments_ws(_p(), _p(), 0, 1, 256, 2, 128, 0, _p(), _p(), _p(), 1024, None),
         WORKSPACE, b"needed"),
        ("moments ws null", lambda: lib.tdb200_sla_linear_moments_ws(_p(), _p(), 0, 1, 256, 2, 128, 0, _p(), _p(), None, 1 << 30, None),
         INVALID, b"null"),
        ("moments ws head dim", lambda: lib.tdb200_sla_linear_moments_ws(_p(), _p(), 0, 1, 256, 2, 96, 0, _p(), _p(), _p(), 1 << 30, None),
         UNSUPPORTED, b"head dim"),
        ("moments ws ksum misaligned", lambda: lib.tdb200_sla_linear_moments_ws(_p(), _p(), 0, 1, 256, 2, 128, 0, _p(), _p(4100), _p(),
                                                                                 1 << 30, None), INVALID, b"aligned"),
        ("moments workspace shape", lambda: lib.tdb200_sla_linear_moments_workspace(0, 256, 2, 128, ctypes.byref(ctypes.c_int64())),
         INVALID, b"shape"),
        ("attn v2 head dim", lambda: lib.tdb200_sla_attn_fwd_v2(_p(), _p(), _p(), _p(), _p(), _p(), 0, _p(), 4, _p(), _p(), _p(), _p(), 1, 256,
                                                                256, 2, 96, 0.088, 0, None), UNSUPPORTED, b"head dim"),
        ("gelu quant k", lambda: lib.tdb200_gelu_quant_int8_block128(_p(), 0, 128, 100, _p(), _p(), None), UNSUPPORTED, b"multiple of 8"),
        ("attn kseq batch", lambda: lib.tdb200_sla_attn_fwd_kseq(_p(), _p(), _p(), _p(), _p(), _p(), 0, _p(), 4, _p(), _p(), _p(), _p(), 2, 256,
                                                                 256, 2, 128, 0.088, None), UNSUPPORTED, b"batch"),
        ("split parts", lambda: lib.tdb200_gemm_w8a8_split(_p(), _p(), _p(), _p(), None, _p(), 0, 128, 768, 128, 2, None), UNSUPPORTED,
         b"parts"),
        ("split null", lambda: lib.tdb200_gemm_w8a8_split(_p(), _p(), _p(), _p(), None, None, 0, 128, 512, 128, 2, None), INVALID, b"null"),
        ("kmean partial head dim", lambda: lib.tdb200_sla_kmean_partial(_p(), 0, 1, 256, 2, 96, _p(), None), UNSUPPORTED, b"head dim"),
        ("kmean final null", lambda: lib.tdb200_sla_kmean_final(None, 1, 2, 2, 128, 256, _p(), None), INVALID, b"null"),
        ("quant k seq null", lambda: lib.tdb200_sla_quant_k_seq(_p(), None, 0, 1, 256, 2, 128, _p(), _p(), _p(), None), INVALID, b"null"),
        ("project moments head dim", lambda: lib.tdb200_sla_project_moments(_p(), _p(), 0, 4, 96, _p(), None), UNSUPPORTED, b"head dim"),
        ("rope table null", lambda: lib.tdb200_rms_norm_rope_table(None, 0, _p(), _p(), _p(), 64, 2, 128, 1e-6, None), INVALID, b"null"),
        ("attn null", lambda: lib.tdb200_sla_attn_fwd(None, _p(), _p(), _p(), _p(), _p(), 0, _p(), 4, _p(), _p(), _p(), _p(), 1, 256, 256, 2,
                                                      128, 0.088, None), INVALID, b"null"),
        ("attn topk", lambda: lib.tdb200_sla_attn_fwd(_p(), _p(), _p(), _p(), _p(), _p(), 0, _p(), 9, _p(), _p(), _p(), _p(), 1, 256, 256, 2,
                                                      128, 0.088, None), INVALID, b"topk"),
    ]
    for name, call, code, needle in cases:
        rc = call()
        msg = lib.tdb200_last_error() or b""
        assert rc == code, (name, rc, msg)
        assert needle in msg, (name, msg)


def test_moments_workspace_size_is_a_function_of_the_shape(libpath):
    """The size query runs on the host: splits = min(tiles, max(1, 148 // (b * head units))) slots of kv [b,h,d,d] + ksum
    [b,h,d] fp32; 64-wide heads are paired into one unit."""
    from turbodiffusion_b200 import _lib
    lib = _lib.lib()

    def size(b, l, h, d):
        n = ctypes.c_int64(-1)
        assert lib.tdb200_sla_linear_moments_workspace(b, l, h, d, ctypes.byref(n)) == 0, lib.tdb200_last_error()
        return n.value

    assert size(1, 32760, 12, 128) == 12 * 12 * 128 * 129 * 4      # shape A: 12 splits of the 256 key tiles
    assert size(1, 75600, 40, 128) == 3 * 40 * 128 * 129 * 4       # 14B: 3 splits
    assert size(1, 32760, 24, 64) == 12 * 24 * 64 * 65 * 4         # 12 pairs of 64-wide heads
    assert size(1, 32760, 23, 64) == 12 * 23 * 64 * 65 * 4         # an odd head count: the last pair is half empty
    assert size(1, 200, 2, 128) == 2 * 2 * 128 * 129 * 4            # no more splits than 128-row tiles
    assert size(4, 1000, 40, 128) == 1 * 4 * 40 * 128 * 129 * 4     # more head units than SMs: one split
    rc = lib.tdb200_sla_linear_moments_ws(_p(), _p(), 0, 1, 32760, 12, 128, 0, _p(), _p(), _p(), size(1, 32760, 12, 128) - 16, None)
    assert rc == -5 and b"needed" in lib.tdb200_last_error()


def test_valid_calls_without_a_gpu_report_an_error_code(libpath):
    """On a CUDA-less host a well-formed call must come back with a negative code and a message (no fallback, no crash)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("this check is for hosts without a GPU")
    from turbodiffusion_b200 import _lib
    lib = _lib.lib()
    rc = lib.tdb200_gemm_w8a8(_p(), _p(), _p(), _p(), None, _p(), 0, 128, 128, 128, None)
    assert rc in (-3, -4) and lib.tdb200_last_error()
    rc = lib.tdb200_quant_int8_block128(_p(), 0, 128, 128, _p(), _p(), None)
    assert rc in (-3, -4) and lib.tdb200_last_error()
