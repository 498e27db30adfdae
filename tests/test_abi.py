"""The C-ABI shared library loads on a CPU-only box and exports every symbol include/*.h declares
(no compute calls here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    import mv_native
    return mv_native.lib()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mv_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_expected_surface():
    syms = declared_symbols()
    for s in ("mv_float_quantize", "mv_fixed_point_quantize", "mv_block_quantize", "mv_gemm",
              "mv_layernorm_q_fwd", "mv_layernorm_q_bwd", "mv_attention_fwd", "mv_attention_bwd",
              "mv_quantize_weight", "mv_last_error"):
        assert s in syms


def declared_fields(struct):
    text = open(os.path.join(ROOT, "include", "mv_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\} %s;" % struct, text).group(1)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        first, *rest = decl.split(",")
        names += [re.findall(r"\w+", first)[-1]] + [r.strip() for r in rest]
    return names


@pytest.mark.parametrize("struct,cls", [("mv_gemm_args", "GemmArgs"), ("mv_layernorm_bwd_args", "LayerNormBwdArgs")])
def test_ctypes_structs_mirror_the_header(struct, cls):
    import mv_native
    assert [f[0] for f in getattr(mv_native, cls)._fields_] == declared_fields(struct)


def test_every_declared_symbol_is_exported(lib):
    for s in declared_symbols():
        assert hasattr(lib, s), "libmv_b200.so does not export " + s


def test_error_reporting_without_a_gpu(lib):
    lib.mv_last_error.restype = ctypes.c_char_p
    rc = lib.mv_float_quantize(None, None, 0, ctypes.c_int64(8), 9, 10, 0, ctypes.c_uint64(0),
                               ctypes.c_uint64(0), None)
    assert rc != 0
    assert b"exp_bits" in lib.mv_last_error()
    assert lib.mv_version() >= 100


@pytest.mark.parametrize("field", ["a_dtype", "out_dtype"])
def test_gemm_rejects_other_element_types_without_a_gpu(lib, field):
    """mv_gemm takes MV_F16 / MV_F32 operands and outputs only; type 2 (bf16, which no kernel reads or writes) is
    rejected before anything touches a device.  The pointers are never dereferenced."""
    import mv_native
    lib.mv_last_error.restype = ctypes.c_char_p
    a = mv_native.GemmArgs()
    a.M = a.N = a.K = a.lda = a.ldb = a.ld_out = 128
    a.A = a.B = a.out = 1 << 20
    a.a_dtype = a.b_dtype = a.out_dtype = mv_native.F16
    if field == "a_dtype":
        a.a_dtype = a.b_dtype = 2
    else:
        a.out_dtype = 2
    assert lib.mv_gemm(ctypes.byref(a), None) != 0
    assert b"MV_F16" in lib.mv_last_error()


def test_missing_library_fails_loudly(monkeypatch):
    import mv_native
    monkeypatch.setattr(mv_native, "_lib", None)
    monkeypatch.setattr(mv_native, "_SO", "/nonexistent/libmv_b200.so")
    with pytest.raises(mv_native.MvError, match="no CPU fallback"):
        mv_native.lib()
