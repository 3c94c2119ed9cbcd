"""The C-ABI library builds for sm_100a, loads, and exports every symbol include/usflows_b200.h declares
(no compute calls: this runs without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(usf_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_bound_and_versioned():
    from usflows_b200 import _lib
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in _lib.py"
    assert lib.usf_abi_version() == 10


def test_planes_struct_layout_matches_header():
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_planes \{(.*?)\} usf_planes;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b([A-Za-z_0-9]+);", body)
    assert fields == [f[0] for f in _lib.Planes._fields_]
    assert ctypes.sizeof(_lib.Planes) == 10 * 8


def test_linear_args_layout_matches_header():
    """ctypes mirror vs the C struct: field order and count."""
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_linear_args \{(.*?)\} usf_linear_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b([A-Za-z_0-9]+);", body)
    assert fields == [f[0] for f in _lib.LinearArgs._fields_]
    assert ctypes.sizeof(_lib.LinearArgs) == 8 + 4 * 4 + 6 * 8 + 8 + 4 + 4 + 3 * 8 + 2 * 8 + 2 * 8 + 3 * 8 + 2 * 8 + 7 * 8 + 8


def test_glue_args_layout_matches_header():
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_glue_args \{(.*?)\} usf_glue_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b([A-Za-z_0-9]+);", body)
    assert fields == [f[0] for f in _lib.GlueArgs._fields_]
    assert ctypes.sizeof(_lib.GlueArgs) == 21 * 8


def test_invalid_arguments_fail_loudly_without_gpu():
    from usflows_b200 import _lib
    lib = _lib.load()
    rc = lib.usf_linear(None, None)
    assert rc == -1 and b"null args" in lib.usf_last_error()
    with pytest.raises(RuntimeError, match="usflows_b200"):
        _lib.check(rc)


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    """tcgen05.mma -> UTC*MMA, TMA -> UTMALDG, tcgen05.ld -> LDTM (B200_PROFILING.md); the fp64 products of the weight
    preparation -> DMMA (mma.sync.m8n8k4.f64: the fp64 tensor-core path of sm_100a)."""
    import shutil
    import subprocess
    from usflows_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    _lib.load()
    sass = subprocess.run([cuobjdump, "-sass", _lib.library_path()], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM", "DMMA"):
        assert mnemonic in sass, mnemonic
    assert "sm_100a" in sass


def test_plan_linear_layout_matches_header():
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_plan_linear \{(.*?)\} usf_plan_linear;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [n for decl in body.split(";") for n in re.findall(r"([A-Za-z_0-9]+)\s*(?:,|$)", decl.strip().replace("\n", " "))
              if n not in ("int32_t", "int64_t", "float", "const", "void")]
    assert fields == [f[0] for f in _lib.PlanLinear._fields_], fields
    assert ctypes.sizeof(_lib.PlanLinear) == 4 * 4 + 3 * 8 + 8 + 4 * 4 + 4 + 4


def test_plan_entry_points_reject_bad_input_without_gpu():
    from usflows_b200 import _lib
    lib = _lib.load()
    assert lib.usf_plan_create(None, 8, 0, 16) == -1 and b"bad input" in lib.usf_last_error()
    h = ctypes.c_void_p()
    assert lib.usf_plan_create(ctypes.byref(h), 8, 0, 16) == 0 and h.value
    assert lib.usf_plan_finalize(h) == -1                       # no steps
    assert lib.usf_flow_logprob(h, None, 0, 0, None, None, None) == -1
    assert lib.usf_plan_destroy(h) == 0


def test_conv_pix_args_layout_matches_header():
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_conv_pix_args \{(.*?)\} usf_conv_pix_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [n for decl in body.split(";") for n in re.findall(r"([A-Za-z_0-9]+)\s*(?:,|$)", decl.strip().replace("\n", " "))
              if n not in ("int32_t", "int64_t", "float", "const", "void")]
    assert fields == [f[0] for f in _lib.ConvPixArgs._fields_], fields
    assert ctypes.sizeof(_lib.ConvPixArgs) == 2 * 8 + 4 * 4 + 2 * 8 + 4 * 4 + 4 * 8 + 2 * 4 + 3 * 8 + 2 * 4 + 4 * 8


def test_pix_and_store_path_entry_points_reject_bad_input_without_gpu():
    from usflows_b200 import _lib
    lib = _lib.load()
    assert lib.usf_conv2d_pix(None, None) == -1 and b"null args" in lib.usf_last_error()
    a = _lib.ConvPixArgs()
    assert lib.usf_conv2d_pix(ctypes.byref(a), None) == -1                  # null operands
    assert lib.usf_pix_encode(None, 0, 0, 16, 49, None, 0, None, None, None) == -1
    assert lib.usf_debug_set_store_path(16) == -1 and b"store path flags" in lib.usf_last_error()
    assert lib.usf_debug_set_store_path(1 << 30) == -1
    assert lib.usf_debug_set_store_path(4 | 32 | 256) == 0 and lib.usf_debug_set_store_path(0) == 0
