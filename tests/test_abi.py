"""CPU: the C-ABI library builds, loads and exports every symbol include/gstvd.h declares (no compute without a GPU)."""
import ctypes
import os
import re

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from gst_visdial_b200 import _build, _lib
    if not os.path.exists(_lib.LIB_PATH):
        _build.build()
    return _lib


def test_header_symbols_exported():
    L = _lib()
    lib = L.load()
    header = open(os.path.join(ROOT, "include", "gstvd.h")).read()
    declared = set(re.findall(r"\b(gstvd_[a-z0-9_]+)\s*\(", header))
    declared -= {"gstvd_ctx"}
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in gstvd.h but not exported"
    bound = {n for n, _, _ in L.SYMBOLS}
    assert declared == bound, f"ctypes binding and header disagree: {declared ^ bound}"
    assert lib.gstvd_abi_version() == L.GSTVD_ABI_VERSION


def test_config_struct_matches_header_field_order():
    L = _lib()
    header = open(os.path.join(ROOT, "include", "gstvd.h")).read()
    c_types = {"int32_t": ctypes.c_int32, "uint64_t": ctypes.c_uint64, "int64_t": ctypes.c_int64, "float": ctypes.c_float}
    for name, struct in (("gstvd_config", L.GstvdConfig), ("gstvd_gen_params", L.GstvdGenParams)):
        end = header.index("} %s;" % name)
        body = re.sub(r"/\*.*?\*/", "", header[header.rindex("typedef struct {", 0, end):end], flags=re.S)
        fields = []
        for c_type, decl in re.findall(r"\b(u?int(?:32|64)_t|float)\s+([^;]+);", body):
            for part in decl.split(","):
                fields.append((re.sub(r"\[.*\]", "", part).strip(), c_types[c_type]))
        bound = [(f, t._type_ if issubclass(t, ctypes.Array) else t) for f, t in struct._fields_]
        assert fields == bound, name


def test_create_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        return
    L = _lib()
    lib = L.load()
    cfg = L.GstvdConfig()
    cfg.abi_version = L.GSTVD_ABI_VERSION
    ctx = ctypes.c_void_p()
    rc = lib.gstvd_create(ctypes.byref(cfg), 0, ctypes.byref(ctx))
    assert rc < 0 and not ctx.value
    assert lib.gstvd_last_error(None)


def test_engine_refuses_cpu():
    if torch.cuda.is_available():
        return
    import pytest
    from gst_visdial_b200 import weights as W
    from gst_visdial_b200.engine import Engine
    with pytest.raises(RuntimeError):
        Engine(W.load_json_config(W.TINY_ENC_CONFIG), None)
