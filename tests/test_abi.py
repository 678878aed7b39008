"""The C-ABI library builds, loads and exports every symbol include/ctb.h declares.
No compute calls (no GPU needed)."""
import ctypes
import os
import re

import pytest

import __graft_entry__ as G
from climate_toolbox_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    G.build()
    return _native.lib()


def _declared():
    src = open(os.path.join(ROOT, "include", "ctb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ctb_[a-z_]+)\s*\(", src)))


def test_header_and_binding_agree():
    assert _declared() == sorted(_native.SYMBOLS)


def test_library_exports_every_declared_symbol(built):
    L = ctypes.CDLL(_native.LIB_PATH)
    for sym in _declared():
        assert hasattr(L, sym), sym
    assert built.ctb_version() == 100


def test_struct_layouts_match_header(built):
    # sizes follow from the field lists in include/ctb.h
    assert ctypes.sizeof(_native.PlanOpts) == 32 + 8            # 8 x int32 + the cell_gate pointer
    assert ctypes.sizeof(_native.AggOpts) == 8 + 8 + 4 + 4 + 8 + 8 + 8   # groups, t_begin, flush, n_peer_out, day_of_year, peer_out, peer_row
    assert _native.gate_word(0, 511, 0) == _native.GATE_ALWAYS
    assert ctypes.sizeof(_native.PlanInfo) == 4 * 8 + 2 * 4 + 2 * 8 + 8 * 4 + 2 * 8


def test_invalid_calls_fail_cleanly_without_gpu(built):
    # argument validation happens before any CUDA call
    rc = built.ctb_plan_get_info(None, None)
    assert rc == _native.ERR_INVALID and "null" in _native.last_error()
    with pytest.raises(ValueError):
        _native.check(rc)
    assert built.ctb_aggregate_workspace_bytes(None, 10, 1) == 0
    # ctb_push_rows: a column block that does not fit the leading dimension, too many peers
    assert built.ctb_push_rows(None, 10, 8, 4, 1, 1, None, 0, None) == _native.ERR_INVALID
    assert built.ctb_push_rows(None, 10, 0, 4, 1, _native.MAX_PEERS + 1, None, 0, None) == _native.ERR_INVALID
    assert built.ctb_push_rows(None, 10, 0, 0, 1, 1, None, 0, None) == 0          # nothing to copy


# (transform, params, n_out, error text): pairs no kernel is compiled for
UNSUPPORTED_PAIRS = [(9, [0.0], 1, "transform=9"),
                     (_native.TR_POLY, [0.0, 1, 2, 3, 4, 5], 5, "n_out=5"),
                     (_native.TR_IDENTITY, [], 2, "n_out=1")]


def _params(params):
    return (ctypes.c_double * max(len(params), 1))(*params), len(params)


def test_transform_rejects_unsupported_pairs_without_gpu(built):
    dummy = ctypes.c_double(0.0)
    for kind, params, n_out, text in UNSUPPORTED_PAIRS:
        p, n_p = _params(params)
        # n = 0: the call validates its arguments and returns before any CUDA call
        rc = built.ctb_transform(ctypes.addressof(dummy), ctypes.addressof(dummy), _native.F64, 0, kind, p, n_p,
                                 n_out, None, None)
        assert rc == _native.ERR_INVALID and text in _native.last_error(), (kind, n_out, _native.last_error())


@pytest.mark.gpu
def test_aggregate_rejects_unsupported_pairs(built):
    import torch
    from climate_toolbox_b200 import _engine as E
    from climate_toolbox_b200 import synthetic

    lat, lon = synthetic.grid_labels(1.0)
    plan = E.get_plan(E.GridSpec(lat, lon), synthetic.weights_table(1.0, 20, seed=5), "popwt", "hierid",
                      device=torch.device("cuda", 0), cache=False)
    T, ncell = 32, len(lat) * len(lon)
    x = torch.zeros((T, ncell), dtype=torch.float32, device="cuda:0")
    out = torch.zeros((_native.MAX_OUT + 1, plan.R, T), dtype=torch.float64, device="cuda:0")
    for variant in (_native.VARIANT_STAGED, _native.VARIANT_DIRECT):
        for kind, params, n_out, text in UNSUPPORTED_PAIRS:
            p, n_p = _params(params)
            rc = built.ctb_aggregate_ex(plan._h, x.data_ptr(), x.data_ptr(), _native.F32, _native.LAYOUT_TIME_MAJOR,
                                        ncell, None, T, kind, p, n_p, n_out, None, out.data_ptr(), 0, None, 0, variant,
                                        None)
            assert rc == _native.ERR_INVALID and text in _native.last_error(), (variant, kind, n_out)
    torch.cuda.synchronize()
    assert not out.any()


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_native, "_lib", None)
    monkeypatch.setattr(_native, "LIB_PATH", "/nonexistent/libctb.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _native.lib()


def test_no_cuda_no_fallback():
    import torch
    from climate_toolbox_b200 import _engine

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _engine.default_device()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "climate_toolbox_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle", src, flags=re.M), f
