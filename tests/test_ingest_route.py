"""Route selection of host inputs (``_engine._ingest_route``), tabled over every branch and precedence tie.

The precedence: CELL_MAJOR input; zero-copy (full-grid plan, a streaming variant, float32 / float64 inputs, all
pinned); the GPU pull (compact plan, ``ingest`` "auto" or "pull", float32 / float64, 16-byte aligned inputs and
planes on whole 4-cell pieces, all pinned); an ``ingest="pull"`` that cannot be met is an error; otherwise the host
pack on a compact plan and whole-chunk copies on a full-grid plan.  CPU only: the function reads plain values.
"""
import pytest

from climate_toolbox_b200 import _native as N
from climate_toolbox_b200._engine import _ingest_route

TM, CM = N.LAYOUT_TIME_MAJOR, N.LAYOUT_CELL_MAJOR
AUTO, STAGED, DIRECT, MAPPED = N.VARIANT_AUTO, N.VARIANT_STAGED, N.VARIANT_DIRECT, N.VARIANT_MAPPED_HOST

# layout, compact, variant, dtype_ok, aligned, pinned, zero_copy, ingest -> route
ROUTES = [
    # CELL_MAJOR comes first: not zero-copy, not pulled, and an unmeetable ingest="pull" is not an error
    ((CM, False, STAGED, True, True, True, True, "auto"), "cell_major"),
    ((CM, True, AUTO, True, True, True, False, "pull"), "cell_major"),
    ((CM, False, DIRECT, False, False, False, False, "pull"), "cell_major"),
    # zero-copy: full-grid plan, not the direct variant, float inputs, all pinned
    ((TM, False, STAGED, True, True, True, True, "auto"), "zero_copy"),
    ((TM, False, AUTO, True, False, True, True, "auto"), "zero_copy"),
    ((TM, False, STAGED | MAPPED, True, True, True, True, "pack"), "zero_copy"),
    ((TM, False, STAGED, True, False, True, True, "pull"), "zero_copy"),         # before the ingest="pull" error
    ((TM, False, DIRECT, True, True, True, True, "auto"), "full_copy"),
    ((TM, False, DIRECT | MAPPED, True, True, True, True, "auto"), "full_copy"),
    ((TM, False, STAGED, False, True, True, True, "auto"), "full_copy"),
    ((TM, False, STAGED, True, True, False, True, "auto"), "full_copy"),
    ((TM, False, STAGED, True, True, True, False, "auto"), "full_copy"),
    # zero-copy requested on a compact plan: pulled when it can be, else packed on the host
    ((TM, True, STAGED, True, True, True, True, "auto"), "pull"),
    ((TM, True, STAGED, True, True, True, True, "pack"), "host_pack"),
    ((TM, True, STAGED, True, True, False, True, "auto"), "host_pack"),
    # the pull: compact plan, ingest auto or pull, float inputs, aligned, all pinned; any variant
    ((TM, True, AUTO, True, True, True, False, "auto"), "pull"),
    ((TM, True, DIRECT, True, True, True, False, "pull"), "pull"),
    ((TM, True, STAGED, True, True, True, False, "pack"), "host_pack"),          # pinned, but packing asked for
    ((TM, True, AUTO, True, False, True, False, "auto"), "host_pack"),           # misaligned or a ragged grid
    ((TM, True, AUTO, True, True, False, False, "auto"), "host_pack"),           # pageable
    ((TM, True, AUTO, False, True, True, False, "auto"), "host_pack"),           # not float32 / float64
    # unknown ingest strings are neither a pull nor an error
    ((TM, True, AUTO, True, True, True, False, "bogus"), "host_pack"),
    ((TM, False, AUTO, True, True, True, False, "bogus"), "full_copy"),
    # full-grid plans copy whole chunks
    ((TM, False, AUTO, True, True, True, False, "auto"), "full_copy"),
    ((TM, False, AUTO, True, True, False, False, "pack"), "full_copy"),
]

# ingest="pull" that cannot be met
PULL_ERRORS = [
    (TM, False, AUTO, True, True, True, False, "pull"),                           # full-grid plan
    (TM, True, AUTO, True, False, True, False, "pull"),                           # misaligned
    (TM, True, AUTO, True, True, False, False, "pull"),                           # pageable
    (TM, True, AUTO, False, True, True, False, "pull"),                           # not float32 / float64
    (TM, False, DIRECT, True, True, True, True, "pull"),                          # zero-copy refused, full grid
]


@pytest.mark.parametrize("args,route", ROUTES)
def test_route(args, route):
    assert _ingest_route(*args) == route


@pytest.mark.parametrize("args", PULL_ERRORS)
def test_unmet_pull_is_an_error(args):
    with pytest.raises(ValueError, match="ingest='pull'"):
        _ingest_route(*args)


def test_table_reaches_every_route_and_input():
    assert {r for _, r in ROUTES} == {"cell_major", "zero_copy", "pull", "host_pack", "full_copy"}
    rows = [a for a, _ in ROUTES] + PULL_ERRORS
    assert len(set(rows)) == len(rows)
    for i in (1, 3, 4, 5, 6):
        assert {a[i] for a in rows} == {False, True}, i
    assert {a[2] for a in rows} == {AUTO, STAGED, DIRECT, STAGED | MAPPED, DIRECT | MAPPED}
    assert {a[7] for a in rows} == {"auto", "pull", "pack", "bogus"}


def test_environment_is_read_at_call_time(monkeypatch):
    zc = (TM, False, STAGED, True, True, True)
    pull = (TM, True, AUTO, True, True, True)
    monkeypatch.delenv("CTB_ZERO_COPY", raising=False)
    monkeypatch.delenv("CTB_INGEST", raising=False)
    assert _ingest_route(*zc, None, None) == "full_copy"          # zero-copy is opt-in
    assert _ingest_route(*pull, None, None) == "pull"             # ingest defaults to auto
    monkeypatch.setenv("CTB_ZERO_COPY", "1")
    monkeypatch.setenv("CTB_INGEST", "pack")
    assert _ingest_route(*zc, None, None) == "zero_copy"
    assert _ingest_route(*pull, None, None) == "host_pack"
    assert _ingest_route(*zc, False, None) == "full_copy"         # arguments win over the environment
    assert _ingest_route(*pull, None, "auto") == "pull"
    monkeypatch.setenv("CTB_INGEST", "pull")
    with pytest.raises(ValueError):
        _ingest_route(TM, False, AUTO, True, True, True, False, None)
    monkeypatch.setenv("CTB_ZERO_COPY", "0")
    assert _ingest_route(*zc, None, "auto") == "full_copy"

