"""Every aggregation kernel instantiation against a float64 reference at a derived tolerance.

The hot path is one templated kernel family: ``agg_stream_kernel`` (input type x transform x outputs x
growing-season gate x time index), ``agg_direct_kernel`` (input type x transform x outputs x layout) and the
pointwise ``transform_kernel`` behind ``.values``.  Every instantiation is separately compiled code -- its own
unrolling, register allocation and fast paths (the integer widening of float kelvin with its range check and
sticky probe, float-threshold decisions on the stored type, the producer's time-index plane loads) -- so each
one is launched here, and a CPU test keeps the case table equal to the set of kernels the library contains.

The reference restates the operation in float64: rows gathered by exact label, effective weight
``w > 0 ? w : backup``, ``f_j`` in float64 (``oracle.snyder_edd``, ``test_bins.bins_ref``,
``test_rcspline.rcs_ref``), skip-NaN products, the growing-season gate as a dense mask, each region-day summed
exactly (``math.fsum``) and divided by the float64 denominator.

The tolerance follows from the kernel's arithmetic.  A region-day with ``n_r`` kept rows sums ``n_r`` products
of one rounding each, in some order (at most ``n_r - 1`` roundings of partial sums no larger than
``sum |w f|``); ``f`` itself is within a few ulps of its scale; ``den`` is summed in another order and
inverted once.  With ``S_r = sum |w f| / den`` (``rcs_scale`` for the spline terms, ``|EDD_lo| + |EDD_hi|`` for
GDD) every aggregate must satisfy

    |got - ref| <= C_AGG * (n_r + 4) * 2^-53 * S_r  (+ 3e-14 * W_bar per Snyder evaluation)

where ``W_bar`` is the aggregated half-range ``sum |w| W / den``: the kernel's closed form of Snyder's
straddling case is exact to ``3e-14 * W`` (DESIGN.md section 2).  ``C_AGG`` is the smallest integer constant
that passes on a B200; the worst ratio seen per case is kept in ``NEEDED`` for reporting.  Pointwise results
must be within ``C_PT`` ulps of the same scales, with NaN, infinity and zero patterns exactly equal.

Known difference of the closed form: for float64 inputs a few ulps around a threshold the reference's
``arcsin`` can see ``|s| >= 1`` after rounding and give NaN, where the kernel clamps.  The fixture therefore never
pairs a ``tasmin`` and a ``tasmax`` that straddle a threshold within a few ulps; every other threshold-adjacent
case is covered.
"""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pandas as pd
import pytest

import oracle
from test_bins import _adjacent as _edge_adjacent
from test_bins import bins_ref
from test_rcspline import _adjacent as _knot_adjacent
from test_rcspline import rcs_ref, rcs_scale
from climate_toolbox_b200 import _native as N

OFF = 273.15
INF = np.inf
U = 2.0 ** -53
C_AGG = 1          # aggregates: |got - ref| <= C_AGG * (n_r + 4) * 2^-53 * S_r (+ Snyder term)
C_PT = 4           # pointwise: |got - ref| <= C_PT * 2^-53 * scale (+ Snyder term); the spline terms need 3.7
SNYDER_ABS = 3e-14
NEEDED = {}        # case -> worst |got - ref| / ((n_r + 4) 2^-53 S_r) seen (the c that case needs)

# ----------------------------------------------------------------------------
# the matrix as data
# ----------------------------------------------------------------------------
KNOTS3 = (0.0, 12.0, 25.0)
KNOTS5 = (-5.0, 5.0, 12.0, 20.0, 28.0)
KNOTS7 = (-10.0, 0.0, 5.0, 10.0, 15.0, 20.0, 30.0)
EDD_T = (283.15, 291.15, 300.15, 273.15)
GDD_P = ((281.15, 291.15), (283.15, 303.15), (291.15, 300.15), (273.15, 308.15))


def _rcs(knots, first):
    return (OFF, float(first)) + knots


# (kind, n_out, params of every variant run through that instantiation).  "poly" with orders 1..n is the
# streaming kernel's POLY_SEQ instantiation; any other orders take the generic POLY one.
TABLE = [
    ("identity", 1, [()]),
    ("poly_seq", 1, [(OFF, 1.0)]),
    ("poly_seq", 2, [(OFF, 1.0, 2.0)]),
    ("poly_seq", 3, [(OFF, 1.0, 2.0, 3.0)]),
    ("poly_seq", 4, [(OFF, 1.0, 2.0, 3.0, 4.0)]),
    ("poly", 1, [(OFF, 2.0), (OFF, 0.0), (OFF, -2.0)]),
    ("poly", 2, [(OFF, 0.0, 3.0), (OFF, 2.0, 1.0)]),
    ("poly", 3, [(OFF, 3.0, 1.0, -1.0)]),
    ("poly", 4, [(OFF, 4.0, 2.0, 3.0, 1.0)]),
    ("edd", 1, [EDD_T[:1], EDD_T[3:]]),
    ("edd", 2, [EDD_T[:2]]),
    ("edd", 3, [EDD_T[:3]]),
    ("edd", 4, [EDD_T]),
    ("gdd", 1, [GDD_P[0]]),
    ("gdd", 2, [sum(GDD_P[:2], ())]),
    ("gdd", 3, [sum(GDD_P[:3], ())]),
    ("gdd", 4, [sum(GDD_P, ())]),
    ("bins", 1, [(OFF, -INF, 10.0), (OFF, 20.0, INF)]),
    ("bins", 2, [(OFF, 0.0, 10.0, 20.0), (OFF, -INF, 10.0, INF)]),
    ("bins", 3, [(OFF, -INF, 5.0, 15.0, 25.0), (OFF, 0.0, 8.0, 16.0, INF)]),
    ("bins", 4, [(OFF, -INF, 0.0, 10.0, 20.0, 30.0), (OFF, 0.0, 10.0, 20.0, 30.0, INF)]),
    ("rcspline", 1, [_rcs(KNOTS3, 0), _rcs(KNOTS3, 1), _rcs(KNOTS5, 3), _rcs(KNOTS7, 5)]),
    ("rcspline", 2, [_rcs(KNOTS3, 0), _rcs(KNOTS5, 2), _rcs(KNOTS7, 4)]),
    ("rcspline", 3, [_rcs(KNOTS5, 0), _rcs(KNOTS5, 1), _rcs(KNOTS7, 3)]),
    ("rcspline", 4, [_rcs(KNOTS5, 0), _rcs(KNOTS7, 2)]),
]
DTYPES = (np.float32, np.float64)
PUBLIC = {"poly_seq": "poly"}   # the name aggregate_device takes
_CODE = {"identity": N.TR_IDENTITY, "poly": N.TR_POLY, "edd": N.TR_EDD, "gdd": N.TR_GDD, "bins": N.TR_BINS,
         "rcspline": N.TR_RCSPLINE}
POLY_SEQ = 16                   # the streaming kernel's internal kind (ctb_internal.cuh, CTB_TR_POLY_SEQ)


def _public(kind):
    return PUBLIC.get(kind, kind)


def _stream_kind(kind, params, n_out):
    """The kind of the streaming instantiation ``CTB_STREAM_ENTRY`` picks: POLY with orders 1..n is POLY_SEQ."""
    if kind in ("poly", "poly_seq") and tuple(params[1:]) == tuple(float(p) for p in range(1, n_out + 1)):
        return POLY_SEQ
    return _CODE[_public(kind)]


def _n_in(kind):
    return 2 if kind in ("edd", "gdd") else 1


def expected_instantiations():
    """(stream, direct, transform) key sets the table launches: stream (dtype, kind, n_out, gate, tix),
    direct (dtype, kind, n_out, layout), transform (dtype, kind, n_out); dtype 'f' / 'd'."""
    stream, direct, pointwise = set(), set(), set()
    for dt in "fd":
        for kind, n_out, variants in TABLE:
            for params in variants:
                sk = _stream_kind(kind, params, n_out)
                ck = _CODE[_public(kind)]
                for gate in (0, 1):
                    for tix in (0, 1):
                        stream.add((dt, sk, n_out, gate, tix))
                for layout in (N.LAYOUT_TIME_MAJOR, N.LAYOUT_CELL_MAJOR):
                    direct.add((dt, ck, n_out, layout))
                pointwise.add((dt, ck, n_out))
    return stream, direct, pointwise


def _cuobjdump():
    for d in (os.environ.get("CUDA_HOME"), os.path.dirname(os.environ.get("NVCC", "")) + "/..", "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "bin", "cuobjdump")):
            return os.path.join(d, "bin", "cuobjdump")
    return shutil.which("cuobjdump")


def built_instantiations(path):
    """The same key sets parsed from the (mangled) kernel symbols of the library."""
    exe = _cuobjdump()
    syms = subprocess.run([exe, "-symbols", path], check=True, capture_output=True, text=True).stdout
    stream = {(m[0], int(m[1]), int(m[2]), int(m[3]), int(m[4])) for m in set(re.findall(
        r"agg_stream_kernelI([fd])Li(\d+)ELi(\d+)ELi\d+ELi\d+ELb([01])ELb([01])EEEv7AggArgs", syms))}
    direct = {(m[0], int(m[1]), int(m[2]), int(m[3])) for m in set(re.findall(
        r"agg_direct_kernelI([fd])Li(\d+)ELi(\d+)ELi(\d+)EEEv7AggArgs", syms))}
    pointwise = {(m[0], int(m[1]), int(m[2])) for m in set(re.findall(
        r"transform_kernelI([fd])Li(\d+)ELi(\d+)EEEvPKT_", syms))}
    return stream, direct, pointwise, syms


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as G
    G.build()
    return N.lib()


def test_every_kernel_instantiation_has_a_case(built):
    """The case table launches exactly the kernels the library contains: a new instantiation without a case,
    or a case row without its kernel, fails here."""
    if _cuobjdump() is None:
        pytest.skip("cuobjdump not found")
    stream, direct, pointwise, syms = built_instantiations(N.LIB_PATH)
    assert syms.count("transform_kernel") == len(pointwise)          # every symbol parsed
    assert len(re.findall(r"agg_stream_kernelI", syms)) == len(stream)
    assert len(re.findall(r"agg_direct_kernelI", syms)) == len(direct)
    assert (len(stream), len(direct), len(pointwise)) == (200, 84, 42)
    e_stream, e_direct, e_pointwise = expected_instantiations()
    assert e_stream == stream, (sorted(stream - e_stream), sorted(e_stream - stream))
    assert e_direct == direct, (sorted(direct - e_direct), sorted(e_direct - direct))
    assert e_pointwise == pointwise, (sorted(pointwise - e_pointwise), sorted(e_pointwise - pointwise))


def test_table_rows_are_distinct_instantiations():
    """Each row reaches instantiations no other row does (so deleting one is seen), and every row's variants
    agree on the instantiation."""
    rows = {}
    for kind, n_out, variants in TABLE:
        keys = {(_stream_kind(kind, p, n_out), n_out) for p in variants}
        assert len(keys) == 1, (kind, n_out)
        rows[(kind, n_out)] = keys.pop()
    assert len(set(rows.values())) == len(TABLE) == 25
    assert {k for k, n in rows.values() if n == 1} == {0, 1, 2, 3, 4, 5, POLY_SEQ}


def test_numpy_and_the_kernel_agree_that_nan_to_the_zeroth_is_one():
    """``ctb_ipow(NaN, 0)`` is 1 (the loop multiplies nothing); numpy's power gives the same, so the reference's
    order-0 term of a NaN value is 1 and its product is not skipped."""
    with np.errstate(all="ignore"):
        assert np.power(np.float64(np.nan) - OFF, 0.0) == 1.0
        assert _f("poly", (OFF, 0.0, 3.0), 2, np.array([np.nan]), None)[0][:, 0].tolist()[0] == 1.0


# ----------------------------------------------------------------------------
# the reference
# ----------------------------------------------------------------------------
def _f(kind, params, n_out, x0, x1):
    """f_j of every value in float64: (F [n_out, ...], scale [n_out, ...], W or None)."""
    kind = _public(kind)
    a = np.asarray(x0).astype(np.float64)
    with np.errstate(all="ignore"):
        if kind == "identity":
            F = a[None]
            return F, np.abs(F), None
        if kind == "poly":
            d = a - params[0]
            F = np.stack([np.power(d, float(p)) for p in params[1:]])
            return F, np.abs(F), None
        if kind == "bins":
            F = np.stack([bins_ref(x0, params[1 + j], params[2 + j], params[0]) for j in range(n_out)])
            return F, np.abs(F), None
        if kind == "rcspline":
            first, knots = int(params[1]), tuple(params[2:])
            F = np.stack([rcs_ref(x0, knots, first + j, params[0]) for j in range(n_out)])
            S = np.stack([rcs_scale(x0, knots, first + j, params[0]) for j in range(n_out)])
            return F, S, None
        b = np.asarray(x1).astype(np.float64)
        W = np.abs((b - a) / 2)
        if kind == "edd":
            F = np.stack([oracle.snyder_edd(a, b, e) for e in params])
            return F, np.abs(F), W
        lo = np.stack([oracle.snyder_edd(a, b, params[2 * j]) for j in range(n_out)])
        hi = np.stack([oracle.snyder_edd(a, b, params[2 * j + 1]) for j in range(n_out)])
        return lo - hi, np.abs(lo) + np.abs(hi), W


def _xsum(v):
    """Exact sum (``math.fsum``); with infinities the plain IEEE sum (+inf + -inf = NaN)."""
    if np.isfinite(v).all():
        return math.fsum(v)
    return float(np.sum(v))


def reference(fx, kind, params, n_out, X0, X1, tix, gate_on, mutate=None):
    """Daily region aggregates in float64 and their tolerance scale.

    X0 / X1: [days, cells] time-major data; ``tix`` the physical day of every output day (None: identity);
    ``gate_on`` [T, cells] bool or None.  Returns (ref, bound_base, snyder) with the shape [n_out, R, T]:
    the allowed error is ``C_AGG * bound_base + snyder``.  ``mutate`` (the comparator's self-test) changes one
    thing about the computation."""
    mutate = mutate or {}
    days = np.arange(fx["T"]) if tix is None else np.asarray(tix)
    x0 = X0[days]
    x1 = None if X1 is None else X1[days]
    p = tuple(params)
    if mutate.get("f32_threshold"):
        p = (float(np.float32(p[0])),) + p[1:]
    F, S, W = _f(kind, p, n_out, x0, x1)
    evals = {"edd": 1, "gdd": 2}.get(kind, 0)
    T = len(days)
    R = fx["R"]
    ref = np.empty((n_out, R, T))
    base = np.empty((n_out, R, T))
    sny = np.zeros((n_out, R, T))
    for r in range(R):
        rows = fx["members"][r]
        cells, w = fx["row_cell"][rows], fx["w_eff"][rows]
        if mutate.get("drop_smallest") == r:
            keep_rows = np.ones(len(rows), bool)
            keep_rows[np.argmin(w)] = False
            cells_n, w_n = cells[keep_rows], w[keep_rows]
        elif mutate.get("add_padding") == r:
            cells_n, w_n = np.r_[cells, fx["pad_cell"]], np.r_[w, w[0]]
        else:
            cells_n, w_n = cells, w
        den = np.float64(math.fsum(w))
        n_r = len(rows)
        on = np.ones((T, len(cells_n)), bool) if gate_on is None else gate_on[:, cells_n]
        P = F[:, :, cells_n] * w_n
        keep = ~np.isnan(P) & on
        Pk = np.where(keep, P, 0.0)
        with np.errstate(all="ignore"):
            rden = np.float64(np.float32(1.0 / den))
            for j in range(n_out):
                for t in range(T):
                    num = np.float64(_xsum(Pk[j, t]))
                    ref[j, r, t] = num * rden if mutate.get("rden_f32") else num / den   # x/0 = +-inf, 0/0 = NaN
            absP = np.where(keep, np.abs(S[:, :, cells_n] * w_n), 0.0).sum(axis=2)
            base[:, r, :] = (n_r + 4) * U * absP / abs(den)
            if evals:
                onw = on & np.isfinite(W[:, cells_n])
                wbar = np.where(onw, np.abs(w_n) * W[:, cells_n], 0.0).sum(axis=1) / abs(den)
                sny[:, r, :] = evals * SNYDER_ABS * wbar[None, :]
    if mutate.get("shift_region") is not None:
        r = mutate["shift_region"]
        ref[:, r, :-1] = ref[:, r, 1:].copy()
    if mutate.get("swap_outputs"):
        ref[[0, 1]] = ref[[1, 0]]
    return ref, base, sny


def check(got, ref, base, sny, what, c=None):
    """NaN and infinity patterns exactly equal; elsewhere |got - ref| <= c * base + sny.  Records the c the case
    needs in NEEDED[what] and returns it."""
    c = C_AGG if c is None else c
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    nan_g, nan_r = np.isnan(got), np.isnan(ref)
    assert np.array_equal(nan_g, nan_r), "{}: NaN pattern differs at {}".format(
        what, np.argwhere(nan_g != nan_r)[:5].tolist())
    inf_r = np.isinf(ref) | np.isinf(got)
    assert np.array_equal(got[inf_r], ref[inf_r]), "{}: infinities differ at {}".format(
        what, np.argwhere(inf_r & (got != ref))[:5].tolist())
    m = np.isfinite(ref)
    err = np.abs(got[m] - ref[m]) - sny[m]
    with np.errstate(all="ignore"):
        need = np.where(err <= 0, 0.0, err / base[m])
    worst = float(need.max()) if need.size else 0.0
    NEEDED[what] = max(NEEDED.get(what, 0.0), worst)
    if worst > c:
        i = np.flatnonzero(m)[int(np.argmax(need))]
        idx = np.unravel_index(i, ref.shape)
        raise AssertionError("{}: |got - ref| = {:.3g} at [j, r, t] = {} exceeds {} * (n_r + 4) * 2^-53 * S_r + snyder "
                             "(needs c = {:.3g}; got {!r}, ref {!r})".format(
                                 what, abs(got[idx] - ref[idx]), tuple(int(v) for v in idx), c, worst,
                                 float(got[idx]), float(ref[idx])))
    return worst


# ----------------------------------------------------------------------------
# the fixture: a 12 x 40 grid whose regions carry the structures kernels get wrong
# ----------------------------------------------------------------------------
NLAT, NLON = 12, 40
NCELL = NLAT * NLON
T_PHYS, T = 80, 77
LAT = 0.5 + np.arange(NLAT)
LON = -19.5 + np.arange(NLON)
CELSIUS = np.arange(8 * NLON, 10 * NLON)                      # rows 8 and 9 hold whole regions in deg C
SIZES = (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 64, 65)   # every residue of the quad padding
TIX = np.r_[np.arange(0, 40), 39, np.arange(42, 78)]           # day 39 twice, days 40 and 41 removed
DOY = (350 + np.arange(T)) % 365 + 1                            # the day-of-year axis crosses a year end
GATES = (N.GATE_ALWAYS, N.GATE_NEVER, N.gate_word(355, 365, 0), N.gate_word(5, 40, 0), N.gate_word(10, 358, 1),
         N.gate_word(1, 20, 1))
SPECIAL_DAYS = np.arange(2, T_PHYS, 5)                          # one special cell-day per day at most


def _gate_on(words, doy):
    first, last, wrap = words & 511, (words >> 9) & 511, (words >> 18) & 1
    d = np.asarray(doy)[:, None]
    return ((d >= first[None]) & (d <= last[None])) != (wrap[None] == 1)


def _weights_fixture():
    rng = np.random.default_rng(2024)
    reserved = np.array([0, 1, 2])                            # the cancelling pair and the padding stand-in
    kelvin = np.setdiff1d(np.setdiff1d(np.arange(NCELL), CELSIUS), reserved)
    regions = []                                               # rows (cell, primary, backup) per region
    names = []

    def wts(n):
        # primary weight or a fallback to the backup (NaN, zero or negative primary); every kept weight lies
        # in [1, 1000): each entry matters far above the tolerance
        wp = rng.uniform(1.0, 1000.0, n)
        wb = rng.uniform(1.0, 1000.0, n)
        fall = rng.random(n) < 0.2
        wp[fall] = rng.choice([np.nan, 0.0, -3.0], fall.sum())
        return wp, wb

    for n in SIZES:
        cells = rng.choice(kelvin, n, replace=False)
        regions.append((cells,) + wts(n))
        names.append("size{}".format(n))
    dup = np.r_[[kelvin[7]] * 5, kelvin[[30, 31]]]             # duplicate rows of one cell
    regions.append((dup,) + wts(len(dup)))
    names.append("duplicates")
    res = kelvin[kelvin % 4 == 2][:12]                         # every quad in one residue class
    regions.append((res,) + wts(len(res)))
    names.append("one_residue")
    cel = rng.permutation(CELSIUS)
    for a, b in ((0, 6), (6, 19), (19, 39)):
        regions.append((cel[a:b],) + wts(b - a))
        names.append("celsius{}".format(b - a))
    regions.append((kelvin[[40, 41, 42]], np.full(3, np.nan), np.full(3, np.nan)))   # den = 0 -> NaN
    names.append("nan_weights")
    regions.append((kelvin[[50, 51]], np.zeros(2), np.zeros(2)))                     # no kept rows
    names.append("no_rows")
    regions.append((reserved[:2], np.array([0.0, -2.0]), np.array([1.0, -1.0])))    # den == 0 exactly
    names.append("cancel")
    # a region big enough to split over several bundles of the small-tile plan
    big = rng.choice(kelvin, 90, replace=False)
    regions.append((big,) + wts(90))
    names.append("big")
    rows_cell = np.concatenate([r[0] for r in regions])
    wp = np.concatenate([r[1] for r in regions])
    wb = np.concatenate([r[2] for r in regions])
    code = np.concatenate([np.full(len(r[0]), k) for k, r in enumerate(regions)])
    perm = rng.permutation(len(rows_cell))                   # table rows in no particular order
    rows_cell, wp, wb, code = rows_cell[perm], wp[perm], wb[perm], code[perm]
    ii, jj = np.divmod(rows_cell, NLON)
    df = pd.DataFrame({"lat": LAT[ii], "lon": LON[jj], "hierid": code, "popwt": wp, "areawt": wb})
    w_eff = oracle.effective_weights(df, "popwt", "areawt")
    members = [np.flatnonzero((code == r) & np.isfinite(w_eff) & (w_eff != 0)) for r in range(len(regions))]
    gate_words = np.asarray(rng.choice(GATES, NCELL), dtype=np.uint32)
    special_cells = rng.choice(np.setdiff1d(kelvin, np.concatenate([dup, [kelvin[30], kelvin[31]]])),
                               len(SPECIAL_DAYS), replace=False)
    return {"df": df, "row_cell": rows_cell.astype(np.int64), "w_eff": w_eff, "members": members,
            "R": len(regions), "names": names, "gate_words": gate_words, "kelvin": kelvin,
            "cancel": reserved[:2], "pad_cell": reserved[2], "special_cells": special_cells, "T": T}


FX = _weights_fixture()


def _pool(kind, params, dtype):
    """Values next to every edge, knot and threshold of the case, in ``dtype``."""
    kind = _public(kind)
    if kind == "bins":
        return np.concatenate([_edge_adjacent(e, dtype) for e in params[1:] if np.isfinite(e)])
    if kind == "rcspline":
        return np.concatenate([_knot_adjacent(k, dtype) for k in params[2:]])
    if kind in ("edd", "gdd"):
        out = []
        for e in params:
            x = dtype(e)
            out += [np.nextafter(x, dtype(-INF)), x, np.nextafter(x, dtype(INF))]
            out += list(_knot_adjacent(e - OFF, dtype))
        return np.array(out, dtype=dtype)
    return np.array([dtype(OFF), np.nextafter(dtype(OFF), dtype(INF))], dtype=dtype)


def _specials(dtype):
    fi = np.finfo(np.float32)
    sub = np.finfo(dtype).smallest_subnormal * 3
    return np.array([np.nan, INF, -INF, 0.0, -0.0, sub, fi.tiny, fi.max, OFF, -fi.max], dtype=dtype)


def _edd_specials(e, dtype):
    """(tasmin, tasmax) pairs: NaN in either, infinities, zeros, tasmin == tasmax on and off the threshold,
    either end exactly on it."""
    fi = np.finfo(np.float32)
    sub = np.finfo(dtype).smallest_subnormal * 3
    x = dtype(e)
    pairs = [(np.nan, 290.0), (280.0, np.nan), (np.nan, np.nan), (-INF, 290.0), (280.0, INF), (INF, INF),
             (-INF, -INF), (0.0, 0.0), (-0.0, 0.0), (sub, sub), (fi.tiny, fi.max), (x, x), (x, x + 5), (x - 5, x),
             (290.0, 290.0)]
    return np.array(pairs, dtype=dtype)


def make_data(kind, params, n_out, dtype, seed):
    """[T_PHYS, NCELL] time-major inputs (x1 None for one-input transforms): kelvin, deg C regions, edge- and
    threshold-adjacent values, one special cell-day per day, the cancelling pair 0.75 K apart."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(250.0, 320.0, (T_PHYS, NCELL))
    x[:, CELSIUS] = rng.uniform(-20.0, 35.0, (T_PHYS, len(CELSIUS)))
    x = x.astype(dtype)
    pool = _pool(kind, params, dtype)
    kel = FX["kelvin"]
    pick = rng.random((T_PHYS, len(kel))) < 0.25
    vals = rng.choice(pool, (T_PHYS, len(kel)))
    sub = x[:, kel]
    sub[pick] = vals[pick]
    x[:, kel] = sub
    a, b = FX["cancel"]
    x[:, a] = rng.uniform(280.0, 300.0, T_PHYS).astype(dtype)
    x[:, b] = x[:, a] + dtype(0.75)
    if _n_in(kind) == 1:
        for d, c in zip(SPECIAL_DAYS, FX["special_cells"]):
            x[d, c] = rng.choice(_specials(dtype))
        return x, None
    # two inputs: tasmin = x - s, tasmax = x + s.  A threshold-adjacent value is ONE end of its pair, the other
    # end at least 0.5 K away (a pair straddling a threshold within ulps is the closed form's known difference)
    s = rng.uniform(0.5, 8.0, (T_PHYS, NCELL)).astype(dtype)
    lo, hi = x - s, x + s
    sub_lo, sub_hi, sub_s = lo[:, kel], hi[:, kel], s[:, kel]
    as_lo = pick & (rng.random(pick.shape) < 0.5)
    as_hi = pick & ~as_lo
    sub_lo[as_lo] = vals[as_lo]
    sub_hi[as_lo] = vals[as_lo] + 2 * sub_s[as_lo]
    sub_hi[as_hi] = vals[as_hi]
    sub_lo[as_hi] = vals[as_hi] - 2 * sub_s[as_hi]
    lo[:, kel], hi[:, kel] = sub_lo, sub_hi
    for d, c in zip(SPECIAL_DAYS, FX["special_cells"]):
        sp = _edd_specials(params[0], dtype)
        lo[d, c], hi[d, c] = sp[rng.integers(len(sp))]
    assert not (hi < lo).any()
    return lo, hi


def _case_seed(dtype, kind, n_out, v):
    return 1000 * (1 + DTYPES.index(dtype)) + 100 * [k for k, _, _ in TABLE].index(kind) + 10 * n_out + v


# ----------------------------------------------------------------------------
# the comparator rejects every mutant (CPU)
# ----------------------------------------------------------------------------
def _mutation_case(kind, params, n_out):
    x0, x1 = make_data(kind, params, n_out, np.float64, 7)
    gate = _gate_on(FX["gate_words"], DOY)
    ref, base, sny = reference(FX, kind, params, n_out, x0, x1, TIX, gate)
    return x0, x1, gate, ref, base, sny


def test_comparator_accepts_the_reference_and_rejects_every_mutant():
    big = FX["names"].index("size65")
    cases = {"poly": ("poly_seq", (OFF, 1.0, 2.0), 2), "edd": ("edd", EDD_T[2:3], 1)}
    prepared = {k: _mutation_case(*v) for k, v in cases.items()}
    mutants = [("poly", {"drop_smallest": big}), ("poly", {"add_padding": big}), ("poly", {"shift_region": big}),
               ("poly", {"swap_outputs": True}), ("poly", {"rden_f32": True}), ("edd", {"f32_threshold": True})]
    for name, (kind, params, n_out) in cases.items():
        x0, x1, gate, ref, base, sny = prepared[name]
        assert np.isfinite(ref).mean() > 0.7
        check(ref, ref, base, sny, "self")
    for name, mutation in mutants:
        kind, params, n_out = cases[name]
        x0, x1, gate, ref, base, sny = prepared[name]
        bad, _, _ = reference(FX, kind, params, n_out, x0, x1, TIX, gate, mutate=mutation)
        with pytest.raises(AssertionError):
            check(bad, ref, base, sny, "mutant")
    NEEDED.pop("mutant", None)
    NEEDED.pop("self", None)


def test_fixture_covers_the_structures():
    sizes = [len(m) for m in FX["members"]]
    for n in SIZES:
        assert n in sizes
    assert {s % 4 for s in sizes} == {0, 1, 2, 3}
    r_nan, r_none, r_cancel = (FX["names"].index(k) for k in ("nan_weights", "no_rows", "cancel"))
    assert sizes[r_nan] == 0 and sizes[r_none] == 0 and sizes[r_cancel] == 2
    assert math.fsum(FX["w_eff"][FX["members"][r_cancel]]) == 0.0
    gate = _gate_on(FX["gate_words"], DOY)
    assert gate.any() and not gate.all() and (DOY[1:] < DOY[:-1]).any()
    assert len(np.unique(TIX)) == T - 1 and T % 32 != 0


# ----------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------
_PLANS = {}


def _plan(dtype, n_in, split):
    from climate_toolbox_b200 import _engine as E
    import torch
    key = (np.dtype(dtype).itemsize, n_in, split)
    if key not in _PLANS:
        es = key[0]
        stage = n_in * es
        budget = 33 * stage * 16 if split else 0            # 16 cells per bundle: the big regions split
        p = E.get_plan(E.GridSpec(LAT, LON), FX["df"], "popwt", "hierid", stage_bytes=stage,
                       device=torch.device("cuda", 0), smem_budget=budget, cache=False, elem_bytes=es,
                       cell_gate=FX["gate_words"])
        if split:
            i = p.info
            assert i["n_split_regions"] > 0 and i["n_scratch_slots"] > 2 * i["n_split_regions"], i
        _PLANS[key] = p
    return _PLANS[key]


def _run(plan, kind, params, n_out, x0, x1, layout, variant, gate, tix, **kw):
    from climate_toolbox_b200 import _engine as E
    stride = NCELL if layout == N.LAYOUT_TIME_MAJOR else T_PHYS
    return E.aggregate_device(plan, x0, x1, layout, stride, TIX if tix else None, T, _public(kind), params, n_out,
                              variant=variant, doy=DOY if gate else None, **kw)


MATRIX = [(dt, kind, n_out) for dt in DTYPES for kind, n_out, _ in TABLE]


def _variants(kind, n_out):
    return next(v for k, n, v in TABLE if (k, n) == (kind, n_out))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,kind,n_out", MATRIX,
                         ids=["{}-{}-{}".format(np.dtype(d).name, k, n) for d, k, n in MATRIX])
def test_kernel_matrix(dtype, kind, n_out):
    """One (input type, transform, outputs) cell of the matrix: every params variant through the streaming
    kernel (gate x time index, whole and small-tile plans), the direct kernel (time-major and cell-major),
    time groups over two windows, the peer epilogue, and the pointwise kernel."""
    import torch
    dev = torch.device("cuda", 0)
    n_in = _n_in(kind)
    plan, split = _plan(dtype, n_in, False), _plan(dtype, n_in, True)
    for v, params in enumerate(_variants(kind, n_out)):
        name = "{}/{}/{}/{}".format(np.dtype(dtype).name, kind, n_out, params)
        x0, x1 = make_data(kind, params, n_out, dtype, _case_seed(dtype, kind, n_out, v))
        d0 = torch.from_numpy(x0).to(dev)
        d1 = None if x1 is None else torch.from_numpy(x1).to(dev)
        c0 = torch.from_numpy(np.ascontiguousarray(x0.T)).to(dev)
        c1 = None if x1 is None else torch.from_numpy(np.ascontiguousarray(x1.T)).to(dev)
        gate_dense = _gate_on(FX["gate_words"], DOY)
        refs = {}
        for gate in (False, True):
            for tix in (False, True):
                ref, base, sny = reference(FX, kind, params, n_out, x0, x1, TIX if tix else None,
                                           gate_dense if gate else None)
                refs[(gate, tix)] = (ref, base, sny)
                runs = (("stream", plan, d0, d1, N.LAYOUT_TIME_MAJOR, N.VARIANT_STAGED),
                        ("stream_split", split, d0, d1, N.LAYOUT_TIME_MAJOR, N.VARIANT_STAGED),
                        ("direct", plan, d0, d1, N.LAYOUT_TIME_MAJOR, N.VARIANT_DIRECT),
                        ("direct_cell_major", plan, c0, c1, N.LAYOUT_CELL_MAJOR, N.VARIANT_DIRECT))
                for label, p, a0, a1, layout, variant in runs:
                    got = _run(p, kind, params, n_out, a0, a1, layout, variant, gate, tix).cpu().numpy()
                    check(got, ref, base, sny, "{} {} gate={} tix={}".format(name, label, int(gate), int(tix)))
        _check_groups(name, split, kind, params, n_out, d0, d1, refs[(True, True)])
        if v == 0:
            _check_peers(name, split, kind, params, n_out, d0, d1)
        _check_pointwise(name, dtype, kind, params, n_out, dev)


GROUP_LEN = 10                   # groups shorter than a tile: a 32-day tile touches up to 4 of them
WINDOWS = ((0, 64), (64, T))     # t_begin a multiple of 32


def _check_groups(name, plan, kind, params, n_out, d0, d1, daily):
    """The fused time reduction over two input windows (flush on the last), gated with a time index, against the
    group sums of the daily reference; streaming and direct kernel."""
    from climate_toolbox_b200 import _engine as E
    import torch
    god = np.arange(T) // GROUP_LEN
    groups = E.get_time_groups(god, plan.device)
    ref_d, base_d, sny_d = daily
    n_g = int(god[-1]) + 1
    ref = np.zeros((n_out, plan.R, n_g))
    base = np.zeros_like(ref)
    sny = np.zeros_like(ref)
    for g in range(n_g):
        days = god == g
        ref[:, :, g] = ref_d[:, :, days].sum(axis=2)        # a plain sum: NaN and infinities propagate
        # the daily bounds add, and summing len(g) rounded daily values costs len(g) roundings of their sum
        base[:, :, g] = base_d[:, :, days].sum(axis=2) + (days.sum() + 4) * U * np.abs(ref_d[:, :, days]).sum(axis=2)
        sny[:, :, g] = sny_d[:, :, days].sum(axis=2)
    for label, variant in (("stream", N.VARIANT_STAGED), ("direct", N.VARIANT_DIRECT)):
        ws = E._workspace(plan, T, n_out, N.LAYOUT_TIME_MAJOR, variant, groups, None)
        out = torch.full((n_out, plan.R, n_g), -7.0, dtype=torch.float64, device=plan.device)
        for t0, t1 in WINDOWS:
            E.aggregate_device(plan, d0, d1, N.LAYOUT_TIME_MAJOR, NCELL, TIX[t0:t1], t1 - t0, _public(kind), params,
                               n_out, variant=variant, out=out, workspace=ws, groups=groups, t_begin=t0,
                               flush=(t1 == T), doy=DOY)
        with np.errstate(all="ignore"):
            check(out.cpu().numpy(), ref, base, sny, "{} groups {}".format(name, label))


def _check_peers(name, plan, kind, params, n_out, d0, d1):
    """The epilogue that stores to several buffers (peer_out, peer_row) writes what the plain launch writes, bit
    for bit, split regions included; streaming and direct kernel."""
    from climate_toolbox_b200 import _engine as E
    import torch
    row = torch.as_tensor(plan.region_order(), device=plan.device)
    t_total, t0 = T + 21, 13
    for label, variant in (("stream", N.VARIANT_STAGED), ("direct", N.VARIANT_DIRECT)):
        plain = _run(plan, kind, params, n_out, d0, d1, N.LAYOUT_TIME_MAJOR, variant, True, True)
        bufs = [torch.full((n_out, plan.R, t_total), -5.0, device=plan.device, dtype=torch.float64) for _ in range(2)]
        _run(plan, kind, params, n_out, d0, d1, N.LAYOUT_TIME_MAJOR, variant, True, True,
             out=E._OffsetOut(bufs[0], t0), out_ld=t_total, peer_ptrs=[b.data_ptr() + 8 * t0 for b in bufs],
             peer_row=row)
        torch.cuda.synchronize()
        want = plain.cpu().numpy().view(np.int64)
        rows = row.cpu().numpy()
        for b in bufs:
            h = b.cpu().numpy()
            assert np.array_equal(h[:, rows, t0:t0 + T].view(np.int64), want), "{} peers {}".format(name, label)
            assert (h[:, :, :t0] == -5.0).all() and (h[:, :, t0 + T:] == -5.0).all()


def _check_pointwise(name, dtype, kind, params, n_out, dev):
    """ctb_transform (the transform_kernel of this cell) on the adjacent and special pools: within C_PT ulps of
    the scale, NaN, infinity and zero patterns exact."""
    from climate_toolbox_b200 import _engine as E
    import torch
    if _n_in(kind) == 1:
        x0 = np.concatenate([_pool(kind, params, dtype), _specials(dtype),
                             np.linspace(230.0, 330.0, 101).astype(dtype)])
        x1 = None
    else:
        pool = _pool(kind, params, dtype)
        sp = np.concatenate([_edd_specials(e, dtype) for e in params])
        lo = np.r_[pool, pool - dtype(3.0), sp[:, 0]].astype(dtype)
        hi = np.r_[pool + dtype(3.0), pool, sp[:, 1]].astype(dtype)
        x0, x1 = lo, hi
    n = len(x0)
    t0 = torch.from_numpy(x0).to(dev)
    t1 = None if x1 is None else torch.from_numpy(x1).to(dev)
    out = torch.empty((n_out, n), dtype=torch.float64, device=dev)
    pa = np.ascontiguousarray(params, dtype=np.float64)
    rc = N.lib().ctb_transform(C.c_void_p(t0.data_ptr()), C.c_void_p(t1.data_ptr()) if t1 is not None else None,
                               N.F32 if dtype == np.float32 else N.F64, n, _CODE[_public(kind)],
                               pa.ctypes.data_as(C.POINTER(C.c_double)) if pa.size else None, int(pa.size), n_out,
                               C.c_void_p(out.data_ptr()), E._stream_ptr(dev))
    N.check(rc)
    got = out.cpu().numpy()
    F, S, W = _f(kind, params, n_out, x0, x1)
    what = "{} pointwise".format(name)
    evals = {"edd": 1, "gdd": 2}.get(_public(kind), 0)
    sny = np.zeros_like(F) if W is None else np.broadcast_to(evals * SNYDER_ABS * W, F.shape)
    check(got, F, U * S, np.nan_to_num(sny), what, c=C_PT)
    # zeros: exactly where the reference is zero, except rounding noise of a cancelling spline term
    zg, zr = got == 0, F == 0
    if _public(kind) == "rcspline":
        noise = np.abs(F) <= C_PT * U * S
        assert np.array_equal(zg & ~noise, zr & ~noise), what
        assert (got[zr & (S == 0)] == 0).all(), what
    elif evals:
        assert (got[zr & (W == 0)] == 0).all() and (F[zg] == 0).all(), what
    else:
        assert np.array_equal(zg, zr), what


@pytest.mark.gpu
@pytest.mark.parametrize("kind,params,n_out", [("identity", (), 1), ("poly", (OFF, 1.0, 2.0, 3.0, 4.0), 4)])
def test_scheduler_many_units_and_repeated_launches(kind, params, n_out):
    """A shape whose work units (bundles x chunks of several 32-day tiles) outnumber the SMs, against the
    reference; then one launch repeated more often than there are work-counter slots, bit for bit.  The
    reference here sums in float64 (vectorised over 3,000 regions x 1,100 days), so its own rounding,
    ``(n_r - 1) * 2^-53 * S_r``, joins the bound."""
    import torch
    from climate_toolbox_b200 import _engine as E
    from climate_toolbox_b200 import synthetic
    dev = torch.device("cuda", 0)
    d, R, TT = 1.0, 3000, 1100
    lat, lon = synthetic.grid_labels(d)
    df = synthetic.weights_table(d, R, seed=11)
    tas, _, _ = synthetic.tas_field(TT, len(lat), len(lon), seed=5, nan_frac=0.001)
    x = torch.from_numpy(tas).to(dev).view(TT, -1)
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev, cache=False)
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    n_tb = -(-TT // 32)
    chunk = max(1, min(8, plan.info["n_bundles"] * n_tb // (n_sm * 6)))
    n_units = plan.info["n_bundles"] * -(-n_tb // chunk)
    assert chunk > 1 and n_units > n_sm, (chunk, n_units, n_sm)
    got = E.aggregate_device(plan, x, None, N.LAYOUT_TIME_MAJOR, x.shape[1], None, TT, kind, params, n_out)
    w = oracle.effective_weights(df, "popwt", "areawt")
    codes, _ = E.region_codes(df["hierid"].values)
    cells = plan.row_cells()
    keep = np.isfinite(w) & (w != 0)
    order = np.argsort(codes[keep], kind="stable")
    rows = np.flatnonzero(keep)[order]
    starts = np.flatnonzero(np.r_[True, codes[rows][1:] != codes[rows][:-1]])
    present = codes[rows][starts]
    n_r = np.zeros(plan.R)
    n_r[present] = np.diff(np.r_[starts, len(rows)])
    den = np.zeros(plan.R)
    den[present] = np.add.reduceat(w[rows], starts)
    out = got.cpu().numpy()
    xg = tas.reshape(TT, -1)[:, cells[rows]]
    for j in range(n_out):
        pj = params if kind == "identity" else (params[0], params[1 + j])
        F, S, _ = _f(kind, pj, 1, xg, None)
        P = F[0] * w[rows]
        nan = np.isnan(P)
        num = np.zeros((TT, plan.R))
        sc = np.zeros((TT, plan.R))
        num[:, present] = np.add.reduceat(np.where(nan, 0.0, P), starts, axis=1)
        sc[:, present] = np.add.reduceat(np.where(nan, 0.0, np.abs(S[0] * w[rows])), starts, axis=1)
        del F, S, P, nan
        with np.errstate(all="ignore"):
            ref = (num / den).T
            base = ((C_AGG * (n_r + 4) + n_r + 1) * U * sc / np.abs(den)).T
        check(out[j], ref, base / C_AGG, np.zeros_like(ref), "scheduler {} {}".format(kind, j))
    for i in range(40):
        again = E.aggregate_device(plan, x, None, N.LAYOUT_TIME_MAJOR, x.shape[1], None, TT, kind, params, n_out)
        assert torch.equal(again.view(torch.int64), got.view(torch.int64)), i
    plan.close()
