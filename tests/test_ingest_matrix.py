"""Every way data reaches the aggregation kernels, bit for bit against the device-resident full-grid launch.

``test_kernel_matrix.py`` ties the device-resident launch on a full-grid plan to a float64 reference at a derived
bound.  Host data mostly reaches the same kernels another way: a compact plan whose packed planes hold only the
referenced 4-cell pieces, filled by ``ctb_pull_pack`` (pinned or device source), ``ctb_host_pack`` (pageable
source, pinned double buffers) or ``ctb_pull_pack_daily`` (sub-daily source); or a full-grid plan fed whole time
chunks, or read in place (zero-copy).  Each route cuts the time axis into chunks and slices the time index, the
day-of-year axis and the output per chunk, or opens time-group windows.

The oracle is bit identity.  A compact plan and a full-grid plan built with the same options hold the same
bundles: region centroids and the Hilbert order are computed before the compact renumbering, which maps pieces
one-to-one and monotonically and keeps ``col % 4``, so every split, sort and quad of the planner sees the same
keys, and entry offsets are bundle-local.  Each region-day is therefore summed in the same order from the same
values, and every route that feeds a kernel variant must give the bits of the device-resident launch of that
variant.  The baseline of every case is checked once against the float64 reference at ``C_AGG``, so identity
carries the kernel matrix's guarantee to every route with no tolerance to argue about.

Output buffers are pre-filled with a NaN of a payload no kernel produces, so an unwritten column fails, and
results are compared as int64, so NaN payloads and signed zeros count.
"""
import contextlib
import ctypes as C

import numpy as np
import pandas as pd
import pytest

from climate_toolbox_b200 import _native as N
from test_kernel_matrix import (C_AGG, DOY, EDD_T, FX, INF, LAT, LON, NCELL, NLAT, NLON, OFF, T_PHYS, TIX, U,
                                _gate_on, _n_in, check, make_data, reference)

SENT64 = np.int64(0x7FF4DEAD0000BEEF)      # output sentinel: a signalling NaN with a payload
SENT32 = np.int32(0x5A5A5A5A)              # packed-plane sentinel word (f32 and both words of f64)
NAN32 = np.array([0x7FC00123, 0xFFC00456], dtype=np.uint32).view(np.float32)            # NaNs with payloads
NAN64 = np.array([0x7FF8000000000123, 0xFFF8000000000456], dtype=np.uint64).view(np.float64)
GROUP_LEN = 10
CHUNK = 32                                  # the smallest time chunk of the chunked routes (chunk_bytes=1)
_ITYPE = {4: np.int32, 8: np.int64}


# ----------------------------------------------------------------------------
# the packed layout, restated
# ----------------------------------------------------------------------------
def packed_layout(cells):
    """Physical piece of every packed piece (-1: alignment padding) of a compact plan whose kept rows reference
    ``cells``: the sorted distinct 4-cell pieces, each run of consecutive pieces starting on a multiple of 4
    packed pieces, the plane padded to a multiple of 4 pieces (``plan_build_impl``, ``ctb_plan.cu``)."""
    pieces = np.unique(np.asarray(cells, dtype=np.int64) // 4)
    src = []
    for k, p in enumerate(pieces):
        if k == 0 or p != pieces[k - 1] + 1:
            src += [-1] * (-len(src) % 4)
        src.append(int(p))
    src += [-1] * (-len(src) % 4)
    return np.array(src, dtype=np.int64)


def packed_ref(x, src, days):
    """What packing writes: [len(days), 4 len(src)] with day ``days[d]`` of ``x`` [t, ncell] at every referenced
    piece (cells past the end of a ragged grid read as 0) and 0 in padding; and the padding mask per cell."""
    x = np.asarray(x)
    ncell = x.shape[1]
    xz = np.zeros((len(days), -(-ncell // 4) * 4), dtype=x.dtype)
    xz[:, :ncell] = x[np.asarray(days)]
    pad = np.repeat(src < 0, 4)
    cols = (np.maximum(src, 0)[:, None] * 4 + np.arange(4)).ravel()
    exp = xz[:, cols]
    exp[:, pad] = 0
    return exp, pad


def host_pack_zeroed(src, itemsize):
    """Padding cells the streaming-store path of ``ctb_host_pack`` writes: from the end of every run to the
    next 64-byte boundary of the packed plane."""
    z = np.zeros(4 * len(src), dtype=bool)
    k = 0
    while k < len(src):
        if src[k] < 0:
            k += 1
            continue
        e = k
        while e < len(src) and src[e] >= 0 and (e == k or src[e] == src[e - 1] + 1):
            e += 1
        end = 4 * e * itemsize
        z[4 * e: -(-end // 64) * 64 // itemsize] = True
        k = e
    return z


def plane_expected(x, src, days, sentinel_pad, zeroed=None):
    """Expected packed planes as integer words: referenced pieces from ``x``, padding holding the sentinel
    (``sentinel_pad``) or 0 where ``zeroed``, or 0 everywhere (``sentinel_pad=False``)."""
    exp, pad = packed_ref(x, src, days)
    it = _ITYPE[exp.dtype.itemsize]
    w = exp.view(it).copy()
    if sentinel_pad:
        s = SENT32.astype(np.int64) * 0x100000001 if it == np.int64 else SENT32
        w[:, pad] = it(s)
        if zeroed is not None:
            w[:, pad & zeroed] = 0
    return w


# ----------------------------------------------------------------------------
# comparators
# ----------------------------------------------------------------------------
def same_bits(got, want, what):
    """``got`` and ``want`` hold the same bits; a value still holding the output sentinel is named as unwritten."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    it = _ITYPE[got.dtype.itemsize]
    g, w = got.view(it), want.view(it)
    if got.dtype == np.float64:
        assert not (g == SENT64).any(), "{}: unwritten values at {}".format(what, np.argwhere(g == SENT64)[:5].tolist())
    bad = g != w
    assert not bad.any(), "{}: {} of {} values differ, first at {}: got {!r}, want {!r}".format(
        what, int(bad.sum()), bad.size, np.argwhere(bad)[0].tolist(), got[bad][0], want[bad][0])


def same_bits_except_nan(got, want, what):
    """The same bits except that a NaN may carry another payload: NaN positions equal, the rest bit for bit."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), "{}: NaN positions differ at {}".format(what, np.argwhere(gn != wn)[:5].tolist())
    it = _ITYPE[got.dtype.itemsize]
    assert np.array_equal(got.view(it)[~gn], want.view(it)[~wn]), "{}: non-NaN values differ".format(what)


def one_step_mean(a):
    """What the daily mean of one step makes of a value: ``0 + x`` turns -0.0 into +0.0; a NaN (whose payload
    the comparison ignores) stays NaN."""
    b = np.array(a, dtype=np.float64, copy=True)
    b[b == 0] = 0.0
    return b


# ----------------------------------------------------------------------------
# fixtures of any length
# ----------------------------------------------------------------------------
def tix_of(T):
    """A time index of T days with a duplicate day and a two-day gap (T >= 3), like ``TIX``."""
    if T == 77:
        return TIX
    if T < 3:
        return np.arange(T) + 2
    h = T // 2
    return np.r_[np.arange(0, h), h - 1, np.arange(h + 2, T + 1)]


def doy_of(T):
    """Day of year of T days starting at day 351: crosses a year end like ``DOY``."""
    return (350 + np.arange(T)) % 365 + 1


def long_data(kind, params, n_out, dtype, seed, t_phys):
    """``make_data`` on a longer time axis: consecutive 80-day blocks of the fixture's recipe."""
    blocks = [make_data(kind, params, n_out, dtype, seed + 7919 * b) for b in range(-(-t_phys // T_PHYS))]
    x0 = np.ascontiguousarray(np.concatenate([b[0] for b in blocks])[:t_phys])
    x1 = None if blocks[0][1] is None else np.ascontiguousarray(np.concatenate([b[1] for b in blocks])[:t_phys])
    return x0, x1


def group_reference(daily, T):
    """Sums of the daily reference over groups of GROUP_LEN days and their bound (as ``_check_groups``)."""
    ref_d, base_d, sny_d = daily
    god = np.arange(T) // GROUP_LEN
    n_g = int(god[-1]) + 1
    ref, base, sny = (np.zeros(ref_d.shape[:2] + (n_g,)) for _ in range(3))
    for g in range(n_g):
        days = god == g
        ref[:, :, g] = ref_d[:, :, days].sum(axis=2)
        base[:, :, g] = base_d[:, :, days].sum(axis=2) + (days.sum() + 4) * U * np.abs(ref_d[:, :, days]).sum(axis=2)
        sny[:, :, g] = sny_d[:, :, days].sum(axis=2)
    return ref, base, sny


# ----------------------------------------------------------------------------
# the route x feature matrix as data
# ----------------------------------------------------------------------------
KINDS = {"identity": ("identity", (), 1), "poly4": ("poly", (OFF, 1.0, 2.0, 3.0, 4.0), 4),
         "edd2": ("edd", EDD_T[:2], 2), "bins4": ("bins", (OFF, -INF, 0.0, 10.0, 20.0, 30.0), 4)}
ROUTES = ("device_packed", "pull", "host_pack", "full_pinned", "full_pageable", "zero_copy", "direct_compact",
          "cell_major")
LENGTHS = (1, 31, 32, 33, 77, 600)
F32, F64 = np.float32, np.float64

# route, input type, transform, time index, gate, time groups, split-region plan, days
ROWS = [
    ("device_packed", F32, "identity", 1, 1, 0, 0, 77),
    ("device_packed", F64, "edd2", 1, 0, 1, 1, 77),
    ("device_packed", F32, "bins4", 0, 1, 0, 1, 33),
    ("device_packed", F64, "poly4", 1, 1, 0, 0, 600),
    ("pull", F32, "identity", 1, 1, 0, 0, 600),
    ("pull", F64, "poly4", 1, 1, 0, 0, 77),
    ("pull", F32, "edd2", 1, 1, 1, 1, 77),
    ("pull", F64, "bins4", 0, 0, 0, 1, 1),
    ("pull", F32, "poly4", 0, 1, 0, 0, 32),
    ("pull", F64, "identity", 1, 0, 1, 0, 600),
    ("pull", F64, "edd2", 1, 1, 0, 0, 31),
    ("host_pack", F32, "identity", 1, 1, 0, 0, 600),
    ("host_pack", F64, "edd2", 1, 1, 0, 1, 77),
    ("host_pack", F32, "bins4", 1, 0, 1, 0, 77),
    ("host_pack", F64, "poly4", 0, 1, 1, 1, 31),
    ("host_pack", F32, "edd2", 0, 0, 0, 0, 1),
    ("host_pack", F64, "identity", 1, 1, 1, 0, 33),
    ("full_pinned", F32, "poly4", 1, 1, 0, 0, 77),
    ("full_pinned", F64, "identity", 0, 1, 1, 1, 600),
    ("full_pageable", F64, "bins4", 1, 1, 0, 0, 600),
    ("full_pageable", F32, "edd2", 1, 0, 1, 1, 33),
    ("zero_copy", F32, "edd2", 1, 1, 0, 1, 77),
    ("zero_copy", F64, "poly4", 1, 1, 1, 0, 77),
    ("direct_compact", F32, "bins4", 1, 1, 0, 0, 77),
    ("direct_compact", F64, "edd2", 1, 1, 1, 0, 77),
    ("cell_major", F32, "identity", 1, 1, 0, 0, 77),
    ("cell_major", F64, "edd2", 1, 1, 1, 0, 33),
]


def _row_id(row):
    route, dt, kind, tix, gate, groups, split, T = row
    return "{}-{}-{}-T{}{}{}{}{}".format(route, np.dtype(dt).name, kind, T, "-tix" if tix else "",
                                         "-gate" if gate else "", "-groups" if groups else "",
                                         "-split" if split else "")


def _baseline_variant(route):
    return {"direct_compact": "direct", "cell_major": "cell_major"}.get(route, "stream")


# ----------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------
def test_layout_rule_on_hand_made_cells():
    assert packed_layout([0, 1, 2, 3]).tolist() == [0, -1, -1, -1]
    # runs 1..3 and 7: the second run starts on the next multiple of 4 packed pieces
    assert packed_layout([4, 9, 13, 30, 31, 5]).tolist() == [1, 2, 3, -1, 7, -1, -1, -1]
    # a run of 5 pieces, then a run that starts on piece 8 of the plane
    assert packed_layout(np.r_[np.arange(40, 60), 99]).tolist() == [10, 11, 12, 13, 14, -1, -1, -1,
                                                                    24, -1, -1, -1]
    # an exact multiple of 4 pieces needs no padding between runs
    assert packed_layout([0, 4, 8, 12, 20]).tolist() == [0, 1, 2, 3, 5, -1, -1, -1]
    # ragged last piece of a 42-cell grid: cells 42 and 43 do not exist and read as 0
    x = np.arange(2 * 42, dtype=np.float64).reshape(2, 42) + 1
    src = packed_layout([41, 0])
    assert src.tolist() == [0, -1, -1, -1, 10, -1, -1, -1]
    exp, pad = packed_ref(x, src, [1, 0])
    assert exp.shape == (2, 32) and pad.sum() == 24
    assert exp[0, 16:20].tolist() == [83.0, 84.0, 0.0, 0.0] and exp[1, :4].tolist() == [1.0, 2.0, 3.0, 4.0]
    # streaming stores: f32 runs end on 64-byte lines at a multiple of 4 pieces; f64 pieces are 32 bytes
    z4 = host_pack_zeroed(np.array([1, 2, 3, -1, 7, -1, -1, -1]), 4)
    assert z4.tolist() == [False] * 12 + [True] * 4 + [False] * 4 + [True] * 12
    z8 = host_pack_zeroed(np.array([1, 2, 3, -1, 7, -1, -1, -1]), 8)
    assert z8.tolist() == [False] * 12 + [True] * 4 + [False] * 4 + [True] * 4 + [False] * 8


def test_route_table_covers_every_route_and_feature():
    rows = set(ROWS)
    assert len(rows) == len(ROWS)
    assert {r[0] for r in ROWS} == set(ROUTES)
    assert {r[2] for r in ROWS} == set(KINDS)
    assert {r[7] for r in ROWS} == set(LENGTHS)
    for i, name in ((1, "dtype"), (3, "tix"), (4, "gate"), (5, "groups"), (6, "split")):
        assert len({r[i] for r in ROWS}) == 2, name
    for route in ROUTES:
        assert {r[1] for r in ROWS if r[0] == route} == {F32, F64}, route
    # the chunked routes meet 600 days (19 chunks of 32: the time-index cache clears itself mid-call, and the
    # last chunk is ragged) with a time index and the gate, and time groups that cross chunk boundaries
    for route in ("device_packed", "pull", "host_pack", "full_pageable"):
        assert any(r[0] == route and r[7] == 600 and r[3] and r[4] for r in ROWS), route
    for route in ("device_packed", "pull", "host_pack", "full_pinned", "full_pageable"):
        assert any(r[0] == route and r[5] and r[7] > CHUNK for r in ROWS), route
    assert -(-600 // CHUNK) == 19 > 16 and 600 % CHUNK != 0 and GROUP_LEN < CHUNK
    # every length reaches a packed route
    assert {r[7] for r in ROWS if r[0] in ("device_packed", "pull", "host_pack")} == set(LENGTHS)
    # every transform on the pinned pull route and the pageable pack route
    for route in ("pull", "host_pack"):
        assert {r[2] for r in ROWS if r[0] == route} == set(KINDS), route


def test_time_axes_of_any_length():
    for T in LENGTHS:
        t = tix_of(T)
        assert len(t) == T and t.min() >= 0 and not np.array_equal(t, np.arange(T))
        if T >= 3:
            assert len(np.unique(t)) == T - 1 and (np.diff(t) > 1).any()
        assert len(doy_of(T)) == T
    assert np.array_equal(doy_of(77), DOY) and (np.diff(doy_of(33)) < 0).any()
    x0, x1 = long_data("edd", EDD_T[:2], 2, np.float32, 5, 605)
    assert x0.shape == x1.shape == (605, NCELL) and not (x1 < x0).any()
    assert np.array_equal(x0[:T_PHYS], make_data("edd", EDD_T[:2], 2, np.float32, 5)[0], equal_nan=True)


def test_comparators_reject_the_mutants():
    rng = np.random.default_rng(3)
    want = rng.uniform(-1, 1, (2, 5, 77))
    want[0, 1, 3] = -0.0
    want[1, 2, 5] = np.nan
    same_bits(want.copy(), want, "self")
    shifted = want.copy()
    shifted[:, :, 32:64] = want[:, :, 33:65]                 # one chunk read one day late
    swapped = want.copy()
    swapped[:, :, [10, 11]] = want[:, :, [11, 10]]           # the two f64 halves of a 16-byte unit swapped
    unwritten = want.copy()
    unwritten.view(np.int64)[:, :, 40] = SENT64              # a column no launch wrote
    zero = want.copy()
    zero[0, 1, 3] = 0.0                                      # -0.0 / +0.0
    for bad in (shifted, swapped, unwritten, zero):
        with pytest.raises(AssertionError):
            same_bits(bad, want, "mutant")
    with pytest.raises(AssertionError, match="unwritten"):
        same_bits(unwritten, want, "mutant")
    # the packed-plane comparison sees a dropped 4-day tail and an f64 piece whose first half is read twice
    x = rng.uniform(250, 320, (9, 64))
    src = packed_layout([1, 2, 9, 33, 61])
    days = [8, 3, 3, 0, 5]
    good = plane_expected(x, src, days, True)
    dropped = good.copy()
    dropped[4] = np.int64(SENT32.astype(np.int64) * 0x100000001)
    twice = good.copy().reshape(len(days), -1, 2, 2)          # [day, piece, half, 2 cells]
    twice[:, :, 1] = twice[:, :, 0]
    for bad in (dropped, twice.reshape(good.shape)):
        assert not np.array_equal(bad, good)
    # the NaN-payload exception accepts canonical NaNs only where NaNs were
    p = np.array([1.0, NAN64[0], -0.0, NAN64[1]])
    same_bits_except_nan(np.array([1.0, np.nan, -0.0, np.nan]), p, "payloads")
    for bad in ([1.0, np.nan, -0.0, 3.0], [np.nan, np.nan, -0.0, np.nan], [1.0, np.nan, 0.0, np.nan]):
        with pytest.raises(AssertionError):
            same_bits_except_nan(np.array(bad), p, "mutant")
    # the mean's exceptions: -0.0 -> +0.0 and NaN payloads, nothing else
    m = one_step_mean(p)
    assert m.view(np.int64)[[0, 2]].tolist() == [np.float64(1.0).view(np.int64), 0] and np.isnan(m[[1, 3]]).all()
    same_bits_except_nan(np.array([1.0, np.nan, 0.0, np.nan]), m, "mean")
    with pytest.raises(AssertionError):
        same_bits_except_nan(np.array([1.0, np.nan, -0.0, np.nan]), m, "mean")


def test_time_index_cache_keys_on_dtype_and_shape():
    """An int32 [5, 0] and an int64 [5] have the same bytes; each must get its own device copy."""
    import torch
    from climate_toolbox_b200 import _engine as E
    plan = E.Plan.__new__(E.Plan)
    plan.device, plan._tix_cache, plan._h = torch.device("cpu"), {}, None
    a = plan.time_index_device(np.array([5, 0], dtype=np.int32))
    b = plan.time_index_device(np.array([5], dtype=np.int64))
    c = plan.time_index_device(np.array([[5, 0]], dtype=np.int32))
    assert a.tolist() == [5, 0] and b.tolist() == [5] and c.tolist() == [[5, 0]]
    assert plan.time_index_device(np.array([5, 0], dtype=np.int32)) is a


# ----------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    import __graft_entry__ as G
    import torch
    G.build()
    return torch.device("cuda", 0)


_PLANS = {}
INFO_KEYS = ("n_bundles", "n_pieces", "n_quads", "n_quads_conflict", "n_split_regions", "n_scratch_slots",
             "max_meta_bytes")


def plans(es, n_in, split):
    """(full-grid plan, compact plan) of the fixture with the kernel matrix's options; their bundles agree."""
    from climate_toolbox_b200 import _engine as E
    import torch
    key = (es, n_in, split)
    if key not in _PLANS:
        stage = n_in * es
        kw = dict(stage_bytes=stage, device=torch.device("cuda", 0), smem_budget=33 * stage * 16 if split else 0,
                  cache=False, elem_bytes=es, cell_gate=FX["gate_words"])
        full = E.get_plan(E.GridSpec(LAT, LON), FX["df"], "popwt", "hierid", **kw)
        comp = E.get_plan(E.GridSpec(LAT, LON), FX["df"], "popwt", "hierid", compact=True, **kw)
        fi, ci = full.info, comp.info
        assert {k: fi[k] for k in INFO_KEYS} == {k: ci[k] for k in INFO_KEYS}, (fi, ci)
        assert fi["n_split_regions"] > 0 or not split
        _PLANS[key] = (full, comp)
    return _PLANS[key]


def layout_of(plan):
    w = plan.row_weights()
    keep = np.isfinite(w) & (w != 0)
    src = packed_layout(plan.row_cells()[keep])
    assert 4 * len(src) == plan.info["n_packed_cells"]
    return src


def _pin(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
    t.copy_(torch.from_numpy(a))
    return t.numpy()


def _ct(dtype):
    return N.F32 if np.dtype(dtype) == np.float32 else N.F64


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _filled_planes(T, width, dtype, dev):
    import torch
    t = torch.empty((T, width), dtype=torch.float32 if np.dtype(dtype) == np.float32 else torch.float64,
                    device=dev)
    t.view(torch.int32).fill_(int(SENT32))
    return t


def _sentinel_out(shape, dev=None):
    import torch
    t = torch.empty(shape, dtype=torch.float64, device=dev, pin_memory=dev is None)
    t.view(torch.int64).fill_(int(SENT64))
    return t


@contextlib.contextmanager
def _prefilled_outputs(shape):
    """Within the block, every float64 CUDA tensor of ``shape`` that ``torch.empty`` makes is pre-filled with the
    sentinel: the output ``aggregate_host`` allocates for itself.  Yields the list of those tensors."""
    import torch
    empty, made = torch.empty, []

    def filled(*args, **kw):
        t = empty(*args, **kw)
        if t.is_cuda and t.dtype == torch.float64 and tuple(t.shape) == tuple(shape):
            t.view(torch.int64).fill_(int(SENT64))
            made.append(t)
        return t

    mp = pytest.MonkeyPatch()
    mp.setattr(torch, "empty", filled)
    try:
        yield made
    finally:
        mp.undo()


@pytest.mark.gpu
def test_compact_and_full_plans_agree(dev):
    """The compact renumbering leaves the planner's decisions alone: bundles, pieces, quads, conflicts, split
    regions, scratch slots and metadata bytes agree, and the packed width is the restated layout's."""
    for es in (4, 8):
        for n_in in (1, 2):
            for split in (0, 1):
                full, comp = plans(es, n_in, split)
                assert not full.compact and comp.compact
                src = layout_of(comp)
                assert comp.info["n_pieces_distinct"] == (src >= 0).sum()
                print("plan info es={} n_in={} split={}: {}".format(es, n_in, split,
                                                                    {k: comp.info[k] for k in INFO_KEYS}))


def _pack_data(dtype, seed):
    """The fixture's data with NaNs of two payloads and signed zeros on referenced cells of every day."""
    x, _ = make_data("identity", (), 1, dtype, seed)
    rng = np.random.default_rng(seed)
    nan = NAN32 if np.dtype(dtype) == np.float32 else NAN64
    kept = np.isfinite(FX["w_eff"]) & (FX["w_eff"] != 0)
    pool = np.intersect1d(FX["kelvin"], FX["row_cell"][kept])
    for d in range(T_PHYS):
        x[d, rng.choice(pool, 6, replace=False)] = np.r_[nan, [-0.0, 0.0, np.inf, -np.inf]].astype(dtype)
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, F64])
def test_pack_kernels_bit_exact(dev, dtype):
    """``ctb_pull_pack`` from device and pinned memory, with and without a time index and with t_begin > 0,
    at every remainder of its 4-day groups; ``ctb_host_pack`` with 1 and 8 threads into aligned and misaligned
    destinations.  Referenced pieces equal the source bit for bit; the alignment padding keeps the sentinel
    except where the streaming stores of ``ctb_host_pack`` zero it."""
    import torch
    from climate_toolbox_b200 import _engine as E
    es = np.dtype(dtype).itemsize
    _, comp = plans(es, 1, 0)
    src = layout_of(comp)
    width = 4 * len(src)
    x = _pack_data(dtype, 11 + es)
    xd = torch.from_numpy(x).to(dev)
    xp = _pin(x)
    L = N.lib()
    long_tix = np.r_[TIX, TIX[::-1]]                     # gaps, a duplicate, and days that run backwards
    tix_d = comp.time_index_device(long_tix)
    for T in (1, 3, 4, 5, 33, 77):
        for use_tix, t_begin in ((True, 7), (False, 3)):
            days = long_tix[t_begin: t_begin + T] if use_tix else np.arange(t_begin, t_begin + T)
            want = plane_expected(x, src, days, True)
            for label, ptr in (("device", xd.data_ptr()), ("pinned", xp.ctypes.data)):
                dst = _filled_planes(T, width, dtype, dev)
                N.check(L.ctb_pull_pack(comp._h, C.c_void_p(ptr), _ct(dtype), NCELL, _ptr(tix_d) if use_tix else None,
                                        t_begin, T, _ptr(dst), E._stream_ptr(dev)))
                got = dst.cpu().numpy().view(_ITYPE[es])
                assert np.array_equal(got, want), ("pull_pack", label, T, use_tix, np.argwhere(got != want)[:4])
            # ctb_host_pack: the same pieces from a pageable source
            t64 = np.ascontiguousarray(long_tix, dtype=np.int64)
            for threads in (1, 8):
                for aligned in (True, False):
                    nbytes = T * width * es
                    raw = np.empty(nbytes + 128, dtype=np.uint8)
                    off = (-raw.ctypes.data) % 64 + (0 if aligned else 16)
                    buf = raw[off: off + nbytes]
                    buf.view(np.int32)[:] = SENT32
                    N.check(L.ctb_host_pack(comp._h, C.c_void_p(x.ctypes.data), _ct(dtype), NCELL,
                                            t64.ctypes.data_as(C.POINTER(C.c_int64)) if use_tix else None,
                                            t_begin, T, C.c_void_p(buf.ctypes.data), threads))
                    hw = plane_expected(x, src, days, True, host_pack_zeroed(src, es) if aligned else None)
                    got = buf.view(_ITYPE[es]).reshape(T, width)
                    assert np.array_equal(got, hw), ("host_pack", T, use_tix, threads, aligned,
                                                     np.argwhere(got != hw)[:4])


def _ragged_case(nlat, nlon, dtype, seed):
    """A grid whose cell count is not a multiple of 4, weights on every piece including the ragged last one,
    and the reference fixture of its regions."""
    from climate_toolbox_b200 import _engine as E
    import torch
    rng = np.random.default_rng(seed)
    ncell = nlat * nlon
    lat, lon = 0.5 + np.arange(nlat), 10.5 + np.arange(nlon)
    cells = np.r_[rng.choice(ncell - 1, 30), ncell - 1, ncell - 2, ncell - 1]
    code = np.r_[rng.permutation(np.arange(30) % 6), 6, 6, 6]
    wp = rng.uniform(1.0, 100.0, len(cells))
    ii, jj = np.divmod(cells, nlon)
    df = pd.DataFrame({"lat": lat[ii], "lon": lon[jj], "hierid": code, "popwt": wp, "areawt": wp})
    es = np.dtype(dtype).itemsize
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=es, device=torch.device("cuda", 0),
                      cache=False, compact=True, elem_bytes=es)
    w = np.asarray(df["popwt"].values)
    fx = {"R": 7, "row_cell": cells.astype(np.int64), "w_eff": w,
          "members": [np.flatnonzero(code == r) for r in range(7)]}
    return plan, fx, ncell


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,nlat,nlon", [(F32, 7, 9), (F64, 6, 7)])
def test_ragged_grid(dev, dtype, nlat, nlon):
    """A grid of 63 (f32) or 42 (f64, 16-byte aligned planes) cells: ``ctb_host_pack`` copies what exists and
    zero-fills the rest of the last piece; the GPU pack kernels refuse it; ``aggregate_host`` on a pinned source
    falls back to host packing and stays within the derived bound of the reference."""
    import torch
    from climate_toolbox_b200 import _engine as E
    plan, fx, ncell = _ragged_case(nlat, nlon, dtype, 5)
    src = layout_of(plan)
    assert 4 * src.max() + 4 > ncell                                   # the ragged piece is referenced
    es = np.dtype(dtype).itemsize
    T = 40
    x = np.random.default_rng(9).uniform(250.0, 320.0, (T, ncell)).astype(dtype)
    width = 4 * len(src)
    L = N.lib()
    for threads in (1, 4):
        buf = np.full(T * width * es // 4, SENT32, dtype=np.int32).view(dtype)
        N.check(L.ctb_host_pack(plan._h, C.c_void_p(x.ctypes.data), _ct(dtype), ncell, None, 0, T,
                                C.c_void_p(buf.ctypes.data), threads))
        want = plane_expected(x, src, np.arange(T), True)
        got = buf.view(_ITYPE[es]).reshape(T, width)
        assert np.array_equal(got[:, ~np.repeat(src < 0, 4)], want[:, ~np.repeat(src < 0, 4)]), threads
    xp = _pin(x)
    dst = _filled_planes(T, width, dtype, dev)
    assert L.ctb_pull_pack(plan._h, C.c_void_p(xp.ctypes.data), _ct(dtype), ncell, None, 0, T, _ptr(dst),
                           E._stream_ptr(dev)) == N.ERR_UNSUPPORTED
    d8 = _filled_planes(T, width, F64, dev)
    assert L.ctb_pull_pack_daily(plan._h, C.c_void_p(xp.ctypes.data), _ct(dtype), ncell, 1, None, 0, T,
                                 N.DAILY_MAX if es == 4 else N.DAILY_MEAN, _ptr(d8), _ptr(dst), _ptr(dst),
                                 E._stream_ptr(dev)) == N.ERR_UNSUPPORTED
    before = E.TRANSFER_BYTES["h2d"]
    out = E.aggregate_host(plan, [xp], N.LAYOUT_TIME_MAJOR, ncell, None, T, chunk_bytes=1)
    assert E.TRANSFER_BYTES["h2d"] - before == T * width * es         # packed chunks, not pulled pieces
    ref, base, sny = reference(dict(fx, T=T), "identity", (), 1, x, None, None, None)
    check(out.cpu().numpy(), ref, base, sny, "ragged {}".format(np.dtype(dtype).name))


# one fault per call of ctb_pull_pack: (arguments changed, status, a word of the message)
PULL_FAULTS = (
    ("non-compact plan", {"plan": "full"}, N.ERR_INVALID, "compact"),
    ("dtype 7", {"dtype": 7}, N.ERR_INVALID, "dtype=7"),
    ("misaligned source", {"offset": 4}, N.ERR_UNSUPPORTED, "aligned"),
    ("T < 0", {"T": -1}, N.ERR_INVALID, "T=-1"),
    ("T >= 2^31", {"T": 2 ** 31}, N.ERR_INVALID, "T=2147483648"),
    ("t_begin < 0", {"t_begin": -1}, N.ERR_INVALID, "t_begin=-1"),
)


@pytest.mark.gpu
def test_pull_pack_refuses_single_faults(dev):
    """``ctb_pull_pack`` refuses each fault of ``PULL_FAULTS`` alone, with its status and message, and writes
    nothing; the same call without the fault succeeds.  The source starts one plane into its buffer, so that
    even plane t_begin - 1 lies inside it."""
    import torch
    from climate_toolbox_b200 import _engine as E
    full, comp = plans(4, 1, 0)
    n_days = 8
    buf = torch.zeros((n_days + 1, NCELL), dtype=torch.float32, device=dev)
    width = 4 * len(layout_of(comp))
    L = N.lib()

    def call(plan="comp", dtype=N.F32, offset=0, t_begin=0, T=n_days):
        dst = _filled_planes(n_days, width, F32, dev)
        rc = L.ctb_pull_pack((full if plan == "full" else comp)._h, C.c_void_p(buf[1].data_ptr() + offset), dtype,
                             NCELL, None, t_begin, T, _ptr(dst), E._stream_ptr(dev))
        torch.cuda.synchronize(dev)
        return rc, bool((dst.view(torch.int32) == int(SENT32)).all())

    assert call() == (N.OK, False)
    for label, change, status, word in PULL_FAULTS:
        rc, untouched = call(**change)
        assert rc == status and word in N.last_error(), (label, rc, N.last_error())
        assert untouched, label


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, F64])
def test_padding_is_never_read(dev, dtype):
    """One set of packed planes aggregated with NaN, with 1e30 and with the pack's untouched sentinel words in
    every padding cell gives the same bits, streaming and direct kernel, gated, one and two inputs.  NaN products
    are skipped, so a kernel that read a padding cell with a real weight would add a finite nonzero term under
    the other two fills (0 would not do: f(0) is 0 for the identity and for Snyder at (0, 0))."""
    import torch
    from climate_toolbox_b200 import _engine as E
    es = np.dtype(dtype).itemsize
    T = 77
    for kind_key in ("identity", "edd2"):
        kind, params, n_out = KINDS[kind_key]
        _, comp = plans(es, _n_in(kind), 0)
        src = layout_of(comp)
        width = 4 * len(src)
        pad = torch.as_tensor(np.repeat(src < 0, 4), device=dev)
        xs = [v for v in make_data(kind, params, n_out, dtype, 31) if v is not None]
        planes = []
        tix_d = comp.time_index_device(TIX)
        for x in xs:
            xd = torch.from_numpy(x).to(dev)
            p = _filled_planes(T, width, dtype, dev)
            N.check(N.lib().ctb_pull_pack(comp._h, _ptr(xd), _ct(dtype), NCELL, _ptr(tix_d), 0, T, _ptr(p),
                                          E._stream_ptr(dev)))
            planes.append(p)
        torch.cuda.synchronize()
        for variant in (N.VARIANT_STAGED, N.VARIANT_DIRECT):
            res = []
            for fill in (float("nan"), 1e30, None):
                ps = [p.clone() for p in planes]
                for p in ps:
                    if fill is None:
                        assert (p[:, pad].view(torch.int32) == int(SENT32)).all()     # as packed: untouched
                    else:
                        p[:, pad] = fill
                res.append(E.aggregate_device(comp, ps[0], ps[1] if len(ps) > 1 else None, N.LAYOUT_TIME_MAJOR,
                                              width, None, T, kind, params, n_out, variant=variant,
                                              doy=DOY).cpu().numpy())
            for r, fill in zip(res[1:], ("1e30", "sentinel")):
                same_bits(r, res[0], "padding {} {} {} {}".format(kind_key, np.dtype(dtype).name, variant, fill))


_CASES = {}


def _case(dtype, kind_key, tix, gate, groups, split, T, variant):
    """Data, time axes, plans and the baseline of one case, the baseline checked once against the reference."""
    import torch
    from climate_toolbox_b200 import _engine as E
    key = (np.dtype(dtype).name, kind_key, tix, gate, groups, split, T, variant)
    if key in _CASES:
        return _CASES[key]
    kind, params, n_out = KINDS[kind_key]
    es = np.dtype(dtype).itemsize
    full, comp = plans(es, _n_in(kind), split)
    t = tix_of(T) if tix else None
    t_phys = max(T_PHYS, T + 1)
    seed = 50000 + 1000 * LENGTHS.index(T) + 10 * list(KINDS).index(kind_key) + es
    x0, x1 = long_data(kind, params, n_out, dtype, seed, t_phys)
    doy = doy_of(T) if gate else None
    grp = E.get_time_groups(np.arange(T) // GROUP_LEN, full.device) if groups else None
    d = torch.device("cuda", 0)
    if variant == "cell_major":
        a0 = torch.from_numpy(np.ascontiguousarray(x0.T)).to(d)
        a1 = None if x1 is None else torch.from_numpy(np.ascontiguousarray(x1.T)).to(d)
        layout, stride, var = N.LAYOUT_CELL_MAJOR, t_phys, N.VARIANT_DIRECT
    else:
        a0 = torch.from_numpy(x0).to(d)
        a1 = None if x1 is None else torch.from_numpy(x1).to(d)
        layout, stride = N.LAYOUT_TIME_MAJOR, NCELL
        var = N.VARIANT_DIRECT if variant == "direct" else N.VARIANT_STAGED
    base = E.aggregate_device(full, a0, a1, layout, stride, t, T, kind, params, n_out, variant=var, groups=grp,
                              doy=doy).cpu().numpy()
    ref = reference(dict(FX, T=T), kind, params, n_out, x0, x1, t, None if doy is None else _gate_on(FX["gate_words"], doy))
    if groups:
        ref = group_reference(ref, T)
    with np.errstate(all="ignore"):
        check(base, *ref, "baseline {}".format(key))
    c = dict(kind=kind, params=params, n_out=n_out, full=full, comp=comp, tix=t, doy=doy, groups=grp, x0=x0, x1=x1,
             t_phys=t_phys, base=base, es=es)
    if len(_CASES) > 8:
        _CASES.clear()
    _CASES[key] = c
    return c


def _route(route, c, T, dev):
    """Run one route of a case: (device result, pinned host result or None).  Pinned sources live until the
    device is done with them: ``ctb_pull_pack`` and the zero-copy kernel read them with no event recorded."""
    import torch
    keep = []
    res = _launch_route(route, c, T, dev, keep)
    torch.cuda.synchronize()
    return res


def _pinned(xs, keep):
    keep.extend(_pin(x) for x in xs)
    return keep[-len(xs):]


def _launch_route(route, c, T, dev, keep):
    import torch
    from climate_toolbox_b200 import _engine as E
    kind, params, n_out, groups, doy, tix = c["kind"], c["params"], c["n_out"], c["groups"], c["doy"], c["tix"]
    full, comp = c["full"], c["comp"]
    xs = [c["x0"]] + ([c["x1"]] if c["x1"] is not None else [])
    shape = (n_out, full.R, T if groups is None else groups.n_groups)
    L = N.lib()
    if route in ("device_packed", "direct_compact"):
        ds = [torch.from_numpy(x).to(dev) for x in xs]
        tix_d = comp.time_index_device(tix)

        def pack(t0, n, bufs):
            for x, b in zip(ds, bufs):
                N.check(L.ctb_pull_pack(comp._h, _ptr(x), _ct(xs[0].dtype), NCELL,
                                        _ptr(tix_d), t0, n, _ptr(b), E._stream_ptr(dev)))

        out = _sentinel_out(shape, dev)
        if route == "device_packed":
            E._aggregate_packed(comp, pack, len(xs), c["es"], T, kind, params, n_out, N.VARIANT_STAGED, groups, out,
                                chunk_bytes=1, doy=doy)
            return out, None
        width = comp.info["n_packed_cells"]
        bufs = [_filled_planes(T, width, xs[0].dtype, dev) for _ in xs]
        pack(0, T, bufs)
        E.aggregate_device(comp, bufs[0], bufs[1] if len(bufs) > 1 else None, N.LAYOUT_TIME_MAJOR, width, None, T,
                           kind, params, n_out, variant=N.VARIANT_DIRECT, out=out, groups=groups, doy=doy)
        return out, None
    if route == "pull":
        out = _sentinel_out(shape, dev)
        host = _sentinel_out(shape) if groups is None else None
        out, filled = E._aggregate_pull(comp, _pinned(xs, keep), NCELL, tix, T, kind, params, n_out,
                                        N.VARIANT_STAGED, groups, out, host_out=host, chunk_bytes=1, doy=doy)
        assert filled == (groups is None)
        return out, host
    kw = dict(kind=kind, params=params, n_out=n_out, groups=groups, doy=doy)
    with _prefilled_outputs(shape) as made:
        if route == "host_pack":
            out = E.aggregate_host(comp, xs, N.LAYOUT_TIME_MAJOR, NCELL, tix, T, variant=N.VARIANT_STAGED,
                                   chunk_bytes=1, ingest="pack", **kw)
        elif route in ("full_pinned", "full_pageable", "zero_copy"):
            src = _pinned(xs, keep) if route != "full_pageable" else xs
            before = E.TRANSFER_BYTES["h2d"]
            out = E.aggregate_host(full, src, N.LAYOUT_TIME_MAJOR, NCELL, tix, T, variant=N.VARIANT_STAGED,
                                   chunk_bytes=1, zero_copy=(route == "zero_copy"), **kw)
            assert (E.TRANSFER_BYTES["h2d"] == before) == (route == "zero_copy"), route   # read in place, or copied
        else:
            assert route == "cell_major"
            cm = [np.ascontiguousarray(x.T) for x in xs]
            out = E.aggregate_host(full, cm, N.LAYOUT_CELL_MAJOR, c["t_phys"], tix, T, variant=N.VARIANT_DIRECT, **kw)
    assert len(made) == 1 and made[0].data_ptr() == out.data_ptr(), route    # the output started as the sentinel
    return out, None


@pytest.mark.gpu
@pytest.mark.parametrize("row", ROWS, ids=[_row_id(r) for r in ROWS])
def test_route_matrix(dev, row):
    """One route x feature row: the route's result (and its pinned host copy) equals the device-resident
    full-grid launch of the same kernel variant bit for bit."""
    route, dtype, kind_key, tix, gate, groups, split, T = row
    c = _case(dtype, kind_key, tix, gate, groups, split, T, _baseline_variant(route))
    out, host = _route(route, c, T, dev)
    same_bits(out.cpu().numpy(), c["base"], _row_id(row))
    if host is not None:
        same_bits(host.numpy(), c["base"], _row_id(row) + " host_out")


def _subdaily_var(x, S, where):
    """The deferred daily mean of ``x`` [days * S, NLAT, NLON] on the fixture's grid (``utils.resample_daily``)."""
    import torch
    from climate_toolbox_b200 import Dataset
    from climate_toolbox_b200.utils.utils import resample_daily
    data = torch.from_numpy(x).cuda() if where == "device" else x
    times = pd.date_range("2003-12-20", periods=x.shape[0], freq="{}min".format(24 * 60 // S)).values
    ds = Dataset({"tas": (("time", "lat", "lon"), data)}, coords={"time": times, "lat": LAT, "lon": LON})
    return resample_daily(ds, "mean")._vars["tas"]


@pytest.mark.gpu
def test_staging_reuse_across_calls(dev, monkeypatch):
    """Back-to-back host calls with different data and sizes share the pinned staging buffers through their
    events: a pack route, then a larger chunk (the buffer grows), a two-input call after one-input ones, a
    float64 call, and a pageable sub-daily call whose two daily staging slots alternate many times.  Each
    result equals its own device-resident baseline bit for bit."""
    import torch
    from climate_toolbox_b200 import _engine as E
    from test_subdaily import resample_daily_ref
    calls = [("identity", F32, 77, 32), ("identity", F32, 600, 128), ("edd2", F32, 77, 32), ("poly4", F64, 33, 32),
             ("edd2", F32, 600, 64)]                       # (transform, input type, days, days per chunk)
    results = []
    for i, (kind_key, dtype, T, days) in enumerate(calls):
        kind, params, n_out = KINDS[kind_key]
        es = np.dtype(dtype).itemsize
        full, comp = plans(es, _n_in(kind), 0)
        chunk = days * comp.info["n_packed_cells"] * es * _n_in(kind)
        x0, x1 = long_data(kind, params, n_out, dtype, 700 + i, max(T_PHYS, T + 1))
        xs = [x0] + ([x1] if x1 is not None else [])
        t, doy = tix_of(T), doy_of(T)
        out = E.aggregate_host(comp, xs, N.LAYOUT_TIME_MAJOR, NCELL, t, T, kind, params, n_out,
                               variant=N.VARIANT_STAGED, chunk_bytes=chunk, ingest="pack", doy=doy)
        results.append((full, xs, t, doy, T, kind, params, n_out, out))
    # sub-daily, pageable: 3 days per staging slot
    S, T = 4, 77
    x = np.random.default_rng(77).uniform(250.0, 320.0, (T * S, NLAT, NLON)).astype(np.float32)
    x[5, 3, 7] = np.nan
    x[8:12, 4, 4] = np.nan
    monkeypatch.setattr(E, "DAILY_STAGE_BYTES", 3 * S * NCELL * 4)
    full8, comp8 = plans(8, 1, 0)
    sub = E.aggregate_daily(comp8, [(E.DailySource(_subdaily_var(x, S, "pageable")), "mean")])
    torch.cuda.synchronize()
    for k, (full, xs, t, doy, T_, kind, params, n_out, out) in enumerate(results):
        ds = [torch.from_numpy(v).to(dev) for v in xs]
        base = E.aggregate_device(full, ds[0], ds[1] if len(ds) > 1 else None, N.LAYOUT_TIME_MAJOR, NCELL, t, T_,
                                  kind, params, n_out, variant=N.VARIANT_STAGED, doy=doy)
        same_bits(out.cpu().numpy(), base.cpu().numpy(), "call {}".format(k))
    mean = resample_daily_ref(x.reshape(T * S, NCELL), S, "mean")
    base = E.aggregate_device(full8, torch.from_numpy(mean).to(dev), None, N.LAYOUT_TIME_MAJOR, NCELL, None, T,
                              variant=N.VARIANT_STAGED).cpu().numpy()
    check(base, *reference(dict(FX, T=T), "identity", (), 1, mean, None, None, None), "sub-daily baseline")
    same_bits(sub.cpu().numpy(), base, "sub-daily pageable")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [F32, F64])
def test_subdaily_one_step_equals_plain_packing(dev, dtype):
    """With one step per day, ``ctb_pull_pack_daily`` MIN and MAX write the planes ``ctb_pull_pack`` writes
    except for NaN payloads, and MEAN (float64) except that -0.0 becomes +0.0 and NaN the canonical NaN.
    Aggregating any of them gives the pull route's bits: NaN products are skipped whatever their payload."""
    import torch
    from climate_toolbox_b200 import _engine as E
    es = np.dtype(dtype).itemsize
    _, comp = plans(es, 1, 0)
    src = layout_of(comp)
    width = 4 * len(src)
    pad = np.repeat(src < 0, 4)
    x = _pack_data(dtype, 23 + es)
    xd = torch.from_numpy(x).to(dev)
    L = N.lib()
    t_begin, T = 5, 70
    tix_d = comp.time_index_device(TIX)
    st = E._stream_ptr(dev)
    plain = _filled_planes(T, width, dtype, dev)
    N.check(L.ctb_pull_pack(comp._h, _ptr(xd), _ct(dtype), NCELL, _ptr(tix_d), t_begin, T, _ptr(plain), st))
    mn, mx = _filled_planes(T, width, dtype, dev), _filled_planes(T, width, dtype, dev)
    N.check(L.ctb_pull_pack_daily(comp._h, _ptr(xd), _ct(dtype), NCELL, 1, _ptr(tix_d), t_begin, T,
                                  N.DAILY_MIN | N.DAILY_MAX, None, _ptr(mn), _ptr(mx), st))
    p = plain.cpu().numpy()
    assert np.isnan(p[:, ~pad]).any() and (np.signbit(p[:, ~pad]) & (p[:, ~pad] == 0)).any()
    sets = {"min": mn, "max": mx}
    for name, planes in sets.items():
        got = planes.cpu().numpy()
        same_bits_except_nan(got[:, ~pad], p[:, ~pad], "daily {} {}".format(name, np.dtype(dtype).name))
        assert (got[:, pad].view(_ITYPE[es]) == plane_expected(x, src, TIX[t_begin: t_begin + T], True)[:, pad]).all()
    if es == 8:
        mean = _filled_planes(T, width, F64, dev)
        N.check(L.ctb_pull_pack_daily(comp._h, _ptr(xd), N.F64, NCELL, 1, _ptr(tix_d), t_begin, T, N.DAILY_MEAN,
                                      _ptr(mean), None, None, st))
        got = mean.cpu().numpy()
        same_bits_except_nan(got[:, ~pad], one_step_mean(p[:, ~pad]), "daily mean float64")
        assert len(np.unique(got[:, ~pad][np.isnan(got[:, ~pad])].view(np.int64))) == 1   # one canonical NaN
        assert (got[:, pad].view(np.int64) == plane_expected(x, src, TIX[t_begin: t_begin + T], True)[:, pad]).all()
        sets["mean"] = mean
    kind, params, n_out = "poly", (OFF, 1.0, 2.0), 2
    doy = DOY[t_begin: t_begin + T]
    want = E.aggregate_device(comp, plain, None, N.LAYOUT_TIME_MAJOR, width, None, T, kind, params, n_out,
                              variant=N.VARIANT_STAGED, doy=doy).cpu().numpy()
    for name, planes in sets.items():
        got = E.aggregate_device(comp, planes, None, N.LAYOUT_TIME_MAJOR, width, None, T, kind, params, n_out,
                                 variant=N.VARIANT_STAGED, doy=doy).cpu().numpy()
        same_bits(got, want, "aggregate of daily {} {}".format(name, np.dtype(dtype).name))
