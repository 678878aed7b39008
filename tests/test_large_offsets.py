"""Every kernel at element offsets past 2^31 and byte offsets past 4 GiB, against a float64 reference.

Real inputs pass these sizes: 0.25 degree daily data (1,036,800 cells) passes 2^31 elements after 2,072 days,
hourly ERA5 at 0.25 degree after 86 days, and a float64 plane passes 4 GiB at 2^29 cells (the plan accepts up to
2^30).  An address formed in 32 bits there does not fault: it reads another element of the same allocation.
So every input element here holds ``value(i)``, a function of its flat index ``i`` that differs at ``i`` and
``i +- 2^29, 2^30, 2^31, 2^32``: an address that wraps at 32 bits reads a visibly different number.  The reference
recomputes ``value`` in numpy for the indices it needs, and ``test_kernel_matrix.reference`` / ``check`` compare
(exact ``math.fsum`` per region-day, bound ``(n_r + 4) 2^-53 S_r``).  Referenced cells are gathered on the
device, so no test copies gigabytes to the host.

Address expressions covered, with their largest value at the tested shape (Q = the 0.25 degree grid,
1,036,800 cells; the float32 buffer holds 2,088 of its planes, 8.7 GB; the float64 one 2,080, 17.3 GB):

=====================  ===========================================================  ===================================
kernel                 expression                                                   largest value tested
=====================  ===========================================================  ===================================
agg_stream_kernel      ``X0 + ro + off``, ``ro = (tb*32 + l4) * stride``             2,164,838,399 elements (case A)
  no time index        (elements, int64 row offset + int32 unit offset)
agg_stream_kernel      ``(int64)plane * stride_b``                                   17,252,351,992 bytes (case B, f64)
  time index           ``+ (uint64)(uint32)off * sizeof(TIN)``, ``r1 = X1 + ro``     4,299,161,584 bytes (C: f64, a
                                                                                    2^29+ cell plan); 4,294,967,264
                                                                                    (D: f32, 2^30 - 4 cells)
agg_stream_kernel      ``((size_t)j * R + target) * out_ld + t``                     2,164,838,399 (case G)
  epilogue
agg_direct_kernel      ``tp * stride + c`` / ``c * stride + tp`` (int64)             2,164,838,399 / 2,164,838,399 (F)
transform_kernel       grid-stride ``i`` (int64), ``(size_t)j * n + i``              2,164,838,399 (case H)
gather_rows_kernel     ``tp * stride + c`` / ``c * stride + tp``, ``out[i]``         2,164,838,399 (case I)
pull_pack_kernel       ``src + tp * stride16 + so`` (16-byte units)                  8,659,353,596 bytes (case J)
subdaily_step_loop     ``src + step0 * stride16 + p * halves + u % halves``          8,659,353,596 bytes (case J, both
  (both sub-daily      ``+ (h0 + k) * stride16``                                    kernels: subdaily_pack_kernel
  kernels)                                                                          and subdaily_steps_kernel)
=====================  ===========================================================  ===================================

The float64 time-indexed byte offset (row C) wrapped at 2^32 before: ``(uint32_t)off * (uint32_t)sizeof(TIN)``
read the cell 2^29 positions earlier for every cell at or past 2^29.  Case C fails without the 64-bit product.

Audited and not reachable within 180 GB (limits the library checks, so no test): the plan refuses grids of 2^30
cells or more and 2^31 weights rows (case D checks the first refusal), so unit offsets, row cells and CSR indices
fit int32; ``T`` and every time index are below 2^31 (``ctb_aggregate`` and the three ``ctb_pull_pack*`` entry
points refuse more), so ``tb * 32 + lane`` and the day of a tile fit int32; the streaming
scheduler refuses 2^31 work units; a packed plane has fewer than 2^30 cells, so ``n_units`` of the pull kernels
fits int32.  The split-region scratch ``((size_t)j * n_scratch + slot) * scratch_ld + t`` and the time-group
partial sums are size_t products reached only at small sizes here.

B with ``tix = arange(T)`` equals A bit for bit: the producers copy the same bytes into the same tile slots,
and the consumer code is shared.  E runs Snyder EDD and GDD with thresholds below every value (-100 and 600 K),
where both are linear in the mean ``(x0 + x1) / 2``: the pair ``x0 = buf[t]``, ``x1 = buf[t + 1]`` is not ordered,
and the transform is symmetric in it there, so the reference takes the ordered pair.

Every GPU case checks ``torch.cuda.mem_get_info()`` first and skips, naming bytes needed and free, when the device
lacks room; the float32 buffer is shared by a module fixture, everything else is freed at the end of its case.
Measured on one NVIDIA B200 (1,000 W power limit): the GPU cases take 9.7 s in all, with a peak of 29.1 GB
allocated through torch (G and H: the 8.7 GB input, 17.3 GB of results and the chunks compared on the device).
"""
import ctypes as C

import numpy as np
import pandas as pd
import pytest

import oracle
from test_kernel_matrix import NEEDED, U, check, reference
from test_subdaily import resample_daily_ref
from test_subdaily_steps import steps_ref
from climate_toolbox_b200 import _native as N

# ----------------------------------------------------------------------------
# the element values
# ----------------------------------------------------------------------------
LO_BITS = 29
HI_MUL = 0x1D2B5           # odd: s * HI_MUL != 0 mod 2^22 for s = 1, 2, 4, 8 -- strides 2^29 .. 2^32 never alias
FRAC = 2.0 ** -15
BASE_K = 200.0             # kelvin values in [200, 328): positive normal floats, the widening fast path
CELSIUS_SHIFT = 256.0      # cells in a Celsius range hold value - 256, in [-56, 72): the exact path
STRIDES = (2 ** 29, 2 ** 30, 2 ** 31, 2 ** 32)


def _mix(i, xp):
    """22-bit code of flat index ``i`` (int64 array, numpy or torch): a mixer of the low 29 bits plus an odd
    multiple of the bits above, so that i and i + s * 2^29 differ for |s| in 1, 2, 4, 8.  Every intermediate is
    non-negative and below 2^62 (the same result under numpy and torch int64 arithmetic)."""
    lo = i & ((1 << LO_BITS) - 1)
    hi = i >> LO_BITS
    x = lo * 0x9E3779B1
    x = x ^ (x >> 17)
    x = (x & 0x7FFFFFFF) * 0x2C1B3C6D
    x = x ^ (x >> 23)
    return (x + hi * HI_MUL) & 0x3FFFFF


def value_np(i, ncell, celsius=()):
    """float64 value of flat indices ``i``; exactly representable in float32.  ``celsius``: (c0, c1) ranges of
    cells (``i % ncell``) that hold degrees Celsius."""
    i = np.asarray(i, dtype=np.int64)
    v = BASE_K + _mix(i, np).astype(np.float64) * FRAC
    c = i % ncell
    for c0, c1 in celsius:
        v = np.where((c >= c0) & (c < c1), v - CELSIUS_SHIFT, v)
    return v


def value_torch(i, ncell, celsius=()):
    import torch
    v = BASE_K + _mix(i, torch).to(torch.float64) * FRAC
    c = i % ncell
    for c0, c1 in celsius:
        v = torch.where((c >= c0) & (c < c1), v - CELSIUS_SHIFT, v)
    return v


# ----------------------------------------------------------------------------
# grids, regions, reference
# ----------------------------------------------------------------------------
QLAT, QLON = 720, 1440                     # 0.25 degree
QCELL = QLAT * QLON                        # 1,036,800
QLAT_L = -90 + 0.125 + 0.25 * np.arange(QLAT)
QLON_L = -180 + 0.125 + 0.25 * np.arange(QLON)
T32 = 2088                                 # float32 planes: 87 hourly days; plane 2071 crosses 2^31 elements
T64 = 2080                                 # float64 planes
Q_CELSIUS = ((600 * QLON, 602 * QLON),)
CROSS = (1 << 31) // QCELL                 # 2071: the plane that crosses 2^31 elements

C_LAT, C_LON = 16400, 32768                # case C: 537,395,200 cells >= 2^29, float64
C_CELL = C_LAT * C_LON
C_CELSIUS = ((2 ** 29 + 1024, 2 ** 29 + 1536),)
D_LAT, D_LON = 18705, 57404                # case D: 2^30 - 4 cells, float32
D_CELL = D_LAT * D_LON
D_CELSIUS = ((2 ** 29 + 4096, 2 ** 29 + 4608),)


def q_regions():
    """Regions of the 0.25 degree grid: plane ends and starts, the rows whose cell-major offsets pass 2^31,
    every quad residue, a Celsius region and one big enough to split over bundles."""
    rng = np.random.default_rng(31)
    last_rows = np.arange(715 * QLON, QCELL)
    cel = np.arange(*Q_CELSIUS[0])
    return [np.array([0]), np.array([QCELL - 1]), np.arange(QCELL - 8, QCELL),
            rng.choice(last_rows, 3, replace=False), rng.integers(0, QCELL, 17), rng.integers(0, QCELL, 33),
            rng.choice(last_rows, 64, replace=False), rng.integers(0, QCELL, 90), rng.choice(cel, 20, replace=False),
            rng.integers(0, QCELL, 5), np.array([5, QCELL - 5]), np.arange(2 ** 19, 2 ** 19 + 4)]


def c_regions(ncell, b, celsius):
    """Regions on the cells just below and just above ``b`` (the offset whose bytes pass 2^32), across it, at
    the plane's end and start, in a Celsius range and spread over the plane (one big enough to split)."""
    rng = np.random.default_rng(int(b) % 1000)
    c0 = celsius[0][0]
    return [np.arange(b - 4, b), np.arange(b, b + 4), np.arange(b - 6, b + 7), np.arange(b - 64, b - 31),
            np.arange(b + 31, b + 64), np.array([b - 1]), np.array([b]), np.arange(ncell - 8, ncell),
            np.arange(0, 5), np.arange(c0, c0 + 17), rng.integers(0, ncell, 90),
            np.r_[np.arange(b - 2, b + 2), np.arange(ncell - 2, ncell)]]


def region_table(lat, lon, groups, seed, unit_weights=False):
    """(weights DataFrame, fixture dict for ``test_kernel_matrix.reference``, the distinct cells).  Region r is
    ``groups[r]``; weights in [1, 1000) with a fifth of the primaries falling back to the backup.  ``unit_weights``:
    powers of two, so a one-cell region's aggregate is its value exactly."""
    rng = np.random.default_rng(seed)
    nlon = len(lon)
    cells = np.concatenate(groups).astype(np.int64)
    code = np.repeat(np.arange(len(groups)), [len(g) for g in groups])
    if unit_weights:
        wp = 2.0 ** rng.integers(-3, 4, len(cells))
        wb = np.ones(len(cells))
    else:
        wp = rng.uniform(1.0, 1000.0, len(cells))
        wb = rng.uniform(1.0, 1000.0, len(cells))
        wp[rng.random(len(cells)) < 0.2] = np.nan
    df = pd.DataFrame({"lat": np.asarray(lat)[cells // nlon], "lon": np.asarray(lon)[cells % nlon], "hierid": code,
                       "popwt": wp, "areawt": wb})
    w_eff = oracle.effective_weights(df, "popwt", "areawt")
    ucells, inv = np.unique(cells, return_inverse=True)
    kept = np.flatnonzero(np.isfinite(w_eff) & (w_eff != 0))           # code is sorted: rows of a region adjoin
    bounds = np.searchsorted(code[kept], np.arange(len(groups) + 1))
    members = [kept[bounds[r]:bounds[r + 1]] for r in range(len(groups))]
    fx = {"R": len(groups), "members": members, "row_cell": inv.astype(np.int64), "w_eff": w_eff}
    return df, fx, ucells


def tm_index(planes, ucells, stride, base=0):
    """Flat element index [t, u] of a TIME_MAJOR read: base + plane * stride + cell."""
    return base + np.asarray(planes, np.int64)[:, None] * stride + np.asarray(ucells, np.int64)[None, :]


def cm_index(tps, ucells, stride):
    """Flat element index [t, u] of a CELL_MAJOR read: cell * stride + tp."""
    return np.asarray(ucells, np.int64)[None, :] * stride + np.asarray(tps, np.int64)[:, None]


def ref_of(fx, kind, params, n_out, idx0, ncell, celsius, idx1=None):
    """(ref, base, sny) of the region-days whose inputs sit at flat indices idx0 (and idx1) [T, cells]."""
    x0 = value_np(idx0, ncell, celsius)
    x1 = None
    if idx1 is not None:   # the symmetric range of the Snyder forms here: the ordered pair (module docstring)
        x1 = value_np(idx1, ncell, celsius)
        x0, x1 = np.minimum(x0, x1), np.maximum(x0, x1)
    return reference(dict(fx, T=idx0.shape[0]), kind, params, n_out, x0, x1, None, None)


def wrap_elements(idx):
    """The element index a 32-bit signed element offset reads: wrapped modulo 2^31."""
    return np.asarray(idx, np.int64) % (1 << 31)


def wrap_plane_bytes(idx, ncell, es):
    """The element a 32-bit byte offset inside a plane reads: (cell * es mod 2^32) / es in the same plane."""
    idx = np.asarray(idx, np.int64)
    plane, cell = np.divmod(idx, ncell)
    return plane * ncell + ((cell * es) % (1 << 32)) // es


# ----------------------------------------------------------------------------
# CPU: the values and the comparator catch the bug class
# ----------------------------------------------------------------------------
def _sample_indices():
    rng = np.random.default_rng(5)
    near = np.concatenate([k * 2 ** 29 + np.arange(-64, 64) for k in range(1, 70)])
    return np.unique(np.r_[np.arange(0, 256), near, rng.integers(0, 2 ** 36, 20000)]).astype(np.int64)


def test_values_differ_at_every_wrap_stride():
    i = _sample_indices()
    for ncell, cel in ((QCELL, Q_CELSIUS), (C_CELL, C_CELSIUS), (D_CELL, D_CELSIUS)):
        v = value_np(i, ncell, cel)
        for s in STRIDES:
            for j in (i + s, i - s):
                ok = j >= 0
                assert (value_np(j[ok], ncell, cel) != v[ok]).all(), (ncell, s)
        assert np.array_equal(v.astype(np.float32).astype(np.float64), v)   # exact in float32
        assert (v > 0).mean() > 0.99 and v.min() > -57 and v.max() < 328


def test_values_agree_between_numpy_and_torch():
    import torch
    i = _sample_indices()
    for ncell, cel in ((QCELL, Q_CELSIUS), (C_CELL, C_CELSIUS)):
        got = value_torch(torch.from_numpy(i), ncell, cel).numpy()
        assert np.array_equal(got, value_np(i, ncell, cel))
    c = np.arange(*Q_CELSIUS[0])
    assert (value_np(c + 7 * QCELL, QCELL, Q_CELSIUS) < 72).all()
    assert (value_np(c + 7 * QCELL, QCELL, Q_CELSIUS) < 0).any()


def _assert_rejected(fx, idx_good, idx_bad, ncell, cel, kind="identity", params=(), n_out=1, what=""):
    assert not np.array_equal(idx_good, idx_bad), what
    ref, base, sny = ref_of(fx, kind, params, n_out, idx_good, ncell, cel)
    bad, _, _ = ref_of(fx, kind, params, n_out, idx_bad, ncell, cel)
    check(ref, ref, base, sny, "large self")
    with pytest.raises(AssertionError):
        check(bad, ref, base, sny, "large mutant " + what)


def test_comparator_rejects_32_bit_addresses():
    """The references of cases A, C, F and I computed with addresses wrapped at 32 bits (elements mod 2^31,
    bytes mod 2^32) fail ``check``: the suite sees the bug class."""
    _, fq, uq = region_table(QLAT_L, QLON_L, q_regions(), 1)
    days = np.arange(CROSS - 3, T32)
    a = tm_index(days, uq, QCELL)                                                    # A
    _assert_rejected(fq, a, wrap_elements(a), QCELL, Q_CELSIUS, what="A")
    cm = cm_index(days, uq, T32)                                                     # F, cell-major
    _assert_rejected(fq, cm, wrap_elements(cm), QCELL, Q_CELSIUS, what="F")
    tix = np.array([2087, 5, CROSS, CROSS + 1, 0, 2080, 1036])                       # I (as an aggregate)
    gi = tm_index(tix, uq, QCELL)
    _assert_rejected(fq, gi, wrap_elements(gi), QCELL, Q_CELSIUS, what="I")
    _, fc, uc = region_table(np.arange(C_LAT, dtype=float), np.arange(C_LON, dtype=float),
                             c_regions(C_CELL, 2 ** 29, C_CELSIUS), 2)
    ci = tm_index([1, 0, 1], uc, C_CELL)                                             # C
    _assert_rejected(fc, ci, wrap_plane_bytes(ci, C_CELL, 8), C_CELL, C_CELSIUS, what="C")
    # ... and I's gathered values themselves differ at every wrapped position past 2^31
    over = gi >= (1 << 31)
    assert over.any() and (value_np(gi[over], QCELL, Q_CELSIUS)
                           != value_np(wrap_elements(gi)[over], QCELL, Q_CELSIUS)).all()
    for k in ("large self", "large mutant A", "large mutant F", "large mutant I", "large mutant C"):
        NEEDED.pop(k, None)


def test_shapes_cross_their_boundaries():
    assert (T32 - 1) * QCELL + QCELL - 1 > 2 ** 31 > CROSS * QCELL
    assert QCELL * T32 - 1 >= 2 ** 31                       # G: R * T results, H: n, F: c * T + tp
    assert C_CELL > 2 ** 29 and C_CELL * 8 < 2 ** 33 and C_CELL % 4 == 0
    assert 2 ** 30 - 4 == D_CELL and (D_CELL - 4) * 4 == 2 ** 32 - 32
    assert 1036 * QCELL * 4 > 2 ** 32 and 86 * 24 < CROSS < 87 * 24 <= T32


# ----------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------
GB = 1 << 30
MARGIN = 1 << 30           # workspaces, plans and the gathered pieces


def _need(nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + MARGIN:
        pytest.skip("needs {:,} bytes of device memory ({:.1f} GB) and {:,} are free".format(
            nbytes + MARGIN, (nbytes + MARGIN) / 1e9, free))


def _release():
    import gc
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _fill(n, ncell, celsius, dtype):
    """A flat device buffer of n elements holding value(i), filled 2^26 elements at a time."""
    import torch
    dev = torch.device("cuda", 0)
    buf = torch.empty(n, dtype=dtype, device=dev)
    step = 1 << 26
    for s in range(0, n, step):
        i = torch.arange(s, min(s + step, n), dtype=torch.int64, device=dev)
        buf[s:s + len(i)] = value_torch(i, ncell, celsius).to(dtype)
        del i
    torch.cuda.synchronize()
    return buf


def _gather(buf2d, rows, cols):
    """buf2d[rows][:, cols] gathered on the device, as float64 numpy."""
    import torch
    dev = buf2d.device
    r = torch.as_tensor(np.asarray(rows, np.int64), device=dev)
    c = torch.as_tensor(np.asarray(cols, np.int64), device=dev)
    if len(r) * buf2d.shape[1] <= len(c) * buf2d.shape[0]:      # the smaller intermediate first
        return buf2d.index_select(0, r).index_select(1, c).double().cpu().numpy()
    return buf2d.index_select(1, c).index_select(0, r).double().cpu().numpy()


def _assert_filled(buf2d, rows, cols, idx, ncell, celsius):
    """The device holds value() where the reference reads it."""
    got = _gather(buf2d, rows, cols)
    assert np.array_equal(got, value_np(idx, ncell, celsius)), "fill differs from value()"


@pytest.fixture(scope="module")
def q32():
    """The float32 buffer [T32, QCELL] (8.7 GB), shared by the 0.25 degree cases."""
    import torch
    _need(T32 * QCELL * 4)
    buf = _fill(T32 * QCELL, QCELL, Q_CELSIUS, torch.float32)
    yield buf
    del buf
    _release()


def _plan(lat, lon, df, es, n_in=1, split=False, compact=False):
    import torch
    from climate_toolbox_b200 import _engine as E
    stage = n_in * es
    return E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=stage,
                      device=torch.device("cuda", 0), smem_budget=33 * stage * 16 if split else 0, cache=False,
                      compact=compact, elem_bytes=es)


def _agg(plan, x0, x1, stride, tix, T, kind="identity", params=(), n_out=1, variant=N.VARIANT_STAGED,
         layout=N.LAYOUT_TIME_MAJOR):
    from climate_toolbox_b200 import _engine as E
    return E.aggregate_device(plan, x0, x1, layout, stride, tix, T, kind, params, n_out, variant=variant)


def _check_split(plan_split, label):
    assert plan_split.info["n_split_regions"] > 0, (label, plan_split.info)


@pytest.mark.gpu
def test_a_and_b_streaming_past_2_31_elements_f32(q32):
    """A: the streaming kernel without a time index over 2,088 float32 planes, whole and split plans.  B: a
    time index picking planes on both sides of 2^31 (repeated, out of order); with tix = arange(T) it equals A
    bit for bit."""
    import torch
    df, fx, uq = region_table(QLAT_L, QLON_L, q_regions(), 1)
    x = q32.view(T32, QCELL)
    whole, split = _plan(QLAT_L, QLON_L, df, 4), _plan(QLAT_L, QLON_L, df, 4, split=True)
    _check_split(split, "A")
    idx = tm_index(np.arange(T32), uq, QCELL)
    _assert_filled(x, np.arange(T32), uq, idx, QCELL, Q_CELSIUS)
    ref = ref_of(fx, "identity", (), 1, idx, QCELL, Q_CELSIUS)
    a = _agg(whole, x, None, QCELL, None, T32)
    check(a.cpu().numpy(), *ref, "A whole")
    check(_agg(split, x, None, QCELL, None, T32).cpu().numpy(), *ref, "A split")
    b_id = _agg(whole, x, None, QCELL, np.arange(T32), T32)
    assert torch.equal(b_id.view(torch.int64), a.view(torch.int64)), "B with tix = arange(T) differs from A"
    tix = _b_tix()
    ref = ref_of(fx, "identity", (), 1, tm_index(tix, uq, QCELL), QCELL, Q_CELSIUS)
    check(_agg(whole, x, None, QCELL, tix, len(tix)).cpu().numpy(), *ref, "B f32")
    # the polynomial instantiation with its time index: four outputs of every value
    params = (273.15, 1.0, 2.0, 3.0, 4.0)
    ref = ref_of(fx, "poly", params, 4, tm_index(tix, uq, QCELL), QCELL, Q_CELSIUS)
    check(_agg(split, x, None, QCELL, tix, len(tix), "poly", params, 4).cpu().numpy(), *ref, "B f32 poly split")
    whole.close()
    split.close()


def _b_tix(T=T32):
    rng = np.random.default_rng(8)
    around = np.r_[np.arange(CROSS - 20, min(CROSS + 17, T)), np.arange(T - 16, T)]
    t = np.r_[around, rng.choice(around, 40), rng.integers(0, T, 25), [CROSS, CROSS, 0, T - 1, 1035, 1036]]
    return rng.permutation(t).astype(np.int64)


@pytest.mark.gpu
def test_b_streaming_time_index_past_2_31_elements_f64():
    """B in float64: 2,080 planes (17.3 GB), a time index on both sides of 2^31 elements (and of 2^32 bytes at
    plane 518), whole and split plans; tix = arange(T) against no time index bit for bit."""
    import torch
    _need(T64 * QCELL * 8)
    buf = _fill(T64 * QCELL, QCELL, Q_CELSIUS, torch.float64)
    x = buf.view(T64, QCELL)
    df, fx, uq = region_table(QLAT_L, QLON_L, q_regions(), 3)
    whole, split = _plan(QLAT_L, QLON_L, df, 8), _plan(QLAT_L, QLON_L, df, 8, split=True)
    tix = np.r_[_b_tix(T64), [517, 518, 519]]
    idx = tm_index(tix, uq, QCELL)
    _assert_filled(x, tix, uq, idx, QCELL, Q_CELSIUS)
    ref = ref_of(fx, "identity", (), 1, idx, QCELL, Q_CELSIUS)
    check(_agg(whole, x, None, QCELL, tix, len(tix)).cpu().numpy(), *ref, "B f64")
    check(_agg(split, x, None, QCELL, tix, len(tix)).cpu().numpy(), *ref, "B f64 split")
    days = np.r_[np.arange(0, 64), np.arange(CROSS - 40, T64)]
    a = _agg(whole, x, None, QCELL, None, T64)
    assert torch.equal(_agg(whole, x, None, QCELL, np.arange(T64), T64).view(torch.int64), a.view(torch.int64))
    ref = ref_of(fx, "identity", (), 1, tm_index(days, uq, QCELL), QCELL, Q_CELSIUS)
    check(a[:, :, days].cpu().numpy(), *ref, "A f64")
    whole.close()
    split.close()
    del x, buf, a
    _release()


def _c_case(nlat, nlon, es, celsius, b, n_planes, tix, label):
    """A full-grid plan of nlat x nlon cells with regions around cell b, n_planes planes, time index tix:
    whole and split plans against the reference."""
    import torch
    ncell = nlat * nlon
    _need(n_planes * ncell * es)
    lat, lon = np.arange(nlat, dtype=np.float64), np.arange(nlon, dtype=np.float64)
    df, fx, uc = region_table(lat, lon, c_regions(ncell, b, celsius), 2)
    whole = _plan(lat, lon, df, es)
    split = _plan(lat, lon, df, es, split=True)
    _check_split(split, label)
    buf = _fill(n_planes * ncell, ncell, celsius, torch.float32 if es == 4 else torch.float64)
    x = buf.view(n_planes, ncell)
    idx = tm_index(tix, uc, ncell)
    _assert_filled(x, tix, uc, idx, ncell, celsius)
    ref = ref_of(fx, "identity", (), 1, idx, ncell, celsius)
    check(_agg(whole, x, None, ncell, tix, len(tix)).cpu().numpy(), *ref, label + " whole")
    check(_agg(split, x, None, ncell, tix, len(tix)).cpu().numpy(), *ref, label + " split")
    params = (273.15, 1.0, 2.0)
    ref = ref_of(fx, "poly", params, 2, idx, ncell, celsius)
    check(_agg(whole, x, None, ncell, tix, len(tix), "poly", params, 2).cpu().numpy(), *ref, label + " poly")
    whole.close()
    split.close()
    del x, buf
    _release()


@pytest.mark.gpu
def test_c_time_index_f64_plane_past_4_gib():
    """C: a float64 full-grid plan of 16,400 x 32,768 cells (>= 2^29), two planes, tix = [1, 0, 1]: cells at or
    past 2^29 lie 4 GiB or more into their plane.  A 32-bit byte offset reads the cell 2^29 earlier."""
    _c_case(C_LAT, C_LON, 8, C_CELSIUS, 2 ** 29, 2, np.array([1, 0, 1]), "C")


@pytest.mark.gpu
def test_d_time_index_f32_plane_just_under_the_plan_limit():
    """D: float32, a grid of 2^30 - 4 cells (byte offsets up to 2^32 - 32 must still hold) with regions around
    2^29 and at the plane's end; a grid of 2^30 cells is refused with CTB_ERR_INVALID before any launch."""
    import torch
    from climate_toolbox_b200 import _engine as E
    _c_case(D_LAT, D_LON, 4, D_CELSIUS, 2 ** 29, 1, np.array([0, 0]), "D")
    lat = np.arange(32768, dtype=np.float64)
    df = pd.DataFrame({"lat": [0.0], "lon": [0.0], "hierid": [0], "popwt": [1.0], "areawt": [1.0]})
    n0 = E.launch_count()
    with pytest.raises(ValueError, match="invalid sizes"):
        E.get_plan(E.GridSpec(lat, lat), df, "popwt", "hierid", device=torch.device("cuda", 0), cache=False)
    assert E.launch_count() == n0


@pytest.mark.gpu
def test_e_two_input_views_past_2_31_elements(q32):
    """E: Snyder EDD and GDD with x0 = buf[0:T], x1 = buf[1:T+1] (the r1 / X1 addresses), with and without a
    time index, whole and split plans."""
    df, fx, uq = region_table(QLAT_L, QLON_L, q_regions(), 4)
    x = q32.view(T32, QCELL)
    x0, x1 = x[0:T32 - 1], x[1:T32]
    whole, split = _plan(QLAT_L, QLON_L, df, 4, n_in=2), _plan(QLAT_L, QLON_L, df, 4, n_in=2, split=True)
    _check_split(split, "E")
    tix = _b_tix(T32 - 1)
    days = np.r_[np.arange(0, 8), np.arange(CROSS - 24, T32 - 1)]
    for kind, params, n_out in (("edd", (-100.0,), 1), ("gdd", (-100.0, 600.0), 1), ("edd", (-100.0, -80.0), 2)):
        for plan, pl in ((whole, "whole"), (split, "split")):
            ref = ref_of(fx, kind, params, n_out, tm_index(tix, uq, QCELL), QCELL, Q_CELSIUS,
                         idx1=tm_index(tix, uq, QCELL, QCELL))
            got = _agg(plan, x0, x1, QCELL, tix, len(tix), kind, params, n_out)
            check(got.cpu().numpy(), *ref, "E {} {} tix {}".format(kind, n_out, pl))
            ref = ref_of(fx, kind, params, n_out, tm_index(days, uq, QCELL), QCELL, Q_CELSIUS,
                         idx1=tm_index(days, uq, QCELL, QCELL))
            got = _agg(plan, x0, x1, QCELL, None, T32 - 1, kind, params, n_out)
            check(got[:, :, days].cpu().numpy(), *ref, "E {} {} {}".format(kind, n_out, pl))
    whole.close()
    split.close()


@pytest.mark.gpu
def test_f_direct_kernel_past_2_31_elements(q32):
    """F: the direct kernel, time-major (tp * stride + c) with and without a time index, and cell-major on the
    [QCELL, T32] view of the same storage (c * stride + tp past 2^31 for the last rows)."""
    df, fx, uq = region_table(QLAT_L, QLON_L, q_regions(), 5)
    plan = _plan(QLAT_L, QLON_L, df, 4)
    tm = q32.view(T32, QCELL)
    cm = q32.view(QCELL, T32)
    tix = _b_tix()
    days = np.r_[np.arange(0, 8), np.arange(CROSS - 24, T32)]
    ref = ref_of(fx, "identity", (), 1, tm_index(tix, uq, QCELL), QCELL, Q_CELSIUS)
    got = _agg(plan, tm, None, QCELL, tix, len(tix), variant=N.VARIANT_DIRECT)
    check(got.cpu().numpy(), *ref, "F direct time-major tix")
    ref = ref_of(fx, "identity", (), 1, tm_index(days, uq, QCELL), QCELL, Q_CELSIUS)
    got = _agg(plan, tm, None, QCELL, None, T32, variant=N.VARIANT_DIRECT)
    check(got[:, :, days].cpu().numpy(), *ref, "F direct time-major")
    assert cm_index([T32 - 1], uq, T32).max() >= 2 ** 31
    _assert_filled(cm, uq, tix, cm_index(tix, uq, T32).T, QCELL, Q_CELSIUS)
    ref = ref_of(fx, "identity", (), 1, cm_index(tix, uq, T32), QCELL, Q_CELSIUS)
    got = _agg(plan, cm, None, T32, tix, len(tix), variant=N.VARIANT_DIRECT, layout=N.LAYOUT_CELL_MAJOR)
    check(got.cpu().numpy(), *ref, "F direct cell-major tix")
    ref = ref_of(fx, "identity", (), 1, cm_index(days, uq, T32), QCELL, Q_CELSIUS)
    got = _agg(plan, cm, None, T32, None, T32, variant=N.VARIANT_DIRECT, layout=N.LAYOUT_CELL_MAJOR)
    check(got[:, :, days].cpu().numpy(), *ref, "F direct cell-major")
    plan.close()


@pytest.mark.gpu
def test_g_one_region_per_cell_past_2_31_results(q32):
    """G: one region per gridcell of the 0.25 degree grid over 2,088 days: R * T > 2^31 results (17.3 GB of
    float64).  With power-of-two weights a one-cell region's aggregate is its value exactly, so every result is
    compared on the device with the widened input; sampled rows against the fsum reference."""
    import torch
    _need(QCELL * T32 * 8)
    groups = [np.array([c]) for c in range(QCELL)]
    df, fx, _ = region_table(QLAT_L, QLON_L, groups, 6, unit_weights=True)
    plan = _plan(QLAT_L, QLON_L, df, 4)
    assert plan.R == QCELL
    x = q32.view(T32, QCELL)
    out = _agg(plan, x, None, QCELL, None, T32)
    step = 1 << 16
    for r0 in range(0, QCELL, step):
        r1 = min(r0 + step, QCELL)
        assert torch.equal(out[0, r0:r1], x[:, r0:r1].t().double()), "regions {}..{}".format(r0, r1)
    rows = np.r_[0, 1, 2 ** 19, np.arange(QCELL - 6, QCELL)]           # region r is cell r, weights row r
    sub = {"R": len(rows), "members": [np.array([k]) for k in range(len(rows))], "row_cell": np.arange(len(rows)),
           "w_eff": fx["w_eff"][rows]}
    days = np.r_[np.arange(0, 4), np.arange(CROSS - 4, T32)]
    ref = ref_of(sub, "identity", (), 1, tm_index(days, rows, QCELL), QCELL, Q_CELSIUS)
    got = out[:, torch.as_tensor(rows, device=out.device)][:, :, torch.as_tensor(days, device=out.device)]
    check(got.cpu().numpy(), *ref, "G sampled rows")
    plan.close()
    del out, x
    _release()


def _transform(x, n, kind_code, params, n_out, out):
    import torch
    from climate_toolbox_b200 import _engine as E
    pa = np.ascontiguousarray(params, dtype=np.float64)
    N.check(N.lib().ctb_transform(C.c_void_p(x.data_ptr()), None, N.F32 if x.dtype == torch.float32 else N.F64, n,
                                  kind_code, pa.ctypes.data_as(C.POINTER(C.c_double)), int(pa.size), n_out,
                                  C.c_void_p(out.data_ptr()), E._stream_ptr(x.device)))


@pytest.mark.gpu
def test_h_pointwise_transform_past_2_31_elements(q32):
    """H: ctb_transform (the ``.values`` of a tas_poly term) over n = 2,164,838,400 float32 values into 17.3 GB:
    every result equals x - 273.15 in float64 on the device; sampled ones against value()."""
    import torch
    n = T32 * QCELL
    _need(n * 8)
    out = torch.empty(n, dtype=torch.float64, device=q32.device)
    _transform(q32, n, N.TR_POLY, (273.15, 1.0), 1, out)
    step = 1 << 27
    for s in range(0, n, step):
        e = min(s + step, n)
        assert torch.equal(out[s:e], q32[s:e].double() - 273.15), "elements {}..{}".format(s, e)
    rng = np.random.default_rng(9)
    i = np.unique(np.r_[np.arange(2 ** 31 - 64, 2 ** 31 + 64), np.arange(n - 64, n), rng.integers(0, n, 4096)])
    got = out[torch.as_tensor(i, device=out.device)].cpu().numpy()
    want = value_np(i, QCELL, Q_CELSIUS) - 273.15
    check(got[None], want[None], U * np.abs(want)[None], np.zeros((1, len(i))), "H pointwise", c=1)
    del out
    _release()


def _gather_rows(plan, x, stride, layout, tix):
    import torch
    from climate_toolbox_b200 import _engine as E
    t = torch.as_tensor(np.asarray(tix, np.int32), device=x.device)
    out = torch.empty(len(tix) * plan.n_rows, dtype=x.dtype, device=x.device)
    N.check(N.lib().ctb_gather_rows(plan._h, C.c_void_p(x.data_ptr()), N.F32, layout, int(stride),
                                    C.c_void_p(t.data_ptr()), len(tix), C.c_void_p(out.data_ptr()),
                                    E._stream_ptr(x.device)))
    return out.double().cpu().numpy()


@pytest.mark.gpu
def test_i_gather_rows_past_2_31_elements(q32):
    """I: ctb_gather_rows (``.values`` of a reindexed variable) reading planes past 2^31 elements, time-major
    and cell-major on the two views of one buffer, bit for bit."""
    df, fx, uq = region_table(QLAT_L, QLON_L, q_regions(), 7)
    plan = _plan(QLAT_L, QLON_L, df, 4)
    cells = plan.row_cells().astype(np.int64)
    tix = _b_tix()
    got = _gather_rows(plan, q32, QCELL, N.LAYOUT_TIME_MAJOR, tix).reshape(len(tix), -1)
    assert np.array_equal(got, value_np(tm_index(tix, cells, QCELL), QCELL, Q_CELSIUS)), "time-major"
    got = _gather_rows(plan, q32, T32, N.LAYOUT_CELL_MAJOR, tix).reshape(-1, len(tix))
    assert np.array_equal(got, value_np(cm_index(tix, cells, T32).T, QCELL, Q_CELSIUS)), "cell-major"
    plan.close()


def _one_cell_plan(cells, es, seed):
    groups = [np.array([c]) for c in cells]
    df, fx, _ = region_table(QLAT_L, QLON_L, groups, seed, unit_weights=True)
    return _plan(QLAT_L, QLON_L, df, es, compact=True)


J_CELLS = np.r_[np.arange(0, 8), np.arange(QCELL - 16, QCELL), np.arange(2 ** 19 - 3, 2 ** 19 + 5),
                np.arange(*Q_CELSIUS[0])[::97], np.random.default_rng(10).choice(QCELL, 40, replace=False)]
J_TIX = np.array([0, 1035, 1036, 1037, CROSS, CROSS + 1, T32 - 1, 1036, 5, 1039, 2000])


def _pull(plan, src_ptr, tix, es, dev):
    """ctb_pull_pack of the planes ``tix`` of a [*, QCELL] source, then the one-cell-region aggregate of the
    packed planes: [R, T] float64 values, exact."""
    import torch
    from climate_toolbox_b200 import _engine as E
    width = plan.info["n_packed_cells"]
    t = torch.as_tensor(tix.astype(np.int32), device=dev)
    dst = torch.empty((len(tix), width), dtype=torch.float32, device=dev)
    N.check(N.lib().ctb_pull_pack(plan._h, C.c_void_p(src_ptr), N.F32, QCELL, C.c_void_p(t.data_ptr()), 0,
                                  len(tix), C.c_void_p(dst.data_ptr()), E._stream_ptr(dev)))
    return _agg(plan, dst, None, width, None, len(tix))[0]


@pytest.mark.gpu
def test_j_pull_pack_past_4_gib(q32):
    """J: ctb_pull_pack from a device source at planes past 4 GiB (plane 1036 starts at 4,296,499,200 bytes) and
    past 2^31 elements, read back through one-cell regions, bit for bit."""
    plan = _one_cell_plan(J_CELLS, 4, 11)
    got = _pull(plan, q32.data_ptr(), J_TIX, 4, q32.device).cpu().numpy()
    assert np.array_equal(got, value_np(tm_index(J_TIX, J_CELLS, QCELL), QCELL, Q_CELSIUS).T)
    plan.close()


@pytest.mark.gpu
def test_j_pull_pack_pinned_host_past_4_gib(q32):
    """J from pinned host memory: 1,040 planes (4.3 GB, page-locked in place) copied from the device buffer,
    pulled at planes past 4 GiB, equal bit for bit to the pull from the device."""
    import torch
    n = 1040 * QCELL
    host = np.empty(n, dtype=np.float32)
    rt = torch.cuda.cudart()
    rc = rt.cudaHostRegister(host.ctypes.data, host.nbytes, 3)       # portable | mapped
    if int(rc) != 0:
        pytest.skip("cannot pin {:,} bytes of host memory (cudaHostRegister returned {})".format(host.nbytes, rc))
    try:
        torch.from_numpy(host).copy_(q32[:n])
        plan = _one_cell_plan(J_CELLS, 4, 11)
        tix = J_TIX[J_TIX < 1040]
        got = _pull(plan, host.ctypes.data, tix, 4, q32.device)
        want = _pull(plan, q32.data_ptr(), tix, 4, q32.device)
        assert torch.equal(got.view(torch.int64), want.view(torch.int64))
        assert np.array_equal(got.cpu().numpy(), value_np(tm_index(tix, J_CELLS, QCELL), QCELL, Q_CELSIUS).T)
        plan.close()
    finally:
        torch.cuda.synchronize()
        rt.cudaHostUnregister(host.ctypes.data)


@pytest.mark.gpu
def test_j_pull_pack_daily_hourly_past_2_31_steps(q32):
    """J: ctb_pull_pack_daily on the hourly view (S = 24, 87 days) of the float32 buffer: day 86 reads steps
    past 2^31 elements.  Daily mean, min and max bit for bit against ``test_subdaily.resample_daily_ref``."""
    import torch
    from climate_toolbox_b200 import _engine as E
    S = 24
    days = np.array([0, 86, 43, 86, 85, 1, 86])
    dev = q32.device
    day_t = torch.as_tensor(days.astype(np.int32), device=dev)
    steps = (days[:, None] * S + np.arange(S)[None]).reshape(-1)
    hourly = value_np(tm_index(steps, J_CELLS, QCELL), QCELL, Q_CELSIUS).astype(np.float32)
    _assert_filled(q32.view(T32, QCELL), steps, J_CELLS, tm_index(steps, J_CELLS, QCELL), QCELL, Q_CELSIUS)
    for es, ops, hows in ((8, N.DAILY_MEAN, ("mean",)), (4, N.DAILY_MIN | N.DAILY_MAX, ("min", "max"))):
        plan = _one_cell_plan(J_CELLS, es, 12)
        width = plan.info["n_packed_cells"]
        dst = {h: torch.empty((len(days), width), dtype=torch.float64 if h == "mean" else torch.float32, device=dev)
               for h in hows}
        ptr = lambda h: C.c_void_p(dst[h].data_ptr()) if h in dst else None  # noqa: E731
        N.check(N.lib().ctb_pull_pack_daily(plan._h, C.c_void_p(q32.data_ptr()), N.F32, QCELL, S,
                                            C.c_void_p(day_t.data_ptr()), 0, len(days), ops, ptr("mean"),
                                            ptr("min"), ptr("max"), E._stream_ptr(dev)))
        for h in hows:
            got = _agg(plan, dst[h], None, width, None, len(days))[0].cpu().numpy()
            want = resample_daily_ref(hourly, S, h).astype(np.float64).T
            assert np.array_equal(got, want), h
        plan.close()


# thresholds and edges that split both the kelvin values and the Celsius range
J_STEPS = (("edd", N.STEP_EDD, (0.0, 290.0), (0.0, 290.0)),
           ("gdd", N.STEP_GDD, (10.0, 30.0, 250.0, 300.0), ((10.0, 30.0), (250.0, 300.0))),
           ("bins", N.STEP_BINS, (0.0, 260.0, 300.0), (0.0, 260.0, 300.0)))


@pytest.mark.gpu
@pytest.mark.parametrize("op,step_op,params,ref_params", J_STEPS, ids=[s[0] for s in J_STEPS])
def test_j_pull_pack_daily_steps_hourly_past_2_31_steps(q32, op, step_op, params, ref_params):
    """J: ctb_pull_pack_daily_steps on the same hourly view: day 86 reads steps past 2^31 elements through the step
    loop that subdaily_pack_kernel shares.  Two outputs of EDD, GDD and bins, bit for bit against
    ``test_subdaily_steps.steps_ref``."""
    import torch
    from climate_toolbox_b200 import _engine as E
    S = 24
    days = np.array([0, 86, 43, 86, 85, 1, 86])
    dev = q32.device
    day_t = torch.as_tensor(days.astype(np.int32), device=dev)
    steps = (days[:, None] * S + np.arange(S)[None]).reshape(-1)
    hourly = value_np(tm_index(steps, J_CELLS, QCELL), QCELL, Q_CELSIUS).astype(np.float32)
    plan = _one_cell_plan(J_CELLS, 8, 12)
    width = plan.info["n_packed_cells"]
    dst = [torch.empty((len(days), width), dtype=torch.float64, device=dev) for _ in range(2)]
    prm = (C.c_double * len(params))(*params)
    ptrs = (C.c_void_p * 2)(*[d.data_ptr() for d in dst])
    N.check(N.lib().ctb_pull_pack_daily_steps(plan._h, C.c_void_p(q32.data_ptr()), N.F32, QCELL, S,
                                              C.c_void_p(day_t.data_ptr()), 0, len(days), step_op, prm, len(params),
                                              2, ptrs, E._stream_ptr(dev)))
    for j, want in enumerate(steps_ref(hourly, S, op, ref_params)):
        got = _agg(plan, dst[j], None, width, None, len(days))[0].cpu().numpy()
        assert np.array_equal(got, want.T), (op, j)
    plan.close()
