/* ctb.h -- C-ABI of libctb.so: B200 (sm_100a) grid->region aggregation.
 *
 * The reference (ClimateImpactLab/climate_toolbox) has NO FFI layer for this
 * path: it is a plain Python function API over xarray
 * (climate_toolbox/aggregations/aggregations.py:87-124).  This header is the
 * boundary a maintainer would bind (ctypes, see INTEGRATION.md) to replace the
 * bodies of:
 *
 *   _reindex_spatial_data_to_regions      aggregations.py:8-32   -> ctb_plan_build, ctb_gather_rows
 *   _aggregate_reindexed_data_to_regions  aggregations.py:35-84  -> ctb_plan_build (weights, den), ctb_aggregate
 *   tas_poly arithmetic                   transformations.py:189 -> ctb_aggregate(transform=POLY) / ctb_transform
 *   snyder_edd / snyder_gdd arithmetic    transformations.py:69-89, 139-141
 *                                                                 -> ctb_aggregate(transform=EDD|GDD) / ctb_transform
 *   convert_lons_split data shuffle       utils/utils.py:33-40   -> lon_phys[] of ctb_plan_build (index remap, no copy)
 *   remove_leap_days data copy            utils/utils.py:77-80   -> time_index[] of ctb_aggregate
 *
 * Conventions: plain pointers + sizes, no C++/torch types.  "host" pointers are
 * read on the CPU during the call; "device" pointers must be CUDA device memory
 * on the plan's device and are only touched by stream-ordered work on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream).  Every entry
 * point returns CTB_OK (0) or a CTB_ERR_* code; ctb_last_error() gives the
 * thread-local message.  A plan is immutable after build and may be shared
 * across threads and streams.  There is no CPU fallback anywhere: without a
 * CUDA device every compute entry point fails with CTB_ERR_CUDA.
 */
#ifndef CTB_H_
#define CTB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTB_VERSION 100

/* ---- status codes ------------------------------------------------------ */
enum {
  CTB_OK = 0,
  CTB_ERR_LABEL_NOT_FOUND = 1, /* a weights row's lat/lon label is not in the grid
                                  (exact float64 equality; xarray .sel KeyError,
                                  aggregations.py:27).  *bad_row = first such row */
  CTB_ERR_CUDA = 2,
  CTB_ERR_INVALID = 3,
  CTB_ERR_UNSUPPORTED = 4
};

/* ---- enums --------------------------------------------------------------- */
enum { CTB_F32 = 0, CTB_F64 = 1 };

/* memory layout of the gridded input seen as 2-D (time, flat cell):
 *   TIME_MAJOR: x[t * plane_stride + cell]   BCSD netCDF (time, lat, lon)
 *   CELL_MAJOR: x[cell * cell_stride + t]    reference test fixture (lat, lon, time) */
enum { CTB_LAYOUT_TIME_MAJOR = 0, CTB_LAYOUT_CELL_MAJOR = 1 };

/* gridcell-level transforms fused into the gather (params are host doubles):
 *   IDENTITY  n_in=1            f = x
 *   POLY      n_in=1  params = {offset, p_1..p_nout}   f_j = (x - offset)^p_j   transformations.py:189
 *   EDD       n_in=2  params = {e_1..e_nout}           f_j = SnyderEDD(tmin=x0,tmax=x1,e_j)  transformations.py:69-89
 *   GDD       n_in=2  params = {lo_1,hi_1,..}          f_j = EDD(lo_j) - EDD(hi_j)           transformations.py:139-141
 *   BINS      n_in=1  params = {offset, e_0..e_nout}   f_j = [e_j <= x - offset < e_{j+1}]   (NaN for NaN x; edges strictly
 *                     increasing, not NaN, only e_0 may be -inf and only e_nout +inf; n_params = n_out + 2)
 *   RCSPLINE  n_in=1  params = {offset, first, k_1..k_n}   f_j = B_{first+j}(x - offset), the restricted cubic spline
 *                     basis of the knots k (Harrell's unnormalised form), d = x - offset, c(k) = max(d - k, 0)^3:
 *                       B_0(d) = d
 *                       B_i(d) = c(k_i) - c(k_{n-1}) (k_n - k_i)/(k_n - k_{n-1}) + c(k_n) (k_{n-1} - k_i)/(k_n - k_{n-1})
 *                     for 1 <= i <= n-2 (NaN propagates; +inf gives NaN for i >= 1).  3 <= n <= 7 finite, strictly
 *                     increasing knots, a finite offset, an integer first >= 0 with first + n_out <= n - 1;
 *                     n_params = n + 2 */
enum { CTB_TR_IDENTITY = 0, CTB_TR_POLY = 1, CTB_TR_EDD = 2, CTB_TR_GDD = 3, CTB_TR_BINS = 4, CTB_TR_RCSPLINE = 5 };
#define CTB_MAX_OUT 4

typedef struct ctb_plan ctb_plan;

/* Planner knobs (all optional; zero = default). */
typedef struct ctb_plan_opts {
  int32_t stage_bytes_per_cell_day; /* bytes one gridcell-day occupies in the staging
                                       tile: n_in * sizeof(elem); default 4 (one f32) */
  int32_t smem_budget_bytes;        /* cap on one staging tile in bytes (tests use it to force
                                       region splitting); default: 128 16-byte units per day */
  int32_t compact;                  /* 1: the plan addresses a PACKED input [T][n_packed_cells]
                                       holding only the referenced 4-cell pieces (what
                                       ctb_host_pack writes) instead of the full grid */
  int32_t elem_bytes;               /* 4 (default) or 8: element size of the inputs this plan will
                                       aggregate (staged-cell byte offsets are baked into the plan) */
  int32_t reserved[4];
  const uint32_t* cell_gate;        /* HOST [nlat_phys * nlon_phys], nullable: growing-season gate of every
                                       physical gridcell, first_day | last_day << 9 | wrap << 18 (day of year
                                       0..511): the gridcell-day counts when (first <= doy <= last) != wrap.
                                       Replaces the lat x lon x time mask of utils.py:83-153; applied by
                                       ctb_aggregate_ex when day_of_year is given */
} ctb_plan_opts;

typedef struct ctb_plan_info {
  int64_t n_rows;          /* rows of the weights table */
  int64_t nnz;             /* rows kept in the CSR (finite, non-zero weight, valid region) */
  int64_t n_cells_distinct;/* U: distinct referenced gridcells (of kept rows) */
  int64_t n_cells_grid;    /* nlat_phys * nlon_phys */
  int32_t n_regions;       /* R */
  int32_t n_bundles;       /* staging work units (x time blocks = CTAs) */
  int64_t n_pieces;        /* 4-cell pieces staged per time step, summed over bundles */
  int64_t n_pieces_distinct;/* distinct pieces (DRAM-side footprint per time step) */
  int32_t n_split_regions; /* regions larger than one bundle (two-phase reduce) */
  int32_t n_scratch_slots; /* partial-sum rows those regions need */
  int32_t cap_cells;       /* staging capacity per bundle in cells */
  int32_t max_bundle_cells;
  int32_t time_block;      /* days per staging tile */
  int32_t max_region_rows; /* largest region, in kept rows */
  int32_t max_meta_bytes;  /* largest per-bundle metadata blob + piece list, bytes */
  int32_t n_packed_cells;  /* compact plans: cells per packed plane (4 * distinct pieces), else 0 */
  int64_t n_quads;         /* 4-entry groups the streaming kernel reduces per 32-day tile */
  int64_t n_quads_conflict;/* ... of which hold two columns of one residue class (2-way bank conflict) */
} ctb_plan_info;

/* ---- misc ---------------------------------------------------------------- */
int ctb_version(void);
const char* ctb_last_error(void);
/* number of kernel launches issued by this library since load (for gpu_launches). */
int64_t ctb_launch_count(void);

/* ---- K0: one-time plan (region-sorted CSR + staging bundles) on device --- *
 * Replaces aggregations.py:24-27 (label -> index, exact match) and :64-73
 * (per-row fallback weight, region grouping).  All pointer args are HOST.
 *
 *  grid_lat[nlat], grid_lon[nlon] : the dataset's coordinate labels (logical order)
 *  lat_phys[nlat], lon_phys[nlon] : physical position of each label along the
 *        stored axis (NULL = identity).  A lazily standardised 0..360 grid
 *        (utils.py:33-40) passes the sorted -180..180 labels in grid_lon and
 *        the roll permutation in lon_phys.
 *  nlat_phys, nlon_phys           : stored grid extents (cell = i*nlon_phys + j)
 *  row_lat/row_lon[n_rows]        : weights["lat"], weights["lon"]
 *  region_code[n_rows]            : 0..n_regions-1 = rank of weights[agglev] among its
 *        sorted unique values (pd.factorize(sort=True)); -1 = NaN label (dropped)
 *  w_primary/w_backup[n_rows]     : weights[aggwt], weights[backup_aggwt];
 *        w = w_primary > 0 ? w_primary : w_backup            (aggregations.py:73)
 *  bad_row (nullable)             : first row without a match on CTB_ERR_LABEL_NOT_FOUND,
 *        bad_axis: 0 = lat, 1 = lon
 */
int ctb_plan_build(const double* grid_lat, int32_t nlat, const int32_t* lat_phys, int32_t nlat_phys,
                   const double* grid_lon, int32_t nlon, const int32_t* lon_phys, int32_t nlon_phys,
                   const double* row_lat, const double* row_lon, const int32_t* region_code,
                   const double* w_primary, const double* w_backup, int64_t n_rows,
                   int32_t n_regions, const ctb_plan_opts* opts, int device, ctb_plan** out,
                   int64_t* bad_row, int32_t* bad_axis);
void ctb_plan_free(ctb_plan* plan);
int ctb_plan_get_info(const ctb_plan* plan, ctb_plan_info* info);
/* HOST outputs: physical flat cell of every weights row (bit-exact index map), and
 * den[r] = sum of nan->0(w) per region (aggregations.py:79). */
int ctb_plan_row_cells(const ctb_plan* plan, int32_t* cells_out /*[n_rows]*/);
int ctb_plan_den(const ctb_plan* plan, double* den_out /*[n_regions]*/);
int ctb_plan_row_weights(const ctb_plan* plan, double* w_out /*[n_rows]*/);
/* HOST output: position of every region along the plan's bundle sequence (a permutation of 0..R-1 that
 * keeps spatial neighbours together); the row order ctb_agg_opts.peer_row is meant for */
int ctb_plan_region_order(const ctb_plan* plan, int32_t* pos_out /*[n_regions]*/);

/* ---- K1+K2(+K3): fused stage + gather + segmented weighted sum ----------- *
 * Replaces aggregations.py:75-82 (and the gather of :27) with the transform of
 * transformations.py fused at gridcell level.
 *
 *  x0, x1        : DEVICE inputs (x1 only for n_in = 2), dtype CTB_F32 / CTB_F64
 *  layout        : CTB_LAYOUT_*; stride = plane_stride (TIME_MAJOR) or cell_stride
 *                  (CELL_MAJOR), in elements
 *  time_index    : DEVICE int32[T] physical time step of output step t, or NULL
 *                  for identity (leap-day removal, utils.py:77-80)
 *  out, out_ld   : DEVICE double [n_out][R][out_ld], time contiguous, out_ld >= T
 *                  (0 = T): out[(j*R + r)*out_ld + t] = sum_k nan->0(w_k * f_j(x[cell_k])) / den[r].
 *                  A time-chunked caller passes out + t0 with out_ld = total T.
 *  workspace     : DEVICE scratch of ctb_aggregate_workspace_bytes() bytes (may be
 *                  NULL when that is 0)
 *  variant       : 0 = auto; 1 = the streaming kernel (TIME_MAJOR inputs with 16-byte aligned planes;
 *                  others fall back to 2); 2 = direct warp-per-region kernel.  | 0x100: x0/x1 are MAPPED PINNED HOST memory read
 *                  in place over PCIe (zero-copy: only the referenced gridcells cross the bus)
 */
size_t ctb_aggregate_workspace_bytes(const ctb_plan* plan, int64_t T, int n_out);
int ctb_aggregate(const ctb_plan* plan, const void* x0, const void* x1, int dtype, int layout,
                  int64_t stride, const int32_t* time_index, int64_t T, int transform,
                  const double* params, int n_params, int n_out, double* out, int64_t out_ld,
                  void* workspace, size_t workspace_bytes, int variant, void* stream);

/* ---- everything at once: time reduction and/or growing-season gate ---------- *
 * opts->groups / t_begin / flush: as ctb_aggregate_grouped below.  opts->day_of_year: DEVICE int32,
 * day of year of every day of the time axis ([T], or [groups' T] with a window); with it, gridcell-days
 * outside their gridcell's growing season (ctb_plan_opts.cell_gate) do not enter the numerator -- the
 * fused form of multiplying the data by get_daily_growing_season_mask (utils.py:119-153), whose 0 and
 * NaN both leave the weighted sum untouched while the weight still counts in the denominator. */
typedef struct ctb_time_groups ctb_time_groups;
#define CTB_MAX_PEERS 8
typedef struct ctb_agg_opts {
  const ctb_time_groups* groups;
  int64_t t_begin;
  int32_t flush;
  int32_t n_peer_out;               /* 0, or the number of output buffers the kernel writes (<= CTB_MAX_PEERS) */
  const int32_t* day_of_year;
  double* const* peer_out;          /* HOST array of n_peer_out DEVICE pointers, each laid out like `out`
                                       (this GPU's own buffer and peer-GPU buffers opened with ctb_ipc_open):
                                       the kernel's epilogue stores every result to ALL of them -- the
                                       all-gather of a time-sharded job fused into the aggregation kernel,
                                       over NVLink peer memory.  `out` is ignored then.  Not with groups. */
  const int32_t* peer_row;          /* DEVICE int32[n_regions], nullable: row of every region in the peer
                                       buffers.  ctb_plan_region_order keeps one CTA's stores inside a few
                                       pages: with sorted-label rows a CTA touches ~28 pages per peer and tile,
                                       and 8 peers overflow the TLB (measured: 3.2 ms instead of 0.4) */
} ctb_agg_opts;
int ctb_aggregate_ex(const ctb_plan* plan, const void* x0, const void* x1, int dtype, int layout,
                     int64_t stride, const int32_t* time_index, int64_t T, int transform,
                     const double* params, int n_params, int n_out, const ctb_agg_opts* opts,
                     double* out, int64_t out_ld, void* workspace, size_t workspace_bytes, int variant,
                     void* stream);
/* workspace of ctb_aggregate_ex: ctb_aggregate_workspace_bytes without groups, else the grouped one */

/* ---- peer-shared output buffers (CUDA IPC) for the fused gather ------------ *
 * ctb_ipc_alloc: cudaMalloc on `device` + an IPC handle (64 bytes) another process of the node opens
 * with ctb_ipc_open (peer access enabled on demand); the owner frees with ctb_ipc_free, the others
 * detach with ctb_ipc_close. */
#define CTB_IPC_HANDLE_BYTES 64
int ctb_ipc_alloc(size_t bytes, int device, void** ptr, void* handle_out);
int ctb_ipc_open(const void* handle, int device, void** ptr);
int ctb_ipc_close(void* ptr, int device);
int ctb_ipc_free(void* ptr, int device);
/* The gather as a push: copy columns [t0, t0 + n_cols) of n_rows rows (leading dimension ld, doubles)
 * of `src` (this GPU) to the same place in each of the n_peers mapped buffers (a pointer equal to `src`
 * is skipped).  One kernel, every row piece read once and stored to all peers with coalesced stores
 * over NVLink; stream-ordered.  Measured against NCCL's all_gather + layout copy and against the stores
 * fused into the aggregation kernel's epilogue (ctb_agg_opts.peer_out), one 1460-day batch: 2 ranks 0.63 /
 * 0.80 / 0.41-0.57 ms, 4 ranks 0.62 / 0.75 / 0.59, 8 ranks 0.64 / 0.73 / 0.89 -- the epilogue's 256-byte
 * pieces per region and tile are too scattered for 8 destinations.
 * engine: CTB_PUSH_SM = the copy kernel; CTB_PUSH_COPY_ENGINE = one 2-D DMA per peer (no SM: the only
 * form that overlaps a running aggregation kernel, whose CTAs hold every register of their SM). */
#define CTB_PUSH_SM 0
#define CTB_PUSH_COPY_ENGINE 1
int ctb_push_rows(const double* src, int64_t ld, int64_t t0, int64_t n_cols, int64_t n_rows, int n_peers,
                  double* const* peers, int engine, void* stream);

/* Position-sensitive 64-bit fingerprint of a HOST byte buffer (8 interleaved polynomial lanes over the
 * 64-bit words, mod 2^64): the plan cache of the drop-in re-checks every weights column it built a plan
 * from on every call -- the guard behind the analogue of toolz.memoize (aggregations.py:127) -- and
 * this is what it costs (0.1 ms per 3.4 MB column instead of 0.5 ms in numpy).  No CUDA call. */
uint64_t ctb_fingerprint(const void* data, size_t nbytes);

/* ---- pointwise helpers (materialising what the reference materialises) --- */
/* out[j][i] = f_j(x0[i], x1[i]) for i < n; DEVICE pointers (transformations.py:69-89,189). */
int ctb_transform(const void* x0, const void* x1, int dtype, int64_t n, int transform,
                  const double* params, int n_params, int n_out, double* out, void* stream);
/* The (time, reshape_index) / (reshape_index, time) gather of aggregations.py:27:
 * TIME_MAJOR: out[t*n_rows + k] = x[time_index[t]*stride + cell_k]
 * CELL_MAJOR: out[k*T + t]      = x[cell_k*stride + time_index[t]]   (out dtype = in dtype) */
int ctb_gather_rows(const ctb_plan* plan, const void* x, int dtype, int layout, int64_t stride,
                    const int32_t* time_index, int64_t T, void* out, void* stream);

/* ---- host ingest for compact plans ---------------------------------------- *
 * Packs the referenced gridcells of `T` day-planes of a HOST array x[t_phys][stride] (dtype
 * CTB_F32/F64, TIME_MAJOR) into dst[T][n_packed_cells] (HOST, ideally pinned), multi-threaded.
 * Only ~U/ncell of the input (30 % of a global land/ocean grid) then has to cross PCIe.
 * time_index (HOST int64, nullable) selects the physical planes.  n_threads <= 0: all cores. */
int ctb_host_pack(const ctb_plan* plan, const void* x, int dtype, int64_t stride,
                  const int64_t* time_index, int64_t t_begin, int64_t T, void* dst, int n_threads);

/* The same packing done by the GPU: x is a HOST array in pinned, device-accessible memory
 * (cudaHostAlloc / cudaHostRegister); the referenced pieces are read over PCIe by a kernel on `stream`
 * and written to dst[T][n_packed_cells] in DEVICE memory.  No host core touches the data (ranks of a
 * multi-GPU job share the host's cores, not its PCIe links).  time_index: DEVICE int32, nullable.
 * Planes must be 16-byte aligned and hold a multiple of 4 gridcells (else CTB_ERR_UNSUPPORTED). */
int ctb_pull_pack(const ctb_plan* plan, const void* x, int dtype, int64_t stride, const int32_t* time_index,
                  int64_t t_begin, int64_t T, void* dst, void* stream);

/* Sub-daily sources: the same pull, reducing steps_per_day (S >= 1) steps to one day while the referenced
 * pieces are packed.  x[t_phys][stride] is TIME_MAJOR, in DEVICE or pinned HOST memory; day d < n_days
 * reduces steps day_index[t_begin + d] * S + h, h = 0..S-1 (day_index: DEVICE int32, nullable = t_begin + d).
 * ops is a non-empty mask of CTB_DAILY_*, each with its DEVICE destination [n_days][n_packed_cells]:
 *   MEAN -> dst_mean, float64: steps widened to float64, added in step order with NaN steps skipped,
 *           divided by the count of non-NaN steps (NaN for a day without one); needs plan elem_bytes 8;
 *   MIN / MAX -> dst_min / dst_max, in the source dtype: NaN steps skipped (NaN for a day without a value),
 *           exact; needs plan elem_bytes = the source's.  MIN and MAX together read the source once.
 * Errors as ctb_pull_pack: a non-compact plan or a bad argument is CTB_ERR_INVALID, planes or
 * destinations that are not 16-byte aligned CTB_ERR_UNSUPPORTED. */
enum { CTB_DAILY_MEAN = 1, CTB_DAILY_MIN = 2, CTB_DAILY_MAX = 4 };
int ctb_pull_pack_daily(const ctb_plan* plan, const void* x, int dtype, int64_t stride, int steps_per_day,
                        const int32_t* day_index, int64_t t_begin, int64_t n_days, int ops, void* dst_mean,
                        void* dst_min, void* dst_max, void* stream);

/* rows of a pitched DEVICE array -> pitched HOST (pinned) array, one asynchronous 2-D copy on `stream`:
 * the host path returns out[:, :, t0:t1] of a finished time chunk while the next chunk is in flight */
int ctb_copy_rows_to_host(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes,
                          size_t rows, void* stream);

/* ---- fused time reduction (annual sums of the daily region values) -------- *
 * The step after the path in CIL pipelines: EDD_P = sum over the days of a period of the
 * aggregated EDD_d (transformations.py:17-21).  group_of_day (HOST int32[T]) gives the output
 * column of every day: it starts at 0 and grows by 0 or 1 per day (contiguous periods, e.g. year
 * index).  ctb_aggregate_grouped writes out[(j*R + r)*out_ld + g] = sum over the days t of column
 * g of the value ctb_aggregate would have written to out[..][t] -- the region x time block never
 * reaches memory, the output is n_days/n_groups times smaller.  Summation order is fixed
 * (deterministic); NaN and infinities propagate like in a plain sum.
 * A time-chunked caller (host inputs that arrive in pieces) passes the window: the T input days
 * are days [t_begin, t_begin + T) of the groups' time axis (t_begin a multiple of 32, time_index
 * relative to the window's inputs), with flush = 0 for all but the last call; the call with
 * flush != 0 (T may be 0) finishes the sums and writes `out`.  All calls share one workspace
 * (split-region rows + per-tile partial sums) and one stream. */
int ctb_time_groups_create(const int32_t* group_of_day, int64_t T, int device, ctb_time_groups** out);
void ctb_time_groups_free(ctb_time_groups* groups);
int32_t ctb_time_groups_count(const ctb_time_groups* groups);
size_t ctb_aggregate_grouped_workspace_bytes(const ctb_plan* plan, const ctb_time_groups* groups, int n_out);
int ctb_aggregate_grouped(const ctb_plan* plan, const void* x0, const void* x1, int dtype, int layout,
                          int64_t stride, const int32_t* time_index, int64_t T, int transform,
                          const double* params, int n_params, int n_out, const ctb_time_groups* groups,
                          int64_t t_begin, int flush,
                          double* out /*[n_out][R][out_ld >= n_groups]*/, int64_t out_ld, void* workspace,
                          size_t workspace_bytes, int variant, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTB_H_ */
