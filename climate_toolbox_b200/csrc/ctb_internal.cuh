// Internal declarations shared by the translation units of libctb.so.
// Public surface: include/ctb.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstddef>
#include <cstring>
#include <cstdio>
#include <string>
#include <type_traits>
#include <vector>

#include "ctb.h"

// ---------------------------------------------------------------- errors ---
void ctb_set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_ctb_launches;

#define CTB_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      ctb_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__,    \
                    __LINE__);                                                           \
      return CTB_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define CTB_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    g_ctb_launches.fetch_add(1, std::memory_order_relaxed);                              \
    CTB_CUDA(cudaGetLastError());                                                        \
  } while (0)

// ------------------------------------------------------------- constants ---
constexpr int CTB_TB = 32;             // days per staging tile
constexpr int CTB_S = CTB_TB + 1;      // planner's tile budget unit (see CTB_TILE_BYTES)
constexpr int CTB_PIECE = 4;           // gridcells per staged piece (16 B of f32)

// Per-bundle metadata blob (one cp.async.bulk into shared memory per work unit):
//   part A: [CtbBlobHeader][n_pieces x int32 piece]
//   part B: [n_seg x CtbSeg][n_ent_pad x CtbEnt]
// Every segment's entries start at a multiple of 4 ("quads"); a quad holds, whenever the
// region's cells allow it, four staged columns with four different residues mod 4, in residue
// order -- the streaming kernel reads a quad with one conflict-free shared-memory load
// (lane = entry-in-quad x 8 days).  Ranges are padded to whole quads with weight-0 entries.
struct CtbBlobHeader {
  int32_t n_pieces, n_seg;
  int32_t off_seg, off_ent;   // byte offsets from the start of part B
  int32_t n_ent_pad, bytes_a, bytes_b, reserved;
};
struct CtbSeg {
  int32_t target;  // >= 0: region row of `out`; < 0: ~scratch_slot (region split over bundles)
  uint16_t e0_4;   // first entry / 4
  uint16_t n;      // entries (without the padding)
  double rden;     // 1 / (sum of the region's weights); 1.0 for partial rows.  den == 0 gives
                   // inf: 0 * inf = NaN and x * inf = +-inf, like 0/0 and x/0
};
struct CtbEnt {
  double w;        // effective weight of the weights row (aggregations.py:73)
  uint32_t off;    // byte offset of the staged gridcell's column in a tile row: column * elem_bytes
  uint32_t gate;   // growing-season gate of the gridcell (ctb_gate_on), CTB_GATE_ALWAYS without a mask
};

// Growing-season gate (utils.py:83-153): first day | last day << 9 | wrap << 18.  A gridcell-day counts
// when (first <= day_of_year <= last) != wrap; an empty interval gives "never" (wrap = 0: planting date
// missing) or "always" (wrap = 1: harvest date missing).
constexpr uint32_t CTB_GATE_ALWAYS = 0u | (511u << 9);
__host__ __device__ __forceinline__ bool ctb_gate_on(uint32_t g, int doy) {
  return ((doy >= (int)(g & 511u)) & (doy <= (int)((g >> 9) & 511u))) != (bool)(g >> 18);
}
static_assert(sizeof(CtbBlobHeader) == 32 && sizeof(CtbSeg) == 16 && sizeof(CtbEnt) == 16, "blob layout");

// A bundle stages at most CTB_TILE_UNITS 16-byte units per day and input.
#ifdef CTB_TILE_UNITS_OVERRIDE
constexpr int CTB_TILE_UNITS = CTB_TILE_UNITS_OVERRIDE;
#else
constexpr int CTB_TILE_UNITS = 128;
#endif
constexpr int CTB_META_A_CAP = 32 + CTB_TILE_UNITS * 4;           // header + piece list
constexpr int CTB_META_B_CAP = 14304;                             // segment table + entries
constexpr int CTB_META_CAP = CTB_META_A_CAP + CTB_META_B_CAP;     // 14,848 B: one whole blob

// ---- streaming kernel (ctb_stream_impl.cuh): row-major tiles [day][column], filled by cp.async ----
// Row pitch: 128 units + 16 bytes, == 16 (mod 128): the 8 days x 4 columns one warp reads per
// shared-memory load fall into 32 different banks.
constexpr int CTB_ROWB = CTB_TILE_UNITS * 16 + 16;                 // 2,064 B
constexpr int CTB_STREAM_TILE_BYTES = CTB_TB * CTB_ROWB;           // 66,048 B per input
#ifndef CTB_STREAM_THREADS_OVERRIDE
#define CTB_STREAM_THREADS_OVERRIDE 768
#endif
constexpr int CTB_STREAM_THREADS = CTB_STREAM_THREADS_OVERRIDE;
constexpr int CTB_STREAM_PRODUCER_WARPS = 4;

// the planner sizes bundles against this budget: 128 pieces x 4 cells x 33 x 4 bytes (the round-1
// tile; kept because it fixes the bundle sizes the kernels are tuned for: n_pieces * stage_bytes <= 512)
constexpr int CTB_TILE_BYTES = CTB_TILE_UNITS * 4 * CTB_S * 4;    // 67,584
constexpr int CTB_N_WORK_COUNTERS = 64;

// -------------------------------------------------------------- the plan ---
struct ctb_plan {
  int device = 0;
  int32_t R = 0;
  int64_t n_rows = 0, nnz = 0, ncell = 0;
  int32_t nlat_phys = 0, nlon_phys = 0;

  // K0 products (device): region-sorted CSR over kept rows
  int32_t* d_row_cell = nullptr;  // [n_rows]  physical flat cell of every weights row
  int32_t* d_row_ptr = nullptr;   // [R+1]
  int32_t* d_col = nullptr;       // [nnz]
  double* d_w = nullptr;          // [nnz]
  uint32_t* d_gate = nullptr;     // [nnz] growing-season gate of every kept row's gridcell
  int has_gate = 0;
  double* d_den = nullptr;        // [R]

  // staging bundles (device)
  int32_t n_bundles = 0, n_segments = 0;
  int64_t* d_b_blob_off = nullptr;   // [n_bundles+1] byte offsets into d_blob (16 B aligned)
  int4* d_b_desc = nullptr;          // [n_bundles] {off_lo, off_hi, bytes_a + bytes_b, n_units}
  int32_t* d_unit_tab = nullptr;     // [n_bundles][CTB_TILE_UNITS] element offset of every staged 16-byte unit in a day plane
  // dynamic unit scheduler of the fused kernel: CTB_N_WORK_COUNTERS device counters used round-robin,
  // one per launch (zeroed on the launch's stream), so that launches of one plan on different
  // streams do not share a counter
  int* d_work_counter = nullptr;
  mutable std::atomic<uint32_t> work_counter_slot{0};
  uint8_t* d_blob = nullptr;         // per-bundle metadata blobs, see CtbBlobHeader
  // regions split over several bundles: out[r] = sum(scratch[slot0..slot1)) / den[r]
  int32_t n_split = 0, n_scratch = 0;
  int32_t* d_split_region = nullptr;  // [n_split]
  int32_t* d_split_slot_ptr = nullptr;  // [n_split+1]

  // compact plans: physical piece of every packed piece, as runs of consecutive pieces
  struct PackRun { int32_t phys_piece, n_pieces, packed_piece; };
  std::vector<PackRun> h_pack_runs;
  int32_t* d_pack_src = nullptr;   // compact plans: [n_packed_cells / 4] physical piece of every packed piece, -1 = padding
  int compact = 0;
  int elem_bytes = 4;   // element size the staged-cell byte offsets were built for
  int stage_bytes = 4;  // staged bytes per gridcell-day the bundles were sized for (n_in * elem_bytes)

  // host mirrors for queries
  std::vector<int32_t> h_row_cell;
  std::vector<double> h_row_w;
  std::vector<double> h_den;
  std::vector<int32_t> h_region_pos;   // position of every region along the bundle sequence (spatial order)
  ctb_plan_info info{};
};

// ---------------------------------------------------------- time groups ---
// Fused time reduction (annual sums): output column of every day, contiguous groups.
struct ctb_time_groups {
  int device = 0;
  int64_t T = 0;
  int32_t n_groups = 0;
  int32_t gk = 1;                    // max groups one 32-day tile touches
  int32_t* d_group = nullptr;        // [T]
  int32_t* d_t_lo = nullptr;         // [n_groups] first day of the group
  int32_t* d_t_hi = nullptr;         // [n_groups] one past its last day
};

// ------------------------------------------------- gridcell transforms -----
struct CtbTr {
  double a[8];  // thresholds / offset
  int ip[4];    // integer powers (POLY)
  // Snyder thresholds rounded to single precision, up and down: for a float x, x < e <=> x < up(e)
  // and x > e <=> x > dn(e), so the case tests of float inputs run on the fp32 pipe
  float up[8], dn[8];
};
static_assert(offsetof(CtbTr, dn) % 8 == 0, "ctb_rcs_b reads doubles from dn[]");

// internal transform kind: CTB_TR_POLY whose orders are 1..n_out (checked on the host by the
// launcher), so that the kernel carries one running product and no order tests (config 3)
constexpr int CTB_TR_POLY_SEQ = 16;

// inputs a transform reads per gridcell-day: the Snyder forms take tasmin and tasmax
__host__ __device__ constexpr int ctb_tr_nin(int kind) { return (kind == CTB_TR_EDD || kind == CTB_TR_GDD) ? 2 : 1; }

__device__ __forceinline__ double ctb_ipow(double d, int p) {
  // integer power by squaring; p is warp-uniform
  double r = 1.0, b = d;
  int n = p < 0 ? -p : p;
  while (n) {
    if (n & 1) r *= b;
    b *= b;
    n >>= 1;
  }
  return p < 0 ? 1.0 / r : r;
}

// Snyder exceedance degree days, transformations.py:69-89.
//   tmin < e < tmax :  ((M-e)(pi/2 - asin s) + W cos(asin s)) / pi   with s = (e-M)/W
//                    = W * g(s),  g(s) = (sqrt(1-s^2) - s*acos(s)) / pi,  g(-a) = g(a) + a
//   tmax <= e       :  0          (also when tmax is NaN)
//   tmin >= e       :  M - e      (NaN when tmin is NaN)
// g(a) = v^(3/2) * H(v), v = 1 - a: after factoring the (1-a)^(3/2) behaviour at the end point
// the rest is analytic on [0, 1] (nearest singularity at v = 2), and ONE degree-12 polynomial
// fitted to 80-bit reference values (ctb_edd_coeffs.h, gen_edd_coeffs.py) covers the whole
// range.  Against asin/cos in numpy the scheme agrees to 3e-14 * max(|EDD|, W); it replaces an
// fp64 asin, a sqrt and two divisions by 13 FMAs and one sqrt.  `rW` = 1/W is shared by all
// thresholds of a gridcell-day.
#include "ctb_edd_coeffs.h"

// The coefficients live in constant memory so that every DFMA takes its coefficient as a
// constant-bank / uniform-register operand; as literals each one costs two UMOVs per evaluation
// (half of the instructions of the Snyder kernels).
static __constant__ double ctb_edd_H[CTB_EDD_H_N] = CTB_EDD_H_COEFFS;

// 1/w and sqrt(v) of the Snyder form: the hardware's fp64 seeds (rcp.approx / rsqrt.approx: ONE
// special-function instruction each, MUFU.RCP64H / MUFU.RSQ64H, 2^-23) refined by two fp64 Newton
// steps (to 1e-16): 5 + 7 instructions instead of the ~20 + ~34 of the IEEE-rounded division and
// square-root sequences with their slow-path calls -- half of the instructions of an evaluation in
// the SASS of the round-2 kernel.  (Seeds from the SINGLE-precision unit were measured slower: each
// f64<->f32 conversion is another XU instruction.)
__device__ __forceinline__ double ctb_rcp_pos(double w) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(w));
  r = fma(r, fma(-w, r, 1.0), r);
  return fma(r, fma(-w, r, 1.0), r);     // w = 0 / inf / NaN: NaN or inf, only used by unselected forms
}
__device__ __forceinline__ double ctb_sqrt_pos(double v) {   // v in (0, 1]
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(v));
  const double h = 0.5 * y;
  double s = v * y;
  s = fma(fma(-s, s, v), h, s);
  return fma(fma(-s, s, v), h, s);
}

__device__ __forceinline__ double ctb_edd_g(double a) {   // a in [0, 1)
  const double v = 1.0 - a;
  const double t = fma(-2.0, a, 1.0);   // = 2 v - 1
  // even/odd split H(t) = E(t^2) + t*O(t^2): two independent Horner chains instead of one (the
  // Snyder kernels stall on this dependency chain: 4-5 warps per scheduler)
  static_assert(CTB_EDD_H_N % 2 == 1 && CTB_EDD_H_N >= 5, "even/odd split below assumes an even degree");
  constexpr int D = CTB_EDD_H_N - 1;
  const double t2 = t * t;
  double pe = ctb_edd_H[D], po = ctb_edd_H[D - 1];
#pragma unroll
  for (int k = D - 2; k >= 0; k -= 2) pe = fma(pe, t2, ctb_edd_H[k]);
#pragma unroll
  for (int k = D - 3; k >= 1; k -= 2) po = fma(po, t2, ctb_edd_H[k]);
  return v * ctb_sqrt_pos(v) * fma(po, t, pe);
}

// Branch-free: a warp's lanes hold different gridcell-days, so the three cases of the closed form
// diverge inside almost every warp (ncu: 14 of 32 lanes active per instruction when they are
// branches, a quarter of the instructions control flow).  The straddling form is evaluated for all
// lanes -- its argument clamped into the polynomial's range -- and the case is picked by selects;
// what an unselected form computes from NaN / W = 0 never reaches the result.
// The fp64 pipe is the unit this kernel keeps busiest (ncu: 61 %), and double comparisons run on it:
// the clamp and the sign test below read the high word instead (positive doubles order like their bit
// patterns), and |s| is clamped just below 1 so that v = 1 - a is never 0 and the square root needs no
// special case (g(1 - 2^-53) = 1e-24: the straddling form is only selected for tmin < e < tmax, |s| < 1).
// |x| and -x through the high word (integer pipe): as fp64 instructions they are DADDs on the pipe
// the Snyder kernels saturate first
__device__ __forceinline__ double ctb_abs_bits(double x) {
  return __hiloint2double(__double2hiint(x) & 0x7fffffff, __double2loint(x));
}
__device__ __forceinline__ double ctb_neg_bits(double x) {
  return __hiloint2double(__double2hiint(x) ^ (int)0x80000000, __double2loint(x));
}
// the straddling form when tmin < e, else M - e; the caller zeroes (or skips) tmin < e && !(tmax > e)
__device__ __forceinline__ double ctb_edd_pick(bool tmin_below, double M, double W, double rW, double e) {
  const double d = e - M, s = d * rW;
  const int hi = __double2hiint(s);
  // 1 <= |s| < inf: clamp; inf / NaN (non-finite temperatures) pass through and give NaN like the
  // reference's arcsin
  const bool big = (unsigned)((hi & 0x7fffffff) - 0x3ff00000) < 0x40000000u;
  const double a = big ? 0.99999999999999989 : ctb_abs_bits(s);
  const double g = ctb_edd_g(a);
  const double straddle = W * (hi < 0 ? g + a : g);                        // g(-a) = g(a) + a
  return tmin_below ? straddle : ctb_neg_bits(d);                          // tmin >= e or NaN: M - e
}
__device__ __forceinline__ double ctb_edd_cases(bool tmin_below, bool tmax_above, double M, double W, double rW,
                                                double e) {
  const double r = ctb_edd_pick(tmin_below, M, W, rW, e);
  return (tmin_below && !tmax_above) ? 0.0 : r;                            // tmax <= e or NaN: no degree days
}
__device__ __forceinline__ double ctb_edd(double tmin, double tmax, double M, double W, double rW, double e) {
  return ctb_edd_cases(tmin < e, tmax > e, M, W, rW, e);
}

// Temperature bins: in[j] = e_j <= x - offset < e_{j+1} for the contiguous edges a[1..NOUT+1] (offset
// a[0]); one fp64 comparison per edge.  x is the stored value widened exactly to double, so the subtraction
// rounds like the oracle's.  NaN lies in no bin (every comparison is false).
template <int NOUT>
__device__ __forceinline__ void ctb_bins_in(const CtbTr& P, double x, bool (&in)[NOUT]) {
  const double d = x - P.a[0];
  int k = 0;   // edges at or below d; the edges increase, so d lies in bin j exactly when k == j + 1
#pragma unroll
  for (int j = 0; j <= NOUT; ++j) k += d >= P.a[1 + j];
#pragma unroll
  for (int j = 0; j < NOUT; ++j) in[j] = k == j + 1;
}

// The same decisions for a float x on the stored type: up[j] is the least float whose widened value minus
// the offset is >= e_j (ctb_pack_transform), and that predicate grows with x, so x >= up[j] decides it for
// every float -- NaN, infinities and negative values included -- with one fp32 comparison per edge.
template <int NOUT>
__device__ __forceinline__ void ctb_bins_in_f32(const CtbTr& P, float x, bool (&in)[NOUT]) {
  bool ge[NOUT + 1];
#pragma unroll
  for (int j = 0; j <= NOUT; ++j) ge[j] = x >= P.up[j];
#pragma unroll
  for (int j = 0; j < NOUT; ++j) in[j] = ge[j] && !ge[j + 1];
}

// Restricted cubic spline terms f_j = B_{first+j}(d), d = x - offset (CTB_TR_RCSPLINE; packed by
// ctb_pack_transform: a[1 + j] = output j's knot k_i, a[5] = k_{n-1}, a[6] = k_n, b_i of output j in
// ctb_rcs_b(P, j), ip[0] = output 0 is B_0 = d).  With c(k) = max(d - k, 0)^3 and b_i = (k_{n-1} - k_i) / (k_n - k_{n-1}),
//   B_i = c(k_i) - c(k_{n-1}) - b_i (c(k_{n-1}) - c(k_n)),
// the definition with a_i = 1 + b_i: the cubes of k_{n-1} and k_n are computed once per value for every output,
// and both differences are of non-negative terms, so the rounding stays within a few ulps of the scale
// c(k_i) + a_i c(k_{n-1}) + b_i c(k_n) whatever the knots' magnitude.  Below k_{n-1} the result is c(k_i)
// exactly, below k_i exactly 0.  pos(m, t) decides t = d - a[m] > 0 (NaN has to give true, t * t * t = NaN,
// wherever a NaN can reach a kept result).
// b_i of output j: kept in the kernel parameters, where every DFMA reads it as a constant operand (computed in
// the loop or held in registers, the coefficients made the 2- to 4-output streaming kernels spill).  CtbTr::a is
// full, so the four doubles sit in the bytes of dn[], which the spline does not use otherwise.
__host__ __device__ __forceinline__ double ctb_rcs_b(const CtbTr& P, int j) {
  double b;
  memcpy(&b, &P.dn[2 * j], sizeof b);
  return b;
}

template <int NOUT, typename Pos>
__device__ __forceinline__ void ctb_rcs(const CtbTr& P, double d, Pos pos, double (&f)[NOUT]) {
  auto c = [&](int m) {
    const double t = d - P.a[m];
    return pos(m, t) ? t * t * t : 0.0;
  };
  const double cm = c(5), dc = cm - c(6);
#pragma unroll
  for (int j = 0; j < NOUT; ++j) {
    f[j] = fma(-ctb_rcs_b(P, j), dc, c(1 + j) - cm);
  }
  if (P.ip[0]) f[0] = d;
}

template <int KIND, int NOUT>
__device__ __forceinline__ void ctb_apply(const CtbTr& P, double x0, double x1, double (&f)[NOUT]) {
  if constexpr (KIND == CTB_TR_IDENTITY) {
    f[0] = x0;
  } else if constexpr (KIND == CTB_TR_RCSPLINE) {
    ctb_rcs<NOUT>(P, x0 - P.a[0], [](int, double t) { return !(t <= 0.0); }, f);
  } else if constexpr (KIND == CTB_TR_BINS) {
    bool in[NOUT];
    ctb_bins_in<NOUT>(P, x0, in);
#pragma unroll
    for (int j = 0; j < NOUT; ++j) f[j] = x0 != x0 ? x0 : (in[j] ? 1.0 : 0.0);   // NaN stays NaN (.values)
  } else if constexpr (KIND == CTB_TR_POLY_SEQ) {
    const double d = x0 - P.a[0];
    double p = d;
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
      f[j] = p;
      p *= d;
    }
  } else if constexpr (KIND == CTB_TR_POLY) {
    const double d = x0 - P.a[0];
    bool chain = true;
#pragma unroll
    for (int j = 0; j < NOUT; ++j) chain = chain && (P.ip[j] == j + 1);
    if (chain) {  // powers 1..NOUT from one read (config 3)
      double p = d;
#pragma unroll
      for (int j = 0; j < NOUT; ++j) {
        f[j] = p;
        p *= d;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NOUT; ++j) f[j] = ctb_ipow(d, P.ip[j]);
    }
  } else if constexpr (KIND == CTB_TR_EDD) {
    const double M = (x1 + x0) * 0.5, W = (x1 - x0) * 0.5, rW = ctb_rcp_pos(W);
#pragma unroll
    for (int j = 0; j < NOUT; ++j) f[j] = ctb_edd(x0, x1, M, W, rW, P.a[j]);
  } else {  // GDD
    const double M = (x1 + x0) * 0.5, W = (x1 - x0) * 0.5, rW = ctb_rcp_pos(W);
#pragma unroll
    for (int j = 0; j < NOUT; ++j)
      f[j] = ctb_edd(x0, x1, M, W, rW, P.a[2 * j]) - ctb_edd(x0, x1, M, W, rW, P.a[2 * j + 1]);
  }
}

// Two-input transforms on the stored type: float inputs take the case tests in single precision
// against the rounded thresholds of CtbTr (exactly the same decisions; two DSETP fewer per evaluation).
template <int KIND, int NOUT, typename TIN>
__device__ __forceinline__ void ctb_apply2(const CtbTr& P, TIN lo, TIN hi, double (&f)[NOUT]) {
  static_assert(KIND == CTB_TR_EDD || KIND == CTB_TR_GDD, "two-input transforms");
  if constexpr (sizeof(TIN) == 8) {
    ctb_apply<KIND, NOUT>(P, lo, hi, f);
  } else {
    const double x0 = (double)lo, x1 = (double)hi;
    const double M = (x1 + x0) * 0.5, W = (x1 - x0) * 0.5, rW = ctb_rcp_pos(W);
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
      if constexpr (KIND == CTB_TR_EDD) {
        f[j] = ctb_edd_cases(lo < P.up[j], hi > P.dn[j], M, W, rW, P.a[j]);
      } else {
        f[j] = ctb_edd_cases(lo < P.up[2 * j], hi > P.dn[2 * j], M, W, rW, P.a[2 * j]) -
               ctb_edd_cases(lo < P.up[2 * j + 1], hi > P.dn[2 * j + 1], M, W, rW, P.a[2 * j + 1]);
      }
    }
  }
}

// ------------------------------------------------ kernel arguments ---------
struct AggArgs {
  const void* x0;
  const void* x1;
  int64_t stride;
  const int32_t* tix;
  int T;
  int64_t out_ld;
  int64_t ncell;
  int R;
  double* out;
  double* scratch;
  int n_scratch;
  const double* den;
  const unsigned char* blob;
  int n_bundles;
  int n_items;
  const int4* b_desc;
  const int32_t* unit_tab;
  int tile_stride;   // bytes between tile stages
  int n_stages;      // streaming kernel: tile stages in shared memory
  int n_tb;          // time blocks: ceil(T / 32)
  int chunk_tb;      // time blocks per work unit (a CTA keeps one bundle for a whole unit)
  int* work_counter; // {next unit, CTAs done}: dynamic unit scheduling, re-armed by the kernel
  int knobs;         // experiments only (compiled in with -DCTB_EXPERIMENT): 1 = skip the copies, 4 = skip the reduction
  // fused time reduction (ctb_aggregate_grouped): the launch covers days [t_off, t_off + T) of the
  // groups' time axis; day t adds into output column tgroup[t_off + t]
  const int32_t* tgroup;   // [T_total] non-decreasing, steps of 0 or 1; NULL = no time reduction
  double* gpart;           // [n_out][R][g_ntb][gk] per-tile partial sums
  int gk;                  // max output columns one 32-day tile touches
  int g_ntb;               // 32-day tiles of the whole time axis
  int t_off;               // multiple of 32
  int n_groups;
  const int32_t *g_t_lo, *g_t_hi;   // [n_groups] day range of every output column
  int64_t scratch_ld;      // days per partial row of a split region (T, or T_total with time groups)
  // growing-season gate: day of year of day t_off + t; NULL = no gate.  gate: per CSR entry (direct kernel)
  const int32_t* doy;
  const uint32_t* gate;
  // fused gather: n_peers > 0 => every result is stored to peers[0..n_peers) (own + NVLink peer buffers),
  // region r in row peer_row[r] (NULL: r)
  int n_peers;
  double* peers[CTB_MAX_PEERS];
  const int32_t* peer_row;
  const int32_t *row_ptr, *col;
  const double* w;
  const int32_t *split_region, *split_slot_ptr;
  int n_split;
  CtbTr tr;
};

// One region x 32-day tile result (lane = day `t`, `valid` = t < T): normalise and store, or --
// fused time reduction -- add the tile's days into per-tile partial sums per output column
// (fixed shuffle tree: deterministic), or store the partial row of a split region.
template <int NOUT>
__device__ __forceinline__ void ctb_emit(const AggArgs& a, int target, double rden, const double (&v)[NOUT],
                                         int lane, int t, bool valid, int tb, int tg, int tg0) {
  if (target >= 0 && a.tgroup) {
    // columns this tile touches: most 32-day tiles lie inside one period
    const int nk = __reduce_max_sync(0xffffffffu, tg) - tg0 + 1;
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
      const double val = v[j] * rden;
      for (int k = 0; k < nk; ++k) {
        double x = (tg == tg0 + k) ? val : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) a.gpart[(((size_t)j * a.R + target) * a.g_ntb + (a.t_off / CTB_TB + tb)) * a.gk + k] = x;
      }
    }
  } else if (valid) {
    if (target >= 0) {
#pragma unroll
      for (int j = 0; j < NOUT; ++j) {   // written once: leave L2 to the input
        const double val = v[j] * rden;
        if (a.n_peers == 0) {
          __stcs(&a.out[((size_t)j * a.R + target) * a.out_ld + t], val);
        } else {
          const int row = a.peer_row ? __ldg(a.peer_row + target) : target;
          const size_t idx = ((size_t)j * a.R + row) * a.out_ld + t;
          for (int p = 0; p < a.n_peers; ++p) __stcs(&a.peers[p][idx], val);
        }
      }
    } else {
      const int slot_o = ~target;
#pragma unroll
      for (int j = 0; j < NOUT; ++j) a.scratch[((size_t)j * a.n_scratch + slot_o) * a.scratch_ld + a.t_off + t] = v[j];
    }
  }
}

// ctb_stream_impl.cuh: the streaming kernel (IDENTITY / POLY, 16-byte aligned TIME_MAJOR planes)
int ctb_launch_stream(const ctb_plan* P, const AggArgs& a, int dtype, int kind, int n_out, cudaStream_t st);   // a.doy != NULL: gated

// RAII: make the plan's device current for the duration of an entry point
struct CtbDeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t err = cudaSuccess;
  explicit CtbDeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) {
      err = cudaSetDevice(device);
      switched = (err == cudaSuccess);
    }
  }
  ~CtbDeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

// host: validate + pack transform params. returns CTB_OK or error.
int ctb_pack_transform(int transform, const double* params, int n_params, int n_out, CtbTr* out);

// The (transform, outputs) pairs the kernels are compiled for: f(std::integral_constant<int, KIND>{},
// std::integral_constant<int, NOUT>{}) launches the pair's instantiation.  Any other pair is an error.
template <int KIND, typename F>
int ctb_dispatch_nout(int n_out, F&& f) {
  using K = std::integral_constant<int, KIND>;
  switch (n_out) {
    case 1: return f(K{}, std::integral_constant<int, 1>{});
    case 2: return f(K{}, std::integral_constant<int, 2>{});
    case 3: return f(K{}, std::integral_constant<int, 3>{});
    case 4: return f(K{}, std::integral_constant<int, 4>{});
  }
  ctb_set_error("transform=%d n_out=%d unsupported", KIND, n_out);
  return CTB_ERR_INVALID;
}

// Adding a transform kind: one case here, plus its branches in ctb_apply and ctb_pack_transform.
template <typename F>
int ctb_dispatch_transform(int kind, int n_out, F&& f) {
  switch (kind) {
    case CTB_TR_IDENTITY:
      if (n_out != 1) break;
      return f(std::integral_constant<int, CTB_TR_IDENTITY>{}, std::integral_constant<int, 1>{});
    case CTB_TR_POLY: return ctb_dispatch_nout<CTB_TR_POLY>(n_out, f);
    case CTB_TR_EDD: return ctb_dispatch_nout<CTB_TR_EDD>(n_out, f);
    case CTB_TR_GDD: return ctb_dispatch_nout<CTB_TR_GDD>(n_out, f);
    case CTB_TR_BINS: return ctb_dispatch_nout<CTB_TR_BINS>(n_out, f);
    case CTB_TR_RCSPLINE: return ctb_dispatch_nout<CTB_TR_RCSPLINE>(n_out, f);
  }
  ctb_set_error("transform=%d n_out=%d unsupported", kind, n_out);
  return CTB_ERR_INVALID;
}
