// The streaming kernel: stage + gather + segmented weighted sum for TIME_MAJOR inputs
// [T][lat][lon] (the BCSD layout), all transforms.
//
// Replaces climate_toolbox/aggregations/aggregations.py:27 (gather) and :75-82
// (sum(w*x)/sum(w) per region), with transformations.py:189 fused in.
//
// One persistent CTA of 24 warps per SM (fewer, with more registers, for the multi-output and Snyder forms).  A work unit = one bundle (spatially adjacent regions
// whose gridcell footprint fits a shared-memory tile) x a chunk of consecutive 32-day blocks;
// CTA b takes units b, b + grid, ... in chunk-major order, so that CTAs running together read
// neighbouring bundles of the same days (the lines they share meet in L2).
//
//   4 producer warps   copy the footprint of the next tiles -- 32 day rows x up to 128 16-byte
//                      units -- straight from global to shared memory with cp.async (LDGSTS:
//                      no registers, no shared-memory store instructions), row-major
//                      [day][column], into a ring of 3 tile stages; an mbarrier per stage is
//                      armed by cp.async.mbarrier.arrive, so the copies of up to two tiles are
//                      in flight while a third is being reduced.  The bundle's metadata blob
//                      arrives as one cp.async.bulk (TMA 1-D) per unit, double-buffered.
//   20 consumer warps  take the regions of a landed tile from a shared counter (longest
//                      first).  A warp reduces a region four entries at a time: lane = (entry
//                      in quad) x 8 + (day mod 8); one 16-byte shared load brings the lane its
//                      entry's {weight, column offset}, four conflict-free 4-byte loads bring
//                      the entry's value on days d, d+8, d+16, d+24 (the row pitch is == 16
//                      mod 128 and the planner orders a region's columns so that a quad holds
//                      four residues mod 4); fp64 FMA into four accumulators; two
//                      shuffle-and-select steps fold the four entry lanes so that lane l ends
//                      with day l; one coalesced 256-byte streaming store per region and tile.
//   NaN semantics      the reference skips NaN products (aggregations.py:78).  The fast loop
//                      does not look at the values; a region-tile whose result is not finite
//                      on some day (a NaN or an infinity was staged, or a zero-weight padding
//                      entry met one) is reduced again by the checked loop.  Finite data never
//                      pays for the check, and a NaN costs its own region only.
// No atomics on data, fixed summation order: results are deterministic.
#include <algorithm>
#include <cstring>

#include "ctb_internal.cuh"

namespace {

#ifndef CTB_STICKY_ALL
#define CTB_STICKY_ALL 1   // 0: only the single-output kernels skip the widening after a failed range check
#endif

// CTB_NP / CTB_WAIT_NS / CTB_PACE_NS / CTB_STAGES / CTB_TILE_UNITS_OVERRIDE: compile-time knobs of the
// bench_micro/ experiments (profiles/micro/r2_stream_sweeps.md); the defaults are the measured best
#ifdef CTB_NP
constexpr int NP = CTB_NP;
#else
constexpr int NP = CTB_STREAM_PRODUCER_WARPS;
#endif
#ifndef CTB_WAIT_NS
#define CTB_WAIT_NS 0
#endif
#ifndef CTB_PACE_NS
#define CTB_PACE_NS 40   // pause between a producer warp's day groups: bursts of copies crowd out the reduction's loads
#endif
#ifndef CTB_STAGES
#define CTB_STAGES 3
#endif
constexpr int NG = CTB_TILE_UNITS / 8;        // groups of 8 units (128 bytes of a tile row), all inputs together
constexpr int UPW = (NG + NP - 1) / NP;       // ... per producer warp

// Tile geometry.  A stage holds NIN input tiles of 32 day rows; one input's row has room for
// 128 / NIN 16-byte units (the planner sizes the bundles of a two-input plan to half the cells) plus
// 16 bytes, so that the row pitch is == 16 (mod 128) either way.
template <int NIN>
struct Geo {
  static constexpr int UNITS = CTB_TILE_UNITS / NIN;
  static constexpr int ROWB = UNITS * 16 + 16;        // 2,064 / 1,040 bytes
  static constexpr int IN_BYTES = CTB_TB * ROWB;      // one input's tile
  static constexpr int TILE_BYTES = NIN * IN_BYTES;   // 66,048 / 66,560 bytes per stage
  static constexpr int GROUPS_IN = UNITS / 8;         // groups of 8 units per input
};
enum { F_SLOT = 1, F_FIRST = 2, F_LAST = 4, F_EXIT = 8 };

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x989680;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// the same on 32-bit shared-window addresses (no generic -> shared conversion in the hot loops)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x989680;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// consumers: a tile that has not landed yet is polled with a back-off instead of try_wait -- the
// hardware wakes a try_wait sleeper at EVERY arrival on the barrier (129 per tile), not at the
// completion of the phase
__device__ __forceinline__ void mbar_wait_backoff_a(uint32_t bar, uint32_t parity) {
#if CTB_WAIT_NS > 0
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "nanosleep.u32 %2;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity), "n"(CTB_WAIT_NS)
      : "memory");
#else
  mbar_wait_a(bar, parity);
#endif
}
__device__ __forceinline__ int atom_add_a(uint32_t addr, int v) {
  int r;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(r) : "r"(addr), "r"(v) : "memory");
  return r;
}
// bulk async copy global -> shared (TMA 1-D; SASS: UBLKCP), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// 16-byte asynchronous copy global -> shared, L2 only (SASS: LDGSTS.E.BYPASS.128)
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
#ifdef CTB_CP_L2
#define CTB_STR2(x) #x
#define CTB_STR(x) CTB_STR2(x)
  asm volatile("cp.async.cg.shared.global.L2::" CTB_STR(CTB_CP_L2) "B [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
#else
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
#endif
}
// the executing thread's earlier cp.async copies arrive on the mbarrier when they have landed
__device__ __forceinline__ void cp_async_arrive_a(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
template <typename T>
__device__ __forceinline__ T lds_val(uint32_t addr) {
  T v;
  if constexpr (sizeof(T) == 4) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  else asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// acc[j] += w * f_j(x) for one staged value; CHECK: products that are NaN are skipped and so
// are the zero-weight padding entries (aggregations.py:78: skipna sum of x * w)
template <typename TIN, int KIND, int NOUT, bool CHECK>
__device__ __forceinline__ void add_value(const CtbTr& tr, double w, TIN x, bool on, double (&acc)[NOUT]) {
  if constexpr (KIND == CTB_TR_IDENTITY) {
    if constexpr (CHECK) {
      const double p = w * (double)x;
      if (on && w != 0.0 && p == p) acc[0] += p;
    } else {
      if (on) acc[0] = fma(w, (double)x, acc[0]);
    }
  } else if constexpr (KIND == CTB_TR_BINS) {
    // an indicator adds the weight or nothing: no product, and NaN lies in no bin (no check needed)
    // (float inputs never come here: reduce_region_widen decides their bins for every value)
    bool in[NOUT];
    ctb_bins_in<NOUT>(tr, (double)x, in);
#pragma unroll
    for (int j = 0; j < NOUT; ++j)
      if (on && in[j]) acc[j] += w;
  } else {
    double f[NOUT];
    ctb_apply<KIND, NOUT>(tr, (double)x, 0.0, f);
#pragma unroll
    for (int j = 0; j < NOUT; ++j) {
      if constexpr (CHECK) {
        const double p = w * f[j];
        if (on && w != 0.0 && p == p) acc[j] += p;
      } else {
        if (on) acc[j] = fma(w, f[j], acc[j]);
      }
    }
  }
}

// growing-season gate of the lane's entry on its four days (GATE = false: always on, folded away)
template <bool GATE>
__device__ __forceinline__ void gate4(uint32_t g, const int (&doy)[4], bool (&on)[4]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) on[k] = GATE ? ctb_gate_on(g, doy[k]) : true;
}

// fold the four entry lanes (lane bits 3, 4) of the four day-group accumulators:
// lane l = e * 8 + d8 ends with the sum over e of group g = e, i.e. with day l
__device__ __forceinline__ double fold_quads(double a0, double a1, double a2, double a3, int lane) {
  const bool hi = (lane & 16) != 0, lo = (lane & 8) != 0;
  const double s0 = hi ? a0 : a2, s1 = hi ? a1 : a3;
  double k0 = hi ? a2 : a0, k1 = hi ? a3 : a1;
  k0 += __shfl_xor_sync(0xffffffffu, s0, 16);
  k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
  const double s = lo ? k0 : k1;
  const double k = lo ? k1 : k0;
  return k + __shfl_xor_sync(0xffffffffu, s, 8);
}

// One region (segment) of one tile.  tile_a: shared address of the lane's row d8; ent_a: shared
// address of the lane's entry of the first quad.  Returns v[j] = sum over the region's entries
// of w * f_j(x[day = lane]).
template <typename TIN, int KIND, int NOUT, bool CHECK, bool GATE>
__device__ __forceinline__ void reduce_region(const CtbTr& tr, uint32_t tile_a, uint32_t ent_a, int nq,
                                              int lane, const int (&doy)[4], double (&v)[NOUT]) {
  constexpr int CTB_ROWB = Geo<1>::ROWB;
  double acc[4][NOUT];
#pragma unroll
  for (int g = 0; g < 4; ++g)
#pragma unroll
    for (int j = 0; j < NOUT; ++j) acc[g][j] = 0.0;
#pragma unroll 2
  for (int q = 0; q < nq; ++q, ent_a += 4 * (uint32_t)sizeof(CtbEnt)) {
    const uint4 m = lds_u4(ent_a);
    const double w = __hiloint2double((int)m.y, (int)m.x);
    const uint32_t xa = tile_a + m.z;
    const TIN x0 = lds_val<TIN>(xa);
    const TIN x1 = lds_val<TIN>(xa + 8 * CTB_ROWB);
    const TIN x2 = lds_val<TIN>(xa + 16 * CTB_ROWB);
    const TIN x3 = lds_val<TIN>(xa + 24 * CTB_ROWB);
    bool on[4];
    gate4<GATE>(m.w, doy, on);
    add_value<TIN, KIND, NOUT, CHECK>(tr, w, x0, on[0], acc[0]);
    add_value<TIN, KIND, NOUT, CHECK>(tr, w, x1, on[1], acc[1]);
    add_value<TIN, KIND, NOUT, CHECK>(tr, w, x2, on[2], acc[2]);
    add_value<TIN, KIND, NOUT, CHECK>(tr, w, x3, on[3], acc[3]);
  }
#pragma unroll
  for (int j = 0; j < NOUT; ++j) v[j] = fold_quads(acc[0][j], acc[1][j], acc[2][j], acc[3][j], lane);
}

// Fast loop for float inputs whose values are all positive and normal (temperatures in kelvin):
// the float -> double widening is ONE integer multiply-add on the FMA pipe,
//     bits64 = bits32 * 2^29 + (1023 - 127) * 2^52,
// instead of an F2F.F64.F32 on the quarter-rate XU pipe, where it paces the whole reduction
// (ncu, profiles/r2_*).  The identity holds exactly for 2^-126 <= x < 2^128; a running 3-input
// min / max of the raw bit patterns (one ALU instruction per value) tells whether the region-tile
// saw anything else -- zero, a denormal, a negative number, an infinity or a NaN -- and then the
// caller reduces it again with the exact loops.  Returns false in that case.
#ifndef CTB_POLY34_UNROLL
#define CTB_POLY34_UNROLL 2
#endif
#ifndef CTB_QUAD_UNROLL
#define CTB_QUAD_UNROLL 2
#endif
template <int KIND, int NOUT, bool GATE>
__device__ __forceinline__ bool reduce_region_widen(const CtbTr& tr, uint32_t tile_a, uint32_t ent_a, int nq,
                                                    int lane, const int (&doy)[4], double (&v)[NOUT]) {
  constexpr int CTB_ROWB = Geo<1>::ROWB;
  double acc[4][NOUT];
#pragma unroll
  for (int g = 0; g < 4; ++g)
#pragma unroll
    for (int j = 0; j < NOUT; ++j) acc[g][j] = 0.0;
  uint32_t bmin = 0xffffffffu, bmax = 0u;
  auto widen = [](uint32_t b) {
    return __longlong_as_double((long long)((unsigned long long)b * 0x20000000ull + 0x3800000000000000ull));
  };
  constexpr int UNR = NOUT > 2 ? CTB_POLY34_UNROLL : CTB_QUAD_UNROLL;
#pragma unroll(UNR)
  for (int q = 0; q < nq; ++q, ent_a += 4 * (uint32_t)sizeof(CtbEnt)) {
    const uint4 m = lds_u4(ent_a);
    const double w = __hiloint2double((int)m.y, (int)m.x);
    const uint32_t xa = tile_a + m.z;
    const uint32_t b0 = lds_u32(xa);
    const uint32_t b1 = lds_u32(xa + 8 * CTB_ROWB);
    const uint32_t b2 = lds_u32(xa + 16 * CTB_ROWB);
    const uint32_t b3 = lds_u32(xa + 24 * CTB_ROWB);
    bmin = __vimin3_u32(bmin, b0, b1);
    bmax = __vimax3_u32(bmax, b0, b1);
    bmin = __vimin3_u32(bmin, b2, b3);
    bmax = __vimax3_u32(bmax, b2, b3);
    const uint32_t bb[4] = {b0, b1, b2, b3};
    bool on[4];
    gate4<GATE>(m.w, doy, on);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const double x = widen(bb[g]);
      if constexpr (KIND == CTB_TR_IDENTITY) {
        if (on[g]) acc[g][0] = fma(w, x, acc[g][0]);
      } else if constexpr (KIND == CTB_TR_BINS) {
        // no widening: the float thresholds decide every float exactly (ctb_bins_in_f32)
        bool in[NOUT];
        ctb_bins_in_f32<NOUT>(tr, __uint_as_float(bb[g]), in);
#pragma unroll
        for (int j = 0; j < NOUT; ++j)
          if (on[g] && in[j]) acc[g][j] += w;
      } else if constexpr (KIND == CTB_TR_RCSPLINE) {
        // d > k decided on the stored type against the float thresholds up[] (ctb_pack_transform): fp32
        // compares instead of fp64 ones, the same decisions for every float but NaN -- and a NaN fails the
        // range check, so this result is then not kept
        const float xf = __uint_as_float(bb[g]);
        double f[NOUT];
        ctb_rcs<NOUT>(tr, x - tr.a[0], [&](int m, double) { return xf >= tr.up[m]; }, f);
#pragma unroll
        for (int j = 0; j < NOUT; ++j)
          if (on[g]) acc[g][j] = fma(w, f[j], acc[g][j]);
      } else {
        double f[NOUT];
        ctb_apply<KIND, NOUT>(tr, x, 0.0, f);
#pragma unroll
        for (int j = 0; j < NOUT; ++j)
          if (on[g]) acc[g][j] = fma(w, f[j], acc[g][j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NOUT; ++j) v[j] = fold_quads(acc[0][j], acc[1][j], acc[2][j], acc[3][j], lane);
  if constexpr (KIND == CTB_TR_BINS) return true;   // compared on the stored type: no range to check
  const bool ok = bmin >= 0x00800000u && bmax < 0x7f800000u;
  return __all_sync(0xffffffffu, ok);
}

// Two-input transforms (Snyder EDD / GDD from tasmin, tasmax): the same quad loop, the lane's entry
// evaluated on its four days.  fp64 ALU bound; NaN results are skipped by a select (the reference's
// skipna sum), and the zero-weight padding of the last quad never meets a value (0 * inf).
#ifndef CTB_EDD_UNROLL
#define CTB_EDD_UNROLL 1
#endif
template <typename TIN, int KIND, int NOUT, bool GATE>
__device__ __forceinline__ void reduce_region2(const CtbTr& tr, uint32_t tile_a, uint32_t ent_a, int nq,
                                               int lane, const int (&doy)[4], double (&v)[NOUT]) {
  constexpr int ROWB = Geo<2>::ROWB, IN_BYTES = Geo<2>::IN_BYTES;
  double acc[4][NOUT];
#pragma unroll
  for (int g = 0; g < 4; ++g)
#pragma unroll
    for (int j = 0; j < NOUT; ++j) acc[g][j] = 0.0;
  constexpr int UNR = CTB_EDD_UNROLL;
#pragma unroll(UNR)
  for (int q = 0; q < nq; ++q, ent_a += 4 * (uint32_t)sizeof(CtbEnt)) {
    const uint4 m = lds_u4(ent_a);
    const double w = __hiloint2double((int)m.y, (int)m.x);
    const bool wnz = w != 0.0;
    const uint32_t xa = tile_a + m.z;
    TIN lo[4], hi[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      lo[g] = lds_val<TIN>(xa + g * 8 * ROWB);
      hi[g] = lds_val<TIN>(xa + IN_BYTES + g * 8 * ROWB);
    }
    bool on[4];
    gate4<GATE>(m.w, doy, on);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if constexpr (KIND == CTB_TR_EDD && sizeof(TIN) == 4) {
        // the "no degree days" case (tmin < e, tmax <= e) adds nothing: it joins the predicate of the
        // FMA instead of costing a select of its own
        const double x0 = (double)lo[g], x1 = (double)hi[g];
        const double M = (x1 + x0) * 0.5, W = (x1 - x0) * 0.5, rW = ctb_rcp_pos(W);
#pragma unroll
        for (int j = 0; j < NOUT; ++j) {
          const bool tb = lo[g] < tr.up[j], ta = hi[g] > tr.dn[j];
          const double r = ctb_edd_pick(tb, M, W, rW, tr.a[j]);
          if (wnz && on[g] && (ta || !tb) && r == r) acc[g][j] = fma(w, r, acc[g][j]);
        }
      } else {
        double f[NOUT];
        ctb_apply2<KIND, NOUT, TIN>(tr, lo[g], hi[g], f);
#pragma unroll
        for (int j = 0; j < NOUT; ++j)
          if (wnz && on[g] && f[j] == f[j]) acc[g][j] = fma(w, f[j], acc[g][j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NOUT; ++j) v[j] = fold_quads(acc[0][j], acc[1][j], acc[2][j], acc[3][j], lane);
}

// TIX: the launch has a time index (its own instantiation: the two producer loops compile differently,
// and carrying both costs the plain one 2 %)
template <typename TIN, int KIND, int NOUT, int THREADS, int S, bool GATE, bool TIX>
__global__ void __launch_bounds__(THREADS, 1) agg_stream_kernel(const AggArgs a) {
  constexpr int NIN = ctb_tr_nin(KIND);
  using G = Geo<NIN>;
  constexpr int CTB_ROWB = G::ROWB, CTB_STREAM_TILE_BYTES = G::TILE_BYTES;
  constexpr int NWARP = THREADS / 32;
  constexpr int NCW = NWARP - NP;   // consumer warps 0 .. NCW-1; the producers are the LAST warps:
                                    // the issue arbiter prefers high warp ids, and a copy that is
                                    // issued late costs more than a reduction step that is
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_full[S], s_empty[S], s_mfull[2], s_mempty[2];
  __shared__ int4 s_desc[S];
  __shared__ int s_next[S];
  __shared__ int s_units[2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned char* const s_meta = smem_raw + (size_t)S * CTB_STREAM_TILE_BYTES;
  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&s_full[s], NP * 32 + 1);
      mbar_init(&s_empty[s], NCW);
    }
    for (int m = 0; m < 2; ++m) {
      mbar_init(&s_mfull[m], 1);
      mbar_init(&s_mempty[m], NCW);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
#ifdef CTB_EXPERIMENT
  if (a.knobs & 1)   // no copies: the tiles hold a constant
    for (int i = tid; i < S * CTB_STREAM_TILE_BYTES / 4; i += THREADS) reinterpret_cast<float*>(smem_raw)[i] = 288.0f;
#endif
  __syncthreads();
  const uint32_t full_a = smem_u32(s_full), empty_a = smem_u32(s_empty);
  const uint32_t desc_a = smem_u32(s_desc), next_a = smem_u32(s_next);
  const uint32_t tiles_a = smem_u32(smem_raw);

  if (warp >= NCW) {
    // ------------------------------------------------------------------ producers ---
    // lane = (l4 = day within a group of 4) x (l8 = unit within a group of 8): a quarter warp
    // copies 128 contiguous bytes of one tile row, from mostly contiguous global memory
    const int pw = warp - NCW;
    const bool leader = (pw == 0 && lane == 0);
    const int l8 = lane & 7, l4 = lane >> 3;
    const TIN* const X0 = reinterpret_cast<const TIN*>(a.x0);
    const TIN* const X1 = NIN == 2 ? reinterpret_cast<const TIN*>(a.x1) : X0;
    const int64_t row_step = 4 * a.stride;
    const int64_t stride_b = a.stride * (int64_t)sizeof(TIN);
    // this lane's unit groups: group G = pw + NP * gi of the stage's 16 (input G / GROUPS_IN, units
    // (G % GROUPS_IN) * 8 + l8 of that input); dst_of[gi]: byte offset inside the stage's row 0
    int unit_of[UPW];
    uint32_t dst_of[UPW];
    bool second[UPW];
#pragma unroll
    for (int gi = 0; gi < UPW; ++gi) {
      const int Gi = pw + NP * gi;
      second[gi] = NIN == 2 && Gi >= G::GROUPS_IN;
      unit_of[gi] = (Gi % G::GROUPS_IN) * 8 + l8;
      dst_of[gi] = (uint32_t)((second[gi] ? G::IN_BYTES : 0) + unit_of[gi] * 16);
    }
    int offN[UPW];
    int4 dN = make_int4(0, 0, 0, 0);
    auto prefetch_unit = [&](int unit) {   // descriptor + this lane's unit offsets, one unit ahead
      if (unit < a.n_items) {
        const int b = unit % a.n_bundles;
        dN = __ldg(a.b_desc + b);
#pragma unroll
        for (int gi = 0; gi < UPW; ++gi)
          if (pw + NP * gi < NG)
            offN[gi] = __ldg(a.unit_tab + (size_t)b * CTB_TILE_UNITS + unit_of[gi]);
      }
    };
    // Work units: the first one is the CTA's own, the others come from a device counter, fetched by
    // the leader two units ahead (the atomic's latency hides behind a whole unit) and handed to the
    // other producer warps through shared memory + a producers-only named barrier, once per unit.
    int unit = blockIdx.x;
    int nxt = 0;
    if (leader) nxt = (int)gridDim.x + atomicAdd(a.work_counter, 1);
    prefetch_unit(unit);
    int stage = 0;
    uint32_t phase = 0;   // parity of the stage's completed fills
    uint32_t u_local = 0;
    for (; unit < a.n_items; ++u_local) {
      if (leader) s_units[u_local & 1] = nxt;
      asm volatile("bar.sync 1, %0;" ::"n"(NP * 32) : "memory");
      const int unit_next = s_units[u_local & 1];
      if (leader) nxt = (int)gridDim.x + atomicAdd(a.work_counter, 1);
      int off[UPW];
#pragma unroll
      for (int gi = 0; gi < UPW; ++gi) off[gi] = offN[gi];
      const int4 d = dN;
      prefetch_unit(unit_next);
      const int m = u_local & 1;
      if (leader) {
        mbar_wait(&s_mempty[m], ((u_local >> 1) & 1) ^ 1);   // consumers are done with unit u_local - 2
        const int64_t o = ((int64_t)(uint32_t)d.y << 32) | (uint32_t)d.x;
        bulk_g2s(s_meta + (size_t)m * CTB_META_CAP, a.blob + o, (uint32_t)d.z, &s_mfull[m]);
      }
      bool ok[UPW];   // this lane's 16-byte units of the bundle (at most 128 per day and input)
#pragma unroll
      for (int gi = 0; gi < UPW; ++gi) ok[gi] = pw + NP * gi < NG && unit_of[gi] < d.w;
      const int tb_begin = (unit / a.n_bundles) * a.chunk_tb;
      const int tb_end = min(tb_begin + a.chunk_tb, a.n_tb);
      int planeN[CTB_TB / 4] = {};
      auto load_plane = [&](int tb, int dd) {
        const int t = tb * CTB_TB + dd * 4 + l4;
        return t < a.T ? __ldg(a.tix + t) : 0;
      };
      for (int tb = tb_begin; tb < tb_end; ++tb) {
        // physical planes of this lane's 8 day rows (time_index: leap days removed, a ring of year
        // buffers ...): 8 independent loads issued before the wait for the stage, not one dependent
        // load in front of every row's copies
        int plane[CTB_TB / 4];
        if constexpr (TIX) {
#pragma unroll
          for (int dd = 0; dd < CTB_TB / 4; ++dd) plane[dd] = tb == tb_begin ? load_plane(tb, dd) : planeN[dd];
          if (tb + 1 < tb_end) {   // ... and the next tile's a whole tile ahead
#pragma unroll
            for (int dd = 0; dd < CTB_TB / 4; ++dd) planeN[dd] = load_plane(tb + 1, dd);
          }
        }
        mbar_wait_a(empty_a + stage * 8, phase ^ 1);   // the stage's previous tile is reduced
        if (leader) {
          s_desc[stage] = make_int4(tb * CTB_TB, m | (tb == tb_begin ? F_FIRST : 0) | (tb == tb_end - 1 ? F_LAST : 0), tb, 0);
          s_next[stage] = NCW;
        }
#ifdef CTB_EXPERIMENT
        if (!(a.knobs & 1))
#endif
        {
          // one 64-bit multiply-add per copy: the row pointer advances by 4 day planes per step
          uint32_t dst = tiles_a + (uint32_t)stage * CTB_STREAM_TILE_BYTES + (uint32_t)(l4 * CTB_ROWB);
          const int n_days = min(CTB_TB, a.T - tb * CTB_TB);
          if constexpr (!TIX) {
            int64_t ro = (int64_t)(tb * CTB_TB + l4) * a.stride;
#pragma unroll
            for (int dd = 0; dd < CTB_TB / 4; ++dd, dst += 4 * CTB_ROWB, ro += row_step) {
              if (dd * 4 + l4 < n_days) {
#pragma unroll
                for (int gi = 0; gi < UPW; ++gi)
                  if (ok[gi]) cp_async16(dst + dst_of[gi], (second[gi] ? X1 : X0) + ro + off[gi]);
              }
#if CTB_PACE_NS > 0
              __nanosleep(CTB_PACE_NS);
#endif
            }
          } else {
#pragma unroll
            for (int dd = 0; dd < CTB_TB / 4; ++dd, dst += 4 * CTB_ROWB) {
              if (dd * 4 + l4 < n_days) {
                // byte addressing here: row pointer (64-bit, one multiply per row) + the unit's 32-bit byte
                // offset.  (Measured: 0.69 -> 0.63 ms in this branch; the SAME form in the branch above
                // costs it 2 %, 0.60 -> 0.61 ms, so that one keeps the element arithmetic.)
                const int64_t ro = (int64_t)plane[dd] * stride_b;
                const unsigned char* const r0 = reinterpret_cast<const unsigned char*>(X0) + ro;
                const unsigned char* const r1 = reinterpret_cast<const unsigned char*>(X1) + ro;
#pragma unroll
                for (int gi = 0; gi < UPW; ++gi)
                  if (ok[gi])
                    cp_async16(dst + dst_of[gi], (NIN == 2 && second[gi] ? r1 : r0) + (uint32_t)off[gi] * (uint32_t)sizeof(TIN));
              }
#if CTB_PACE_NS > 0
              __nanosleep(CTB_PACE_NS);
#endif
            }
          }
        }
        // every producer thread's copies arrive on the stage's barrier when they have landed; the
        // leader's own arrival releases the descriptor it wrote
        cp_async_arrive_a(full_a + stage * 8);
        if (leader) mbar_arrive_a(full_a + stage * 8);
        if (++stage == S) { stage = 0; phase ^= 1; }
      }
      unit = unit_next;
    }
    // the last CTA out re-arms the counters for the next launch that uses this slot
    if (leader && atomicAdd(a.work_counter + 1, 1) == (int)gridDim.x - 1) {
      a.work_counter[0] = 0;
      a.work_counter[1] = 0;
    }
    // exit marker in the next stage
    mbar_wait_a(empty_a + stage * 8, phase ^ 1);
    if (leader) s_desc[stage] = make_int4(0, F_EXIT, 0, 0);
    mbar_arrive_a(full_a + stage * 8);
    if (leader) mbar_arrive_a(full_a + stage * 8);
  } else {
    // ------------------------------------------------------------------ consumers ---
    const int e = lane >> 3, d8 = lane & 7;
    const uint32_t lane_a = tiles_a + (uint32_t)(d8 * CTB_ROWB);
    uint32_t units_seen = 0;
    int stage = 0, rot = warp;   // rot: this warp's first region of the tile, rotating from tile to tile
    bool skip_fast = false;      // the last region failed the integer widening's range check
    unsigned probe = 0;
    uint32_t phase = 0;
    uint32_t seg_a = 0, ent_a = 0;
    int n_seg = 0;
    for (;;) {
      mbar_wait_backoff_a(full_a + stage * 8, phase);
      const uint4 d = lds_u4(desc_a + stage * 16);
      if (d.y & F_EXIT) break;
      const int m = d.y & F_SLOT;
      if (d.y & F_FIRST) {   // a new bundle: its metadata has (or will have) landed in slot m
        mbar_wait(&s_mfull[m], (units_seen >> 1) & 1);
        ++units_seen;
        const uint32_t blob_a = smem_u32(s_meta) + (uint32_t)m * CTB_META_CAP;
        const uint4 h0 = lds_u4(blob_a), h1 = lds_u4(blob_a + 16);   // CtbBlobHeader
        n_seg = (int)h0.y;
        seg_a = blob_a + h1.y /*bytes_a*/ + h0.z /*off_seg*/;
        ent_a = blob_a + h1.y + h0.w /*off_ent*/ + (uint32_t)(e * sizeof(CtbEnt));
#ifdef CTB_EXPERIMENT
        if (a.knobs & 4) n_seg = 0;
#endif
      }
      const uint32_t tile_a = lane_a + (uint32_t)stage * CTB_STREAM_TILE_BYTES;
      const int t = (int)d.x + lane;
      const bool valid = t < a.T;
      int tg = -1, tg0 = 0;
      if (a.tgroup) {
        tg = valid ? __ldg(a.tgroup + a.t_off + t) : -1;
        tg0 = __shfl_sync(0xffffffffu, tg, 0);
      }
      int doy[4] = {0, 0, 0, 0};   // day of year of the lane's four days d8 + 8 g (growing-season gate)
      if constexpr (GATE) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int tt = (int)d.x + d8 + 8 * g;
          doy[g] = tt < a.T ? __ldg(a.doy + a.t_off + tt) : 0;
        }
      }
      double* const out_t = a.out + t;
      for (int s = rot; s < n_seg;) {
        const uint4 sg = lds_u4(seg_a + (uint32_t)s * (uint32_t)sizeof(CtbSeg));
        const int target = (int)sg.x;
        const int nq = (int)((sg.y >> 16) + 3) >> 2;
        const double rden = __hiloint2double((int)sg.w, (int)sg.z);
        const uint32_t ea = ent_a + (sg.y & 0xffffu) * 4u * (uint32_t)sizeof(CtbEnt);
        double v[NOUT];
        bool done = false;
        if constexpr (NIN == 2) {
          reduce_region2<TIN, KIND, NOUT, GATE>(a.tr, tile_a, ea, nq, lane, doy, v);
          done = true;
        } else if constexpr (sizeof(TIN) == 4) {
          // data that is not positive-normal (Celsius, anomalies, precipitation with zeros) fails the
          // widening's range check in nearly every region-tile: after a failure the warp goes straight
          // to the exact loop and only probes the fast one every 8th region (measured: 0.70 -> 0.60 ms for
          // such data, 0.60 for positive data either way -- bench_micro/sign_cost.py)
          if (!(CTB_STICKY_ALL || NOUT == 1) || !skip_fast || (++probe & 7) == 0) {
            done = reduce_region_widen<KIND, NOUT, GATE>(a.tr, tile_a, ea, nq, lane, doy, v);
            skip_fast = !done;
          }
        }
        if constexpr (NIN == 1) if (!done) {
          reduce_region<TIN, KIND, NOUT, false, GATE>(a.tr, tile_a, ea, nq, lane, doy, v);
          bool bad = false;
#pragma unroll
          for (int j = 0; j < NOUT; ++j) bad |= !(fabs(v[j]) <= 1.7976931348623157e308);
          if (__any_sync(0xffffffffu, bad && valid))
            reduce_region<TIN, KIND, NOUT, true, GATE>(a.tr, tile_a, ea, nq, lane, doy, v);
        }
        if (a.tgroup) {
          ctb_emit<NOUT>(a, target, rden, v, lane, t, valid, (int)d.z, tg, tg0);
        } else if (valid) {
          if (target >= 0) {
#pragma unroll
            for (int j = 0; j < NOUT; ++j) {   // written once: leave L2 to the input
              const double val = v[j] * rden;
              if (a.n_peers == 0) {
                __stcs(out_t + ((size_t)j * a.R + target) * a.out_ld, val);
              } else {
                // fused gather: the tile's 256 bytes go to this GPU's buffer and, over NVLink, to
                // every peer's -- no collective, no staging copy after the kernel.  Rows in bundle
                // order (peer_row): the CTA's stores stay inside a few pages per peer
                const int row = a.peer_row ? __ldg(a.peer_row + target) : target;
                const size_t idx = ((size_t)j * a.R + row) * a.out_ld + t;
                for (int p = 0; p < a.n_peers; ++p) __stcs(a.peers[p] + idx, val);
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < NOUT; ++j)
              a.scratch[((size_t)j * a.n_scratch + ~target) * a.scratch_ld + t] = v[j];
          }
        }
        int nx = 0;
        if (lane == 0) nx = atom_add_a(next_a + stage * 4, 1);
        s = __shfl_sync(0xffffffffu, nx, 0);
      }
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_a(empty_a + stage * 8);
        if (d.y & F_LAST) mbar_arrive(&s_mempty[m]);
      }
      if (++stage == S) { stage = 0; phase ^= 1; }
      if (++rot == NCW) rot = 0;
    }
  }
}

#ifndef CTB_POLY34_THREADS
#define CTB_POLY34_THREADS 640
#endif
#ifndef CTB_BINS34_THREADS
#define CTB_BINS34_THREADS CTB_POLY34_THREADS
#endif
#ifndef CTB_RCS34_THREADS
#define CTB_RCS34_THREADS 512
#endif
#ifndef CTB_RCS2_THREADS
#define CTB_RCS2_THREADS 640
#endif
#ifndef CTB_EDD1_THREADS
#define CTB_EDD1_THREADS 640
#endif
#ifndef CTB_EDD2_THREADS
#define CTB_EDD2_THREADS 384
#endif
#ifndef CTB_EDD34_THREADS
#define CTB_EDD34_THREADS 512
#endif
// CTA size of the streaming kernel, one branch per transform family
constexpr int stream_threads(int kind, int nout) {
  if (kind == CTB_TR_POLY || kind == CTB_TR_POLY_SEQ) {
    // three and four polynomial outputs keep 4 fp64 accumulators per output and lane: 20 warps of 96
    return nout > 2 ? CTB_POLY34_THREADS : nout > 1 ? 768 : CTB_STREAM_THREADS;
  }
  if (kind == CTB_TR_BINS) {
    // temperature bins: the polynomial shapes (the same 4 x NOUT accumulators per lane; measured, config 2
    // shapes, 4 bins: 512 / 640 / 768 threads = 1.278 / 1.233 / 1.228 ms, profiles/micro/r3_bins_cost.log --
    // 768 is within the spread, so the bins keep the polynomial's 640)
    return nout > 2 ? CTB_BINS34_THREADS : nout > 1 ? 768 : CTB_STREAM_THREADS;
  }
  if (kind == CTB_TR_RCSPLINE) {
    // restricted cubic spline terms: more temporaries per value than the polynomial (six cubes shared or
    // not) -- 3 or 4 terms spill at 640 threads (96 registers) when gated, 2 terms at 768 (80): 16 warps of
    // 128 registers (measured, config 2 shapes with a time index, 4 terms: 384 / 512 / 640 threads = 2.078 /
    // 1.814 / 1.809 ms, profiles/micro/r3_rcspline_cost.log), 2 terms the largest CTA without spills (not swept)
    return nout > 2 ? CTB_RCS34_THREADS : nout > 1 ? CTB_RCS2_THREADS : CTB_STREAM_THREADS;
  }
  if (kind == CTB_TR_EDD || kind == CTB_TR_GDD) {
    // Snyder forms: threshold evaluations per gridcell-day -- few warps with many registers: the compiler
    // interleaves the 4 days x evals dependency chains of a quad inside one warp (measured, config 4:
    // 768/640/512/448/384/256 threads = 4.53/4.33/4.12/4.49/3.91/5.31 ms; consumer warps a multiple of 4;
    // EDD with 3 or 4 thresholds: 512 threads 3.00/3.92 ms per 730 days, 384 threads 3.03/4.24;
    // GDD with 2 outputs: 3.57 / 3.28)
    if (kind == CTB_TR_GDD) return CTB_EDD2_THREADS;
    return nout == 1 ? CTB_EDD1_THREADS : nout == 2 ? CTB_EDD2_THREADS : CTB_EDD34_THREADS;
  }
  // 24 warps of 80 registers (measured, config 2: 1024 / 896 / 768 / 640 / 512 threads = 0.619 / 0.609 /
  // 0.599 / 0.611 / 0.672 ms; the reduction alone is fastest with 32 warps, the whole kernel with 24)
  return CTB_STREAM_THREADS;
}

template <typename TIN, int KIND, int NOUT>
int launch(const ctb_plan* P, AggArgs a, cudaStream_t st) {
  constexpr int NIN = ctb_tr_nin(KIND);
  constexpr int THREADS = stream_threads(KIND, NOUT);
  constexpr int S = CTB_STAGES;   // tile stages: one being reduced, up to two landing
  constexpr size_t SMEM = (size_t)S * Geo<NIN>::TILE_BYTES + 2 * CTB_META_CAP;
  static_assert(SMEM <= 227 * 1024 - 512, "shared memory budget");
  static int n_sm[64] = {0};
  static bool attr_set[64][2][2] = {{{false}}};
  const int dev = P->device & 63;
  const bool gate = a.doy != nullptr;   // growing-season gate: its own instantiation (the inner loop tests it)
  const bool tix = a.tix != nullptr;
  auto k = gate ? (tix ? agg_stream_kernel<TIN, KIND, NOUT, THREADS, S, true, true>
                       : agg_stream_kernel<TIN, KIND, NOUT, THREADS, S, true, false>)
                : (tix ? agg_stream_kernel<TIN, KIND, NOUT, THREADS, S, false, true>
                       : agg_stream_kernel<TIN, KIND, NOUT, THREADS, S, false, false>);
  if (!attr_set[dev][gate][tix]) {
    CTB_CUDA(cudaDeviceGetAttribute(&n_sm[dev], cudaDevAttrMultiProcessorCount, P->device));
    CTB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    attr_set[dev][gate][tix] = true;
  }
  a.n_stages = S;
  a.tile_stride = Geo<NIN>::TILE_BYTES;
  a.n_tb = (a.T + CTB_TB - 1) / CTB_TB;
  // units: chunks of up to 8 time blocks, shorter when there would be too few units to fill the GPU
  const int64_t tiles = (int64_t)P->n_bundles * a.n_tb;
  int chunk = (int)std::max<int64_t>(1, std::min<int64_t>(8, tiles / ((int64_t)n_sm[dev] * 6)));
#ifdef CTB_EXPERIMENT
  if (a.chunk_tb > 0) chunk = a.chunk_tb;
#endif
  const int n_chunks = (a.n_tb + chunk - 1) / chunk;
  chunk = (a.n_tb + n_chunks - 1) / n_chunks;
  const int64_t n_units = (int64_t)P->n_bundles * n_chunks;
  if (n_units >= (1ll << 31)) { ctb_set_error("too many work units"); return CTB_ERR_UNSUPPORTED; }
  a.chunk_tb = chunk;
  a.n_bundles = P->n_bundles;
  a.n_items = (int)n_units;
  // {next unit, CTAs done} pairs, zero between launches (the kernel re-arms its pair); launches of
  // one plan that run concurrently on different streams take different pairs
  a.work_counter = P->d_work_counter + 2 * (P->work_counter_slot.fetch_add(1) % (CTB_N_WORK_COUNTERS / 2));
  if (n_units > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>(n_units, n_sm[dev]);
    k<<<grid, THREADS, SMEM, st>>>(a);
    CTB_LAUNCH_CHECK();
  }
  return CTB_OK;
}

}  // namespace

// One translation unit per input type (ctb_stream_f32.cu / ctb_stream_f64.cu: they compile in parallel; the
// instantiations of one type take about a minute and a half).
int CTB_STREAM_ENTRY(const ctb_plan* P, const AggArgs& a, int kind, int n_out, cudaStream_t st) {
  auto go = [&](auto k, auto nout) { return launch<CTB_STREAM_TIN, k, nout>(P, a, st); };
  if (kind == CTB_TR_POLY) {
    bool seq = true;   // orders 1..n_out (tas_poly's usual call): no order tests in the kernel
    for (int j = 0; j < n_out; ++j) seq = seq && a.tr.ip[j] == j + 1;
    if (seq) return ctb_dispatch_nout<CTB_TR_POLY_SEQ>(n_out, go);
  }
  return ctb_dispatch_transform(kind, n_out, go);
}
