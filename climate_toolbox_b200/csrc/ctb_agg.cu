// Dispatch of ctb_aggregate / ctb_aggregate_grouped, and the kernels beside the streaming kernel
// (ctb_stream_impl.cuh, every TIME_MAJOR input whose planes are 16-byte aligned):
//
//   agg_direct_kernel  CELL_MAJOR input [lat][lon][T] (the reference test fixture), and the
//                      fallback for planes that are not 16-byte aligned: one warp per
//                      (region, 32-day tile), lane = day.
//   agg_fixup_kernel   regions split over several bundles, and regions without kept rows:
//                      out[r][t] = (sum of the region's partial rows, fixed order) / den[r].
//   agg_group_finish_kernel  fused time reduction: per-tile partial sums -> output columns.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "ctb_internal.cuh"

namespace {

// one CSR entry: acc_j += w * f_j(x), NaN products skipped (skipna sum, aggregations.py:78)
template <typename TIN, int KIND, int NOUT>
__device__ __forceinline__ void accumulate(const CtbTr& tr, double w, TIN r0, TIN r1, bool on, double (&acc)[NOUT]) {
  double f[NOUT];
  ctb_apply<KIND, NOUT>(tr, (double)r0, (double)r1, f);
#pragma unroll
  for (int j = 0; j < NOUT; ++j) {
    const double p = w * f[j];
    if (on && p == p) acc[j] += p;
  }
}

// time group of the lane's day (fused time reduction), and of the tile's first day
__device__ __forceinline__ void lane_group(const AggArgs& a, int t, bool valid, int& tg, int& tg0) {
  tg = -1;
  tg0 = 0;
  if (a.tgroup) {
    tg = valid ? __ldg(a.tgroup + a.t_off + t) : -1;
    tg0 = __shfl_sync(0xffffffffu, tg, 0);
  }
}

// Regions split over several bundles (and regions with no kept rows):
// out[r][t] = (sum of the region's partial rows, fixed order) / den[r]; with a time reduction
// out[r][g] = sum over the days of column g of that.
__global__ void agg_fixup_kernel(const AggArgs a, int n_out) {
  const int i = blockIdx.x;
  const int r = a.split_region[i];
  const int s0 = a.split_slot_ptr[i], s1 = a.split_slot_ptr[i + 1];
  const double d = a.den[r];
  for (int j = 0; j < n_out; ++j) {
    if (!a.tgroup) {
      for (int t = blockIdx.y * blockDim.x + threadIdx.x; t < a.T; t += gridDim.y * blockDim.x) {
        double s = 0.0;
        for (int q = s0; q < s1; ++q) s += a.scratch[((size_t)j * a.n_scratch + q) * a.scratch_ld + t];
        if (a.n_peers == 0) {
          a.out[((size_t)j * a.R + r) * a.out_ld + t] = s / d;
        } else {
          const int row = a.peer_row ? a.peer_row[r] : r;
          for (int p = 0; p < a.n_peers; ++p) a.peers[p][((size_t)j * a.R + row) * a.out_ld + t] = s / d;
        }
      }
    } else {
      for (int g = blockIdx.y * blockDim.x + threadIdx.x; g < a.n_groups; g += gridDim.y * blockDim.x) {
        double sum = 0.0;
        for (int t = a.g_t_lo[g]; t < a.g_t_hi[g]; ++t) {
          double s = 0.0;
          for (int q = s0; q < s1; ++q) s += a.scratch[((size_t)j * a.n_scratch + q) * a.scratch_ld + t];
          sum += s / d;
        }
        a.out[((size_t)j * a.R + r) * a.out_ld + g] = sum;
      }
    }
  }
}

// fused time reduction: out[j][r][g] = sum over the tiles that touch column g of their partial
// sums, in tile order
__global__ void agg_group_finish_kernel(const AggArgs a, int n_out) {
  const int64_t n = (int64_t)n_out * a.R * a.n_groups;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(i % a.n_groups);
    const int64_t jr = i / a.n_groups;
    const int t_lo = a.g_t_lo[g], t_hi = a.g_t_hi[g];
    double s = 0.0;
    if (t_hi > t_lo) {
      for (int tb = t_lo / CTB_TB; tb <= (t_hi - 1) / CTB_TB; ++tb) {
        const int k = g - a.tgroup[tb * CTB_TB];
        s += a.gpart[((size_t)jr * a.g_ntb + tb) * a.gk + k];
      }
    }
    a.out[(size_t)jr * a.out_ld + g] = s;
  }
}

// ---- direct kernel: warp per (region, 32-day tile) ---------------------------
template <typename TIN, int KIND, int NOUT, int LAYOUT>
__global__ void __launch_bounds__(256) agg_direct_kernel(const AggArgs a) {
  constexpr int NIN = ctb_tr_nin(KIND);
  const int lane = threadIdx.x & 31;
  const int n_tiles = (a.T + 31) / 32;
  const int64_t n_work = (int64_t)a.R * n_tiles;
  const TIN* __restrict__ X0 = reinterpret_cast<const TIN*>(a.x0);
  const TIN* __restrict__ X1 = reinterpret_cast<const TIN*>(a.x1);
  for (int64_t wk = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); wk < n_work;
       wk += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    const int r = (int)(wk / n_tiles);
    const int tb = (int)(wk % n_tiles);
    const int t = tb * 32 + lane;
    const bool tv = t < a.T;
    const int64_t tp = tv ? (a.tix ? a.tix[t] : t) : 0;
    int tg, tg0;
    lane_group(a, t, tv, tg, tg0);
    const int doy = (a.doy && tv) ? __ldg(a.doy + a.t_off + t) : 0;
    double acc[NOUT];
#pragma unroll
    for (int j = 0; j < NOUT; ++j) acc[j] = 0.0;
    const int e0 = a.row_ptr[r], e1 = a.row_ptr[r + 1];
    for (int e = e0; e < e1; ++e) {
      const double w = __ldg(a.w + e);
      const int64_t c = __ldg(a.col + e);
      const int64_t off = (LAYOUT == CTB_LAYOUT_CELL_MAJOR) ? c * a.stride + tp : tp * a.stride + c;
      double x0 = 0.0, x1 = 0.0;
      if (tv) {
        x0 = (double)__ldg(X0 + off);
        if constexpr (NIN == 2) x1 = (double)__ldg(X1 + off);
      }
      accumulate<double, KIND, NOUT>(a.tr, w, x0, x1, a.doy ? ctb_gate_on(__ldg(a.gate + e), doy) : true, acc);
    }
    // 1/den: the same normalisation as the staged kernels (0 * inf = NaN, x * inf = +-inf)
    ctb_emit<NOUT>(a, r, 1.0 / a.den[r], acc, lane, t, tv, tb, tg, tg0);
  }
}

// ------------------------------------------------------------- dispatch -----
template <typename TIN, int KIND, int NOUT>
int launch_direct(const AggArgs& a, int layout, cudaStream_t st) {
  AggArgs b = a;
  b.n_tb = (a.T + CTB_TB - 1) / CTB_TB;
  const int64_t n_work = (int64_t)a.R * b.n_tb;
  if (n_work == 0) return CTB_OK;
  const unsigned grid = (unsigned)std::min<int64_t>((n_work + 7) / 8, 148 * 64);
  if (layout == CTB_LAYOUT_CELL_MAJOR)
    agg_direct_kernel<TIN, KIND, NOUT, CTB_LAYOUT_CELL_MAJOR><<<grid, 256, 0, st>>>(b);
  else
    agg_direct_kernel<TIN, KIND, NOUT, CTB_LAYOUT_TIME_MAJOR><<<grid, 256, 0, st>>>(b);
  CTB_LAUNCH_CHECK();
  return CTB_OK;
}

size_t scratch_bytes(const ctb_plan* plan, int64_t T, int n_out) {
  return (size_t)plan->n_scratch * (size_t)T * (size_t)n_out * sizeof(double);
}
size_t gpart_bytes(const ctb_plan* plan, const ctb_time_groups* g, int n_out) {
  const size_t n_tb = (size_t)((g->T + CTB_TB - 1) / CTB_TB);
  return (size_t)n_out * (size_t)plan->R * n_tb * (size_t)g->gk * sizeof(double);
}

int aggregate_impl(const ctb_plan* P, const void* x0, const void* x1, int dtype, int layout,
                   int64_t stride, const int32_t* time_index, int64_t T, int transform,
                   const double* params, int n_params, int n_out, const ctb_time_groups* G,
                   int64_t t_begin, int flush, const int32_t* day_of_year, double* const* peer_out,
                   int n_peer_out, const int32_t* peer_row, double* out,
                   int64_t out_ld, void* workspace, size_t workspace_bytes, int variant, void* stream) {
  const char* fn = G ? "ctb_aggregate_grouped" : "ctb_aggregate";
  if (day_of_year && P && !P->has_gate) {
    ctb_set_error("%s: day_of_year given, but the plan was built without ctb_plan_opts.cell_gate", fn);
    return CTB_ERR_INVALID;
  }
  if (n_peer_out < 0 || n_peer_out > CTB_MAX_PEERS || (n_peer_out > 0 && (!peer_out || G))) {
    ctb_set_error("%s: peer_out takes 1..%d buffers and no time groups", fn, CTB_MAX_PEERS);
    return CTB_ERR_INVALID;
  }
  if (n_peer_out > 0) out = peer_out[0];
  if (!P || !x0 || (!out && T > 0 && P->R > 0)) { ctb_set_error("%s: null argument", fn); return CTB_ERR_INVALID; }
  const int64_t n_cols = G ? G->n_groups : T;
  if (out_ld == 0) out_ld = n_cols;
  if (T < 0 || T >= (1ll << 31) || stride < 0 || out_ld < n_cols) { ctb_set_error("%s: bad T/stride/out_ld", fn); return CTB_ERR_INVALID; }
  if (G && (t_begin < 0 || t_begin % CTB_TB != 0 || t_begin + T > G->T || G->device != P->device)) {
    ctb_set_error("%s: window [%lld, %lld) does not fit time groups of %lld days on device %d (t_begin must be a multiple of %d)",
                  fn, (long long)t_begin, (long long)(t_begin + T), (long long)G->T, G->device, CTB_TB);
    return CTB_ERR_INVALID;
  }
  if (dtype != CTB_F32 && dtype != CTB_F64) { ctb_set_error("dtype=%d unsupported", dtype); return CTB_ERR_INVALID; }
  if (layout != CTB_LAYOUT_TIME_MAJOR && layout != CTB_LAYOUT_CELL_MAJOR) { ctb_set_error("layout=%d unsupported", layout); return CTB_ERR_INVALID; }
  AggArgs a{};
  int rc = ctb_pack_transform(transform, params, n_params, n_out, &a.tr);
  if (rc) return rc;
  if (ctb_tr_nin(transform) == 2 && !x1) { ctb_set_error("transform needs two inputs"); return CTB_ERR_INVALID; }
  variant &= 0xff;   // bit 8 (inputs in mapped host memory) needs no special handling
  if (variant == 0) variant = (layout == CTB_LAYOUT_TIME_MAJOR) ? 1 : 2;
  if (variant != 2 && layout != CTB_LAYOUT_TIME_MAJOR) { ctb_set_error("staged variant needs TIME_MAJOR input"); return CTB_ERR_INVALID; }
  if (variant != 1 && variant != 2) { ctb_set_error("variant=%d unsupported", variant); return CTB_ERR_INVALID; }
  const size_t es = dtype == CTB_F32 ? 4 : 8;
  const bool vec = (P->ncell % CTB_PIECE == 0) && ((stride * es) % 16 == 0) &&
                   ((uintptr_t)x0 % 16 == 0) && (!x1 || (uintptr_t)x1 % 16 == 0);
  // the streaming kernel copies 16-byte units: planes that are not 16-byte aligned take the direct kernel
  if (variant == 1 && !vec) variant = 2;
  if (variant != 2 && P->elem_bytes != (int)es) {
    ctb_set_error("plan was built for %d-byte elements, input has %d-byte elements: rebuild it with "
                  "elem_bytes=%d", P->elem_bytes, (int)es, (int)es);
    return CTB_ERR_UNSUPPORTED;
  }
  if (variant != 2 && P->stage_bytes < ctb_tr_nin(transform) * (int)es) {
    ctb_set_error("plan stages %d bytes per gridcell-day, the transform needs %d: rebuild it with "
                  "stage_bytes_per_cell_day=%d", P->stage_bytes, ctb_tr_nin(transform) * (int)es,
                  ctb_tr_nin(transform) * (int)es);
    return CTB_ERR_UNSUPPORTED;
  }
  // workspace: [partial rows of split regions][per-tile partial sums of the time reduction]
  const size_t need_s = variant != 2 ? scratch_bytes(P, G ? G->T : T, n_out) : 0;
  const size_t need_g = G ? gpart_bytes(P, G, n_out) : 0;
  if (need_s + need_g > 0 && (!workspace || workspace_bytes < need_s + need_g)) {
    ctb_set_error("workspace of %zu bytes required, got %zu", need_s + need_g, workspace ? workspace_bytes : (size_t)0);
    return CTB_ERR_INVALID;
  }
  if (P->R == 0 || (T == 0 && !(G && flush))) return CTB_OK;

  CtbDeviceGuard guard(P->device);
  if (guard.err != cudaSuccess) { ctb_set_error("cudaSetDevice(%d) failed: %s", P->device, cudaGetErrorString(guard.err)); return CTB_ERR_CUDA; }
  a.x0 = x0; a.x1 = x1; a.stride = stride; a.tix = time_index; a.T = (int)T; a.out_ld = out_ld; a.ncell = P->ncell;
  a.R = P->R; a.out = out; a.scratch = (double*)workspace; a.n_scratch = P->n_scratch;
  a.den = P->d_den;
  a.blob = P->d_blob; a.b_desc = P->d_b_desc; a.unit_tab = P->d_unit_tab; a.row_ptr = P->d_row_ptr; a.col = P->d_col;
  a.w = P->d_w; a.split_region = P->d_split_region; a.split_slot_ptr = P->d_split_slot_ptr;
  a.n_split = P->n_split;
  a.n_tb = (int)((T + CTB_TB - 1) / CTB_TB);
  a.scratch_ld = T;
  a.doy = day_of_year; a.gate = P->d_gate;
  a.n_peers = n_peer_out;
  a.peer_row = n_peer_out ? peer_row : nullptr;
  for (int p = 0; p < n_peer_out; ++p) a.peers[p] = peer_out[p];
  if (G) {
    a.tgroup = G->d_group; a.gk = G->gk; a.n_groups = G->n_groups; a.g_t_lo = G->d_t_lo; a.g_t_hi = G->d_t_hi;
    a.g_ntb = (int)((G->T + CTB_TB - 1) / CTB_TB); a.t_off = (int)t_begin; a.scratch_ld = G->T;
    a.gpart = reinterpret_cast<double*>(static_cast<char*>(workspace) + need_s);
  }
#ifdef CTB_EXPERIMENT
  if (const char* e = getenv("CTB_KNOBS")) a.knobs = atoi(e);
  if (const char* e = getenv("CTB_STAGES")) a.n_stages = atoi(e);
  if (const char* e = getenv("CTB_CHUNK_TB")) a.chunk_tb = atoi(e);
#endif
  cudaStream_t st = (cudaStream_t)stream;
  if (T > 0) {
    // variant 1 = the streaming kernel (ctb_stream_impl.cuh), 2 = direct
    rc = variant == 1 ? ctb_launch_stream(P, a, dtype, transform, n_out, st)
                      : ctb_dispatch_transform(transform, n_out, [&](auto kind, auto nout) {
                          return dtype == CTB_F32 ? launch_direct<float, kind, nout>(a, layout, st)
                                                  : launch_direct<double, kind, nout>(a, layout, st);
                        });
    if (rc) return rc;
  }
  if (G && !flush) return CTB_OK;
  if (G) {
    a.T = (int)G->T;
    const int64_t n = (int64_t)n_out * P->R * G->n_groups;
    agg_group_finish_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 16), 256, 0, st>>>(a, n_out);
    CTB_LAUNCH_CHECK();
  }
  if (variant != 2 && P->n_split > 0) {
    const int64_t cols = G ? G->n_groups : T;
    const dim3 g2(P->n_split, (unsigned)std::min<int64_t>((cols + 255) / 256, 64));
    agg_fixup_kernel<<<g2, 256, 0, st>>>(a, n_out);
    CTB_LAUNCH_CHECK();
  }
  return CTB_OK;
}

}  // namespace

int ctb_pack_transform(int transform, const double* params, int n_params, int n_out, CtbTr* out) {
  std::memset(out, 0, sizeof *out);
  if (n_out < 1 || n_out > CTB_MAX_OUT) {
    ctb_set_error("n_out=%d out of range 1..%d", n_out, CTB_MAX_OUT);
    return CTB_ERR_INVALID;
  }
  auto need = [&](int n) {
    if (n_params == n && (n == 0 || params)) return true;
    ctb_set_error("transform %d with n_out=%d needs %d params, got %d", transform, n_out, n, n_params);
    return false;
  };
  switch (transform) {
    case CTB_TR_IDENTITY:
      if (n_out != 1) { ctb_set_error("IDENTITY has n_out=1"); return CTB_ERR_INVALID; }
      return CTB_OK;
    case CTB_TR_POLY:
      if (!need(1 + n_out)) return CTB_ERR_INVALID;
      out->a[0] = params[0];
      for (int j = 0; j < n_out; ++j) {
        const double p = params[1 + j];
        if (p != (double)(int)p || p < -64 || p > 64) {
          ctb_set_error("POLY power %g is not a small integer", p);
          return CTB_ERR_UNSUPPORTED;
        }
        out->ip[j] = (int)p;
      }
      return CTB_OK;
    case CTB_TR_EDD:
    case CTB_TR_GDD: {
      const int n = transform == CTB_TR_EDD ? n_out : 2 * n_out;
      if (!need(n)) return CTB_ERR_INVALID;
      for (int j = 0; j < n; ++j) {
        const double e = params[j];
        out->a[j] = e;
        const float f = (float)e;          // nearest; then the neighbours that bracket e
        out->up[j] = (double)f < e ? std::nextafterf(f, INFINITY) : f;
        out->dn[j] = (double)f > e ? std::nextafterf(f, -INFINITY) : f;
      }
      return CTB_OK;
    }
    case CTB_TR_BINS: {
      // {offset, e_0..e_nout}: n_out contiguous bins [e_j, e_j+1) (at most 1 + 5 of the 8 slots of CtbTr::a)
      if (!need(n_out + 2)) return CTB_ERR_INVALID;
      if (!std::isfinite(params[0])) {
        ctb_set_error("BINS offset %g is not finite", params[0]);
        return CTB_ERR_INVALID;
      }
      // strictly increasing edges can be infinite only at the ends: -inf first, +inf last
      for (int j = 0; j <= n_out; ++j) {
        const double e = params[1 + j];
        if (std::isnan(e) || (j > 0 && !(e > params[j]))) {
          ctb_set_error("BINS edges must be strictly increasing and not NaN: edge %d is %g", j, e);
          return CTB_ERR_INVALID;
        }
      }
      for (int j = 0; j < n_out + 2; ++j) out->a[j] = params[j];
      // float inputs: up[j] = the least float f with fl64(f - offset) >= e_j (-inf for e_0 = -inf, +inf for
      // e_nout = +inf), so that f >= up[j] decides the edge on the stored type (ctb_bins_in_f32)
      for (int j = 0; j <= n_out; ++j) {
        const double e = params[1 + j];
        auto ge = [&](float f) { return (double)f - params[0] >= e; };
        float f = (float)(e + params[0]);
        while (f > -INFINITY && ge(f)) f = std::nextafterf(f, -INFINITY);
        while (!ge(f)) f = std::nextafterf(f, INFINITY);
        out->up[j] = f;
      }
      return CTB_OK;
    }
    case CTB_TR_RCSPLINE: {
      // {offset, first, k_1..k_n}: outputs B_first .. B_{first+n_out-1} of the n - 1 basis functions
      const int n = n_params - 2;
      if (n < 3 || n > 7 || !params) {
        ctb_set_error("RCSPLINE takes 3..7 knots: n_params = n + 2 = 5..9, got %d", n_params);
        return CTB_ERR_INVALID;
      }
      const double off = params[0], first = params[1];
      const double* k = params + 2;   // k[0] = k_1
      if (!std::isfinite(off)) {
        ctb_set_error("RCSPLINE offset %g is not finite", off);
        return CTB_ERR_INVALID;
      }
      for (int i = 0; i < n; ++i) {
        if (!std::isfinite(k[i]) || (i > 0 && !(k[i] > k[i - 1]))) {
          ctb_set_error("RCSPLINE knots must be finite and strictly increasing: knot %d is %g", i + 1, k[i]);
          return CTB_ERR_INVALID;
        }
      }
      if (first != std::floor(first) || first < 0 || first + n_out > n - 1) {
        ctb_set_error("RCSPLINE first=%g with n_out=%d: need an integer first >= 0 and first + n_out <= %d (n - 1 "
                      "basis functions of %d knots)", first, n_out, n - 1, n);
        return CTB_ERR_INVALID;
      }
      // packed for ctb_rcs: a[0] = offset, a[1 + j] = the knot k_i of output j, i = first + j, and its
      // b_i = (k_{n-1} - k_i) / (k_n - k_{n-1}) in the bytes of dn[2j..2j+1] (ctb_rcs_b); a[1] stays 0 when
      // output 0 is the linear term B_0 (ip[0] = 1); a[5] = k_{n-1}, a[6] = k_n
      const int f0 = (int)first;
      out->a[0] = off;
      out->ip[0] = f0 == 0;
      out->a[5] = k[n - 2];
      out->a[6] = k[n - 1];
      for (int j = 0; j < n_out; ++j) {
        if (f0 + j == 0) continue;
        const double ki = k[f0 + j - 1], b = (k[n - 2] - ki) / (k[n - 1] - k[n - 2]);
        out->a[1 + j] = ki;
        std::memcpy(&out->dn[2 * j], &b, sizeof b);
      }
      // float inputs: up[m] = the least float f with fl64(f) - offset > a[m], so that f >= up[m] decides
      // c(a[m]) != 0 on the stored type (NaN aside)
      for (int m = 1; m <= 6; ++m) {
        if (m > n_out && m < 5) continue;
        auto gt = [&](float f) { return (double)f - off > out->a[m]; };
        float f = (float)(out->a[m] + off);
        while (f > -INFINITY && gt(f)) f = std::nextafterf(f, -INFINITY);
        while (!gt(f)) f = std::nextafterf(f, INFINITY);
        out->up[m] = f;
      }
      return CTB_OK;
    }
  }
  ctb_set_error("transform=%d unsupported", transform);
  return CTB_ERR_INVALID;
}

extern "C" size_t ctb_aggregate_workspace_bytes(const ctb_plan* plan, int64_t T, int n_out) {
  if (!plan || T <= 0 || n_out <= 0) return 0;
  return scratch_bytes(plan, T, n_out);
}

extern "C" int ctb_aggregate(const ctb_plan* P, const void* x0, const void* x1, int dtype,
                             int layout, int64_t stride, const int32_t* time_index, int64_t T,
                             int transform, const double* params, int n_params, int n_out,
                             double* out, int64_t out_ld, void* workspace,
                             size_t workspace_bytes, int variant, void* stream) {
  return aggregate_impl(P, x0, x1, dtype, layout, stride, time_index, T, transform, params, n_params, n_out,
                        nullptr, 0, 1, nullptr, nullptr, 0, nullptr, out, out_ld, workspace, workspace_bytes, variant,
                        stream);
}

// ------------------------------------------------------------ time groups ---
extern "C" int ctb_time_groups_create(const int32_t* group_of_day, int64_t T, int device,
                                      ctb_time_groups** out) {
  if (!out || T < 0 || T >= (1ll << 31) || (T > 0 && !group_of_day)) { ctb_set_error("ctb_time_groups_create: bad argument"); return CTB_ERR_INVALID; }
  *out = nullptr;
  for (int64_t t = 0; t < T; ++t) {
    const int32_t g = group_of_day[t], prev = t ? group_of_day[t - 1] : 0;
    if (g < prev || g > prev + 1 || (t == 0 && g != 0)) {
      ctb_set_error("ctb_time_groups_create: group_of_day must start at 0 and grow by 0 or 1 per day (day %lld: %d after %d)",
                    (long long)t, g, prev);
      return CTB_ERR_INVALID;
    }
  }
  ctb_time_groups* G = new ctb_time_groups();
  G->device = device; G->T = T;
  G->n_groups = T ? group_of_day[T - 1] + 1 : 0;
  std::vector<int32_t> lo(std::max(G->n_groups, 1), 0), hi(std::max(G->n_groups, 1), 0);
  for (int64_t t = T - 1; t >= 0; --t) lo[group_of_day[t]] = (int32_t)t;
  for (int64_t t = 0; t < T; ++t) hi[group_of_day[t]] = (int32_t)t + 1;
  G->gk = 1;
  for (int64_t t0 = 0; t0 < T; t0 += CTB_TB)
    G->gk = std::max(G->gk, group_of_day[std::min<int64_t>(t0 + CTB_TB, T) - 1] - group_of_day[t0] + 1);
  CtbDeviceGuard guard(device);
  auto fail = [&](cudaError_t e) {
    ctb_set_error("ctb_time_groups_create: %s", cudaGetErrorString(e));
    cudaFree(G->d_group); cudaFree(G->d_t_lo); cudaFree(G->d_t_hi);
    delete G;
    return CTB_ERR_CUDA;
  };
  cudaError_t e;
  if (guard.err != cudaSuccess) return fail(guard.err);
  const size_t nT = (size_t)std::max<int64_t>(T, 1), nG = lo.size();
  if ((e = cudaMalloc((void**)&G->d_group, nT * 4)) != cudaSuccess) return fail(e);
  if ((e = cudaMalloc((void**)&G->d_t_lo, nG * 4)) != cudaSuccess) return fail(e);
  if ((e = cudaMalloc((void**)&G->d_t_hi, nG * 4)) != cudaSuccess) return fail(e);
  if (T && (e = cudaMemcpy(G->d_group, group_of_day, (size_t)T * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  if ((e = cudaMemcpy(G->d_t_lo, lo.data(), nG * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  if ((e = cudaMemcpy(G->d_t_hi, hi.data(), nG * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
  *out = G;
  return CTB_OK;
}

extern "C" void ctb_time_groups_free(ctb_time_groups* G) {
  if (!G) return;
  CtbDeviceGuard guard(G->device);
  cudaFree(G->d_group); cudaFree(G->d_t_lo); cudaFree(G->d_t_hi);
  delete G;
}

extern "C" int32_t ctb_time_groups_count(const ctb_time_groups* G) { return G ? G->n_groups : 0; }

extern "C" size_t ctb_aggregate_grouped_workspace_bytes(const ctb_plan* plan, const ctb_time_groups* G,
                                                        int n_out) {
  if (!plan || !G || G->T <= 0 || n_out <= 0) return 0;
  return scratch_bytes(plan, G->T, n_out) + gpart_bytes(plan, G, n_out);
}

extern "C" int ctb_aggregate_grouped(const ctb_plan* P, const void* x0, const void* x1, int dtype,
                                     int layout, int64_t stride, const int32_t* time_index, int64_t T,
                                     int transform, const double* params, int n_params, int n_out,
                                     const ctb_time_groups* groups, int64_t t_begin, int flush,
                                     double* out, int64_t out_ld,
                                     void* workspace, size_t workspace_bytes, int variant, void* stream) {
  if (!groups) { ctb_set_error("ctb_aggregate_grouped: null time groups"); return CTB_ERR_INVALID; }
  return aggregate_impl(P, x0, x1, dtype, layout, stride, time_index, T, transform, params, n_params, n_out,
                        groups, t_begin, flush, nullptr, nullptr, 0, nullptr, out, out_ld, workspace, workspace_bytes,
                        variant, stream);
}

extern "C" int ctb_aggregate_ex(const ctb_plan* P, const void* x0, const void* x1, int dtype, int layout,
                                int64_t stride, const int32_t* time_index, int64_t T, int transform,
                                const double* params, int n_params, int n_out, const ctb_agg_opts* opts,
                                double* out, int64_t out_ld, void* workspace, size_t workspace_bytes,
                                int variant, void* stream) {
  const ctb_agg_opts none{};
  const ctb_agg_opts& o = opts ? *opts : none;
  return aggregate_impl(P, x0, x1, dtype, layout, stride, time_index, T, transform, params, n_params, n_out,
                        o.groups, o.groups ? o.t_begin : 0, o.groups ? o.flush : 1, o.day_of_year, o.peer_out,
                        o.n_peer_out, o.peer_row, out, out_ld, workspace, workspace_bytes, variant, stream);
}

// ------------------------------------------------- peer-shared buffers (CUDA IPC) ---
extern "C" int ctb_ipc_alloc(size_t bytes, int device, void** ptr, void* handle_out) {
  if (!ptr || !handle_out || bytes == 0) { ctb_set_error("ctb_ipc_alloc: bad argument"); return CTB_ERR_INVALID; }
  static_assert(sizeof(cudaIpcMemHandle_t) == CTB_IPC_HANDLE_BYTES, "IPC handle size");
  CtbDeviceGuard guard(device);
  CTB_CUDA(guard.err);
  CTB_CUDA(cudaMalloc(ptr, bytes));
  cudaIpcMemHandle_t h;
  const cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
  if (e != cudaSuccess) {
    cudaFree(*ptr);
    *ptr = nullptr;
    ctb_set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return CTB_ERR_CUDA;
  }
  std::memcpy(handle_out, &h, sizeof h);
  return CTB_OK;
}

extern "C" int ctb_ipc_open(const void* handle, int device, void** ptr) {
  if (!ptr || !handle) { ctb_set_error("ctb_ipc_open: bad argument"); return CTB_ERR_INVALID; }
  CtbDeviceGuard guard(device);
  CTB_CUDA(guard.err);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, sizeof h);
  CTB_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return CTB_OK;
}

extern "C" int ctb_ipc_close(void* ptr, int device) {
  if (!ptr) return CTB_OK;
  CtbDeviceGuard guard(device);
  CTB_CUDA(guard.err);
  CTB_CUDA(cudaIpcCloseMemHandle(ptr));
  return CTB_OK;
}

extern "C" int ctb_ipc_free(void* ptr, int device) {
  if (!ptr) return CTB_OK;
  CtbDeviceGuard guard(device);
  CTB_CUDA(guard.err);
  CTB_CUDA(cudaFree(ptr));
  return CTB_OK;
}
