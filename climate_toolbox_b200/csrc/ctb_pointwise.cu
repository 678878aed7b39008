// Pointwise helpers: materialise what the reference materialises when a caller
// asks for it (`.values` of a transformed or reindexed variable).  Not on the
// fused hot path, which never materialises these intermediates.
//   ctb_transform   : transformations.py:69-89 (Snyder EDD), :139-141 (GDD), :189 (poly), temperature bins,
//                     restricted cubic spline terms
//   ctb_gather_rows : aggregations.py:27 (ds.sel pointwise gather)
#include <algorithm>

#include "ctb_internal.cuh"

namespace {

template <typename TIN, int KIND, int NOUT>
__global__ void transform_kernel(const TIN* __restrict__ x0, const TIN* __restrict__ x1, int64_t n,
                                 CtbTr tr, double* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const double a = (double)x0[i];
    double b = 0.0;
    if constexpr (ctb_tr_nin(KIND) == 2) b = (double)x1[i];
    double f[NOUT];
    ctb_apply<KIND, NOUT>(tr, a, b, f);
#pragma unroll
    for (int j = 0; j < NOUT; ++j) out[(size_t)j * n + i] = f[j];
  }
}

template <typename TIN, int KIND, int NOUT>
int launch_tr(const void* x0, const void* x1, int64_t n, const CtbTr& tr, double* out, cudaStream_t st) {
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 32);
  transform_kernel<TIN, KIND, NOUT><<<grid, 256, 0, st>>>((const TIN*)x0, (const TIN*)x1, n, tr, out);
  CTB_LAUNCH_CHECK();
  return CTB_OK;
}

template <typename TIN, int LAYOUT>
__global__ void gather_rows_kernel(const TIN* __restrict__ x, int64_t stride,
                                   const int32_t* __restrict__ row_cell, int64_t n_rows,
                                   const int32_t* __restrict__ tix, int64_t T, TIN* __restrict__ out) {
  const int64_t total = n_rows * T;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t k, t;
    if (LAYOUT == CTB_LAYOUT_TIME_MAJOR) { t = i / n_rows; k = i % n_rows; }
    else { k = i / T; t = i % T; }
    const int64_t tp = tix ? tix[t] : t;
    const int64_t c = row_cell[k];
    out[i] = (LAYOUT == CTB_LAYOUT_TIME_MAJOR) ? x[tp * stride + c] : x[c * stride + tp];
  }
}

template <typename TIN>
int launch_gather(const ctb_plan* P, const void* x, int layout, int64_t stride, const int32_t* tix, int64_t T,
                  void* out, cudaStream_t st) {
  const unsigned grid = (unsigned)std::min<int64_t>((P->n_rows * T + 255) / 256, 148 * 32);
  auto k = layout == CTB_LAYOUT_TIME_MAJOR ? gather_rows_kernel<TIN, CTB_LAYOUT_TIME_MAJOR>
                                           : gather_rows_kernel<TIN, CTB_LAYOUT_CELL_MAJOR>;
  k<<<grid, 256, 0, st>>>((const TIN*)x, stride, P->d_row_cell, P->n_rows, tix, T, (TIN*)out);
  CTB_LAUNCH_CHECK();
  return CTB_OK;
}

}  // namespace

extern "C" int ctb_transform(const void* x0, const void* x1, int dtype, int64_t n, int transform,
                             const double* params, int n_params, int n_out, double* out, void* stream) {
  if (!x0 || (!out && n > 0) || n < 0) { ctb_set_error("ctb_transform: bad argument"); return CTB_ERR_INVALID; }
  if (dtype != CTB_F32 && dtype != CTB_F64) { ctb_set_error("dtype=%d unsupported", dtype); return CTB_ERR_INVALID; }
  CtbTr tr;
  int rc = ctb_pack_transform(transform, params, n_params, n_out, &tr);
  if (rc) return rc;
  if (ctb_tr_nin(transform) == 2 && !x1) { ctb_set_error("transform needs two inputs"); return CTB_ERR_INVALID; }
  if (n == 0) return CTB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  return ctb_dispatch_transform(transform, n_out, [&](auto kind, auto nout) {
    return dtype == CTB_F32 ? launch_tr<float, kind, nout>(x0, x1, n, tr, out, st)
                            : launch_tr<double, kind, nout>(x0, x1, n, tr, out, st);
  });
}

extern "C" int ctb_gather_rows(const ctb_plan* P, const void* x, int dtype, int layout, int64_t stride,
                               const int32_t* time_index, int64_t T, void* out, void* stream) {
  if (!P || !x || (!out && T > 0 && P->n_rows > 0) || T < 0) { ctb_set_error("ctb_gather_rows: bad argument"); return CTB_ERR_INVALID; }
  if (dtype != CTB_F32 && dtype != CTB_F64) { ctb_set_error("dtype=%d unsupported", dtype); return CTB_ERR_INVALID; }
  if (P->n_rows * T == 0) return CTB_OK;
  CtbDeviceGuard guard(P->device);
  CTB_CUDA(guard.err);
  cudaStream_t st = (cudaStream_t)stream;
  return dtype == CTB_F32 ? launch_gather<float>(P, x, layout, stride, time_index, T, out, st)
                          : launch_gather<double>(P, x, layout, stride, time_index, T, out, st);
}

// Rows of a pitched DEVICE array to a pitched HOST array on `stream` (one DMA): the time-chunked
// result copy of the host path -- out[:, :, t0:t1] of a [n_out*R][T] block -- overlaps the next chunk.
extern "C" int ctb_copy_rows_to_host(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                                     size_t width_bytes, size_t rows, void* stream) {
  if ((!dst || !src) && width_bytes * rows > 0) { ctb_set_error("ctb_copy_rows_to_host: null argument"); return CTB_ERR_INVALID; }
  if (width_bytes * rows == 0) return CTB_OK;
  CTB_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, rows, cudaMemcpyDeviceToHost,
                             (cudaStream_t)stream));
  return CTB_OK;
}

// ---------------------------------------------------------------------------
// Push a column block of a row-major [n_rows][ld] fp64 array to the same place in every peer buffer
// (multi-GPU strong scaling: each rank owns days [t0, t0 + n_cols) of the [R][T] result).  A warp
// takes a row: lane l reads columns l, l+32, ... once (up to 8 per pass, independent loads) and
// stores them to each peer -- coalesced row pieces instead of the 256-byte pieces per region and
// tile the fused epilogue scatters.
namespace {
struct PushPeers { double* p[CTB_MAX_PEERS]; };

__global__ void __launch_bounds__(256) push_rows_kernel(const double* __restrict__ src, int64_t ld, int64_t t0,
                                                         int n_cols, int64_t n_rows, int n_peers, PushPeers peers) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < n_rows; r += n_warps) {
    const int64_t base = r * ld + t0;
    for (int c0 = 0; c0 < n_cols; c0 += 256) {
      double v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c0 + k * 32 + lane;
        v[k] = c < n_cols ? __ldcs(src + base + c) : 0.0;
      }
      for (int p = 0; p < n_peers; ++p) {
        double* const dst = peers.p[p] + base;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = c0 + k * 32 + lane;
          if (c < n_cols) dst[c] = v[k];
        }
      }
    }
  }
}
}  // namespace

extern "C" int ctb_push_rows(const double* src, int64_t ld, int64_t t0, int64_t n_cols, int64_t n_rows, int n_peers,
                             double* const* peers, int engine, void* stream) {
  if (n_peers < 0 || n_peers > CTB_MAX_PEERS || ld < 0 || t0 < 0 || n_cols < 0 || n_rows < 0 || t0 + n_cols > ld ||
      n_cols >= (1ll << 31)) {
    ctb_set_error("ctb_push_rows: bad shape (ld=%lld t0=%lld n_cols=%lld n_rows=%lld n_peers=%d)", (long long)ld,
                  (long long)t0, (long long)n_cols, (long long)n_rows, n_peers);
    return CTB_ERR_INVALID;
  }
  if (n_cols == 0 || n_rows == 0 || n_peers == 0) return CTB_OK;
  if (!src || !peers) { ctb_set_error("ctb_push_rows: null argument"); return CTB_ERR_INVALID; }
  PushPeers pp{};
  int n = 0;
  for (int p = 0; p < n_peers; ++p) {
    if (!peers[p]) { ctb_set_error("ctb_push_rows: null peer pointer %d", p); return CTB_ERR_INVALID; }
    if (peers[p] != src) pp.p[n++] = peers[p];
  }
  if (n == 0) return CTB_OK;
  if (engine == CTB_PUSH_COPY_ENGINE) {
    for (int p = 0; p < n; ++p)
      CTB_CUDA(cudaMemcpy2DAsync(pp.p[p] + t0, (size_t)ld * 8, src + t0, (size_t)ld * 8, (size_t)n_cols * 8, (size_t)n_rows,
                                 cudaMemcpyDefault, (cudaStream_t)stream));
    return CTB_OK;
  }
  if (engine != CTB_PUSH_SM) { ctb_set_error("ctb_push_rows: engine %d", engine); return CTB_ERR_INVALID; }
  const unsigned grid = (unsigned)std::min<int64_t>((n_rows + 7) / 8, 148 * 8);
  push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, ld, t0, (int)n_cols, n_rows, n, pp);
  CTB_LAUNCH_CHECK();
  return CTB_OK;
}
