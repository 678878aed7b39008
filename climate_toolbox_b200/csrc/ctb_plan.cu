// K0: one-time plan build.
//
//  device part  -- exact float64 label -> gridcell index, per-row fallback weight,
//                  stable region sort, CSR row pointers, per-region denominators
//                  (replaces climate_toolbox/aggregations/aggregations.py:24-27, 64-73, 79)
//  host part    -- the planner: groups spatially adjacent regions into staging
//                  "bundles" whose gridcell footprint fits one shared-memory tile,
//                  and splits regions that are larger than a tile.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <numeric>

#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "ctb_internal.cuh"

// ------------------------------------------------------------ error state ---
static thread_local std::string g_err;
std::atomic<int64_t> g_ctb_launches{0};

void ctb_set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
}

extern "C" const char* ctb_last_error(void) { return g_err.c_str(); }
extern "C" int ctb_version(void) { return CTB_VERSION; }
extern "C" int64_t ctb_launch_count(void) { return g_ctb_launches.load(); }

// ------------------------------------------------------------- K0 kernels ---
// Exact-equality lookup of `v` in ascending `sorted[n]`; returns position in the
// ORIGINAL label order via order[], or -1.  NaN never matches; -0.0 == 0.0.
__device__ __forceinline__ int k0_find(const double* __restrict__ sorted,
                                       const int32_t* __restrict__ order, int n, double v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sorted[mid] < v) lo = mid + 1; else hi = mid;
  }
  return (lo < n && sorted[lo] == v) ? order[lo] : -1;
}

__global__ void k0_match_kernel(const double* __restrict__ slat, const int32_t* __restrict__ olat,
                                int nlat, const int32_t* __restrict__ lat_phys,
                                const double* __restrict__ slon, const int32_t* __restrict__ olon,
                                int nlon, const int32_t* __restrict__ lon_phys, int nlon_phys,
                                const double* __restrict__ row_lat,
                                const double* __restrict__ row_lon,
                                const double* __restrict__ wp, const double* __restrict__ wb,
                                int64_t n_rows, int32_t* __restrict__ row_cell,
                                double* __restrict__ row_w, unsigned long long* bad) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n_rows) return;
  const int i = k0_find(slat, olat, nlat, row_lat[k]);
  const int j = k0_find(slon, olon, nlon, row_lon[k]);
  if (i < 0 || j < 0) {
    // first offending row wins; low bit = axis (0 lat, 1 lon)
    atomicMin(bad, ((unsigned long long)k << 1) | (i < 0 ? 0ull : 1ull));
    row_cell[k] = -1;
  } else {
    const int pi = lat_phys ? lat_phys[i] : i;
    const int pj = lon_phys ? lon_phys[j] : j;
    row_cell[k] = pi * nlon_phys + pj;
  }
  const double p = wp[k];
  row_w[k] = (p > 0) ? p : wb[k];  // NaN, 0 and negatives fall back (aggregations.py:73)
}

// row_ptr[r] = first sorted position whose key >= r
__global__ void k0_rowptr_kernel(const uint32_t* __restrict__ keys, int64_t n, int32_t R,
                                 int32_t* __restrict__ row_ptr) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > R) return;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < (uint32_t)r) lo = mid + 1; else hi = mid;
  }
  row_ptr[r] = (int32_t)lo;
}

// den[r] = sum of nan->0(w) over the region's rows in stable (original) order.
__global__ void k0_den_kernel(const int32_t* __restrict__ row_ptr,
                              const int32_t* __restrict__ sorted_row,
                              const double* __restrict__ row_w, int32_t R,
                              double* __restrict__ den) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  double s = 0.0;
  for (int k = row_ptr[r]; k < row_ptr[r + 1]; ++k) {
    const double w = row_w[sorted_row[k]];
    if (w == w) s += w;
  }
  den[r] = s;
}

// ------------------------------------------------------------ host planner ---
namespace {

struct Region {
  int32_t r;
  int32_t e0, e1;  // range in kept-CSR
  uint64_t hkey;   // Hilbert index of the centroid
};

// Hilbert curve index of (x, y) in an n x n grid (n power of two).
uint64_t hilbert_xy2d(uint32_t n, uint32_t x, uint32_t y) {
  uint64_t d = 0;
  for (uint32_t s = n / 2; s > 0; s /= 2) {
    const uint32_t rx = (x & s) > 0, ry = (y & s) > 0;
    d += (uint64_t)s * s * ((3 * rx) ^ ry);
    if (ry == 0) {
      if (rx == 1) { x = n - 1 - x; y = n - 1 - y; }
      std::swap(x, y);
    }
  }
  return d;
}

// Builds the per-bundle metadata blobs (layout: CtbBlobHeader in ctb_internal.cuh).
struct BundleBuilder {
  std::vector<int64_t> b_blob_off{0};
  std::vector<int4> desc;
  std::vector<int32_t> unit_tab;   // [n_bundles][CTB_TILE_UNITS]
  std::vector<uint8_t> blob;
  int32_t max_cells = 0, max_meta = 0, n_segments = 0;
  int64_t n_pieces_total = 0;
  int64_t n_quads = 0, n_quads_conflict = 0;
  int32_t bytes_cd = 4;       // staged bytes per cell-day
  int32_t elem_bytes = 4;     // element size of the staged inputs
  int32_t tile_cap = 0;       // bytes of one staging tile
  int32_t meta_cap = 0;       // bytes of one metadata slot
  const double* den = nullptr;

  // bundle under construction
  std::vector<int32_t> cur_pieces;  // unsorted, unique
  struct Seg { int32_t target; std::vector<int32_t> cols; std::vector<double> ws; std::vector<uint32_t> gates; };
  std::vector<Seg> cur_segs;
  int32_t cur_ent_pad = 0;

  static int32_t pad(int32_t x, int32_t a) { return (x + a - 1) / a * a; }
  static int32_t part_a_bytes(int32_t n_pieces) {
    return (int32_t)sizeof(CtbBlobHeader) + pad(n_pieces * 4, 16);
  }
  static int32_t part_b_bytes(int32_t n_seg, int32_t n_ent_pad) {
    return n_seg * (int32_t)sizeof(CtbSeg) + n_ent_pad * (int32_t)sizeof(CtbEnt);
  }
  int32_t tile_bytes(int32_t n_pieces) const { return n_pieces * CTB_PIECE * CTB_S * bytes_cd; }
  bool fits_counts(int32_t n_pieces, int32_t n_seg, int32_t n_ent_pad) const {
    return tile_bytes(n_pieces) <= tile_cap && part_a_bytes(n_pieces) <= CTB_META_A_CAP &&
           n_pieces * CTB_PIECE * elem_bytes <= CTB_TILE_UNITS * 16 &&
           part_b_bytes(n_seg, n_ent_pad) <= meta_cap &&
           n_pieces * CTB_PIECE <= 65532 && n_ent_pad <= 65532 * 4;
  }
  bool fits(int32_t extra_pieces, int32_t extra_ent) const {
    return extra_ent <= 65535 &&
           fits_counts((int32_t)cur_pieces.size() + extra_pieces, (int32_t)cur_segs.size() + 1,
                       cur_ent_pad + pad(extra_ent, 4));
  }
  void add(Seg&& s) {
    cur_ent_pad += pad((int32_t)s.cols.size(), 4);
    cur_segs.push_back(std::move(s));
  }

  void close() {
    if (cur_segs.empty()) return;
    std::sort(cur_pieces.begin(), cur_pieces.end());
    // LPT order: longest segments first (warps fetch segments dynamically)
    std::stable_sort(cur_segs.begin(), cur_segs.end(),
                     [](const Seg& a, const Seg& b) { return a.cols.size() > b.cols.size(); });
    const int32_t n_seg = (int32_t)cur_segs.size();
    const int32_t n_p = (int32_t)cur_pieces.size();
    const int32_t n_ent_pad = cur_ent_pad;
    CtbBlobHeader h{};
    h.n_pieces = n_p; h.n_seg = n_seg; h.n_ent_pad = n_ent_pad;
    h.off_seg = 0;
    h.off_ent = n_seg * (int32_t)sizeof(CtbSeg);
    h.bytes_a = part_a_bytes(n_p);
    h.bytes_b = pad(h.off_ent + n_ent_pad * (int32_t)sizeof(CtbEnt), 16);
    const size_t base = blob.size();
    const size_t bytes = (size_t)h.bytes_a + h.bytes_b;
    blob.resize(base + bytes, 0);
    std::memcpy(&blob[base], &h, sizeof h);
    std::memcpy(&blob[base + sizeof h], cur_pieces.data(), (size_t)n_p * 4);
    const size_t bb = base + h.bytes_a;
    CtbSeg* segs = reinterpret_cast<CtbSeg*>(&blob[bb + h.off_seg]);
    CtbEnt* ent = reinterpret_cast<CtbEnt*>(&blob[bb + h.off_ent]);
    // staged 16-byte units of a day plane: (piece, half) -> element offset of the unit
    const int32_t halves = elem_bytes / 4, cpu = 16 / elem_bytes;
    const int32_t n_units = n_p * halves;
    desc.push_back(make_int4((int)(base & 0xffffffffu), (int)(base >> 32), (int)bytes, n_units));
    const size_t ut = unit_tab.size();
    unit_tab.resize(ut + CTB_TILE_UNITS, 0);
    for (int32_t u = 0; u < n_units; ++u)
      unit_tab[ut + u] = cur_pieces[u / halves] * CTB_PIECE + (u % halves) * cpu;
    int32_t e = 0;
    std::vector<int32_t> colq;     // staged column of every entry of the segment
    std::vector<int32_t> order;
    for (int32_t i = 0; i < n_seg; ++i) {
      const Seg& s = cur_segs[i];
      const int32_t n = (int32_t)s.cols.size();
      segs[i] = CtbSeg{s.target, (uint16_t)(e / 4), (uint16_t)n,
                       s.target >= 0 ? 1.0 / den[s.target] : 1.0};
      colq.resize(n);
      for (int32_t k = 0; k < n; ++k) {
        const int32_t piece = s.cols[k] / CTB_PIECE;
        const int32_t lp = (int32_t)(std::lower_bound(cur_pieces.begin(), cur_pieces.end(), piece) -
                                     cur_pieces.begin());
        colq[k] = lp * CTB_PIECE + s.cols[k] % CTB_PIECE;
      }
      // quads: no two entries of one residue class (column mod 4) in a quad while the classes
      // allow it.  Classes in descending size; a class spreads its entries over the quads that
      // are emptiest so far (fill levels stay within one of each other, so no quad overflows
      // before all are full); a class with more entries than quads doubles up (2-way conflict).
      const int32_t nq = (n + 3) / 4;
      std::vector<int32_t> bucket[4];
      for (int32_t k = 0; k < n; ++k) bucket[colq[k] & 3].push_back(k);
      int32_t cls[4] = {0, 1, 2, 3};
      std::stable_sort(cls, cls + 4, [&](int a, int b) { return bucket[a].size() > bucket[b].size(); });
      std::vector<std::vector<int32_t>> quad(nq);
      std::vector<int32_t> qorder(nq);
      for (int c = 0; c < 4; ++c) {
        const std::vector<int32_t>& bk = bucket[cls[c]];
        size_t next = 0;
        while (next < bk.size()) {
          // one pass: at most one entry of this class per quad, emptiest quads first
          std::iota(qorder.begin(), qorder.end(), 0);
          std::stable_sort(qorder.begin(), qorder.end(),
                           [&](int a, int b) { return quad[a].size() < quad[b].size(); });
          bool placed = false;
          for (int32_t qi = 0; qi < nq && next < bk.size(); ++qi) {
            std::vector<int32_t>& q = quad[qorder[qi]];
            // the last quad holds n - 4 (nq - 1) entries
            const size_t cap = (qorder[qi] == nq - 1) ? (size_t)(n - 4 * (nq - 1)) : 4;
            if (q.size() < cap) { q.push_back(bk[next++]); placed = true; }
          }
          if (!placed) break;   // cannot happen: total capacity == n
        }
      }
      order.clear();
      for (int32_t q = 0; q < nq; ++q) {
        std::stable_sort(quad[q].begin(), quad[q].end(), [&](int a, int b) { return (colq[a] & 3) < (colq[b] & 3); });
        bool conflict = false;
        for (size_t k = 1; k < quad[q].size(); ++k)
          conflict |= ((colq[quad[q][k]] & 3) == (colq[quad[q][k - 1]] & 3));
        for (int32_t k : quad[q]) order.push_back(k);
        ++n_quads;
        if (conflict) ++n_quads_conflict;
      }
      for (int32_t k = 0; k < n; ++k) {
        ent[e + k].w = s.ws[order[k]];
        ent[e + k].off = (uint32_t)colq[order[k]] * (uint32_t)elem_bytes;
        ent[e + k].gate = s.gates[order[k]];
      }
      // padding of the last quad: weight 0 on a copy of the quad's first entry -- the same shared
      // address (a broadcast, no bank conflict) and a value of the region's own (a NaN elsewhere in
      // the tile must not send this region to the checked loop)
      for (int32_t k = n; k < pad(n, 4); ++k) {
        ent[e + k].w = 0.0;
        ent[e + k].off = ent[e + (n & ~3)].off;
        ent[e + k].gate = ent[e + (n & ~3)].gate;
      }
      e += pad(n, 4);
    }
    b_blob_off.push_back((int64_t)blob.size());
    n_segments += n_seg;
    n_pieces_total += n_p;
    max_cells = std::max<int32_t>(max_cells, n_p * CTB_PIECE);
    max_meta = std::max<int32_t>(max_meta, h.bytes_b);
    cur_pieces.clear();
    cur_segs.clear();
    cur_ent_pad = 0;
  }
};

template <typename T>
int upload(T** dptr, const std::vector<T>& h) {
  const size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
  CTB_CUDA(cudaMalloc((void**)dptr, bytes));
  if (!h.empty()) CTB_CUDA(cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return CTB_OK;
}

}  // namespace

extern "C" void ctb_plan_free(ctb_plan* p) {
  if (!p) return;
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(p->device);
  cudaFree(p->d_row_cell); cudaFree(p->d_row_ptr); cudaFree(p->d_col); cudaFree(p->d_w); cudaFree(p->d_gate);
  cudaFree(p->d_den); cudaFree(p->d_b_blob_off); cudaFree(p->d_b_desc); cudaFree(p->d_unit_tab); cudaFree(p->d_work_counter); cudaFree(p->d_pack_src);
  cudaFree(p->d_blob); cudaFree(p->d_split_region); cudaFree(p->d_split_slot_ptr);
  cudaSetDevice(prev);
  delete p;
}

static int plan_build_impl(const double* grid_lat, int32_t nlat, const int32_t* lat_phys,
                           int32_t nlat_phys, const double* grid_lon, int32_t nlon,
                           const int32_t* lon_phys, int32_t nlon_phys, const double* row_lat,
                           const double* row_lon, const int32_t* region_code,
                           const double* w_primary, const double* w_backup, int64_t n_rows,
                           int32_t R, const ctb_plan_opts* opts, ctb_plan* P, int64_t* bad_row,
                           int32_t* bad_axis) {
  const int64_t ncell = (int64_t)nlat_phys * nlon_phys;
  if (nlat <= 0 || nlon <= 0 || n_rows < 0 || R < 0 || nlat_phys < nlat || nlon_phys < nlon ||
      ncell >= (1ll << 30) || n_rows >= (1ll << 31)) {
    ctb_set_error("ctb_plan_build: invalid sizes (nlat=%d nlon=%d n_rows=%lld R=%d)", nlat, nlon,
                  (long long)n_rows, R);
    return CTB_ERR_INVALID;
  }
  for (int64_t k = 0; k < n_rows; ++k)
    if (region_code[k] < -1 || region_code[k] >= R) {
      ctb_set_error("ctb_plan_build: region_code[%lld]=%d out of range", (long long)k,
                    region_code[k]);
      return CTB_ERR_INVALID;
    }
  P->R = R; P->n_rows = n_rows; P->ncell = ncell; P->nlat_phys = nlat_phys; P->nlon_phys = nlon_phys;

  // ---- sorted label tables (host sort of <= a few thousand labels) ----
  auto sort_labels = [](const double* lab, int n, std::vector<double>& s, std::vector<int32_t>& o) {
    o.resize(n);
    std::iota(o.begin(), o.end(), 0);
    std::stable_sort(o.begin(), o.end(), [&](int a, int b) { return lab[a] < lab[b]; });
    s.resize(n);
    for (int i = 0; i < n; ++i) s[i] = lab[o[i]];
  };
  std::vector<double> slat, slon;
  std::vector<int32_t> olat, olon;
  sort_labels(grid_lat, nlat, slat, olat);
  sort_labels(grid_lon, nlon, slon, olon);

  // ---- device K0 ----
  double *d_slat = nullptr, *d_slon = nullptr, *d_rlat = nullptr, *d_rlon = nullptr, *d_wp = nullptr,
         *d_wb = nullptr, *d_row_w = nullptr;
  int32_t *d_olat = nullptr, *d_olon = nullptr, *d_latp = nullptr, *d_lonp = nullptr;
  uint32_t *d_keys = nullptr, *d_keys_s = nullptr;
  int32_t *d_rows = nullptr, *d_rows_s = nullptr;
  unsigned long long* d_bad = nullptr;
  void* d_tmp = nullptr;
  struct Guard {
    std::vector<void**> v;
    ~Guard() { for (void** p : v) cudaFree(*p); }
  } guard;
  guard.v = {(void**)&d_slat, (void**)&d_slon, (void**)&d_rlat, (void**)&d_rlon, (void**)&d_wp,
             (void**)&d_wb, (void**)&d_row_w, (void**)&d_olat, (void**)&d_olon, (void**)&d_latp,
             (void**)&d_lonp, (void**)&d_keys, (void**)&d_keys_s, (void**)&d_rows,
             (void**)&d_rows_s, (void**)&d_bad, &d_tmp};

  const size_t nr = (size_t)std::max<int64_t>(n_rows, 1);
  CTB_CUDA(cudaMalloc(&d_slat, nlat * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_slon, nlon * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_olat, nlat * sizeof(int32_t)));
  CTB_CUDA(cudaMalloc(&d_olon, nlon * sizeof(int32_t)));
  CTB_CUDA(cudaMemcpy(d_slat, slat.data(), nlat * sizeof(double), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_slon, slon.data(), nlon * sizeof(double), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_olat, olat.data(), nlat * sizeof(int32_t), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_olon, olon.data(), nlon * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (lat_phys) {
    CTB_CUDA(cudaMalloc(&d_latp, nlat * sizeof(int32_t)));
    CTB_CUDA(cudaMemcpy(d_latp, lat_phys, nlat * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  if (lon_phys) {
    CTB_CUDA(cudaMalloc(&d_lonp, nlon * sizeof(int32_t)));
    CTB_CUDA(cudaMemcpy(d_lonp, lon_phys, nlon * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  CTB_CUDA(cudaMalloc(&d_rlat, nr * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_rlon, nr * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_wp, nr * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_wb, nr * sizeof(double)));
  CTB_CUDA(cudaMalloc(&d_row_w, nr * sizeof(double)));
  CTB_CUDA(cudaMalloc(&P->d_row_cell, nr * sizeof(int32_t)));
  CTB_CUDA(cudaMalloc(&d_bad, sizeof(unsigned long long)));
  CTB_CUDA(cudaMemset(d_bad, 0xff, sizeof(unsigned long long)));
  CTB_CUDA(cudaMemcpy(d_rlat, row_lat, n_rows * sizeof(double), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_rlon, row_lon, n_rows * sizeof(double), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_wp, w_primary, n_rows * sizeof(double), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_wb, w_backup, n_rows * sizeof(double), cudaMemcpyHostToDevice));

  if (n_rows > 0) {
    k0_match_kernel<<<(unsigned)((n_rows + 255) / 256), 256>>>(
        d_slat, d_olat, nlat, d_latp, d_slon, d_olon, nlon, d_lonp, nlon_phys, d_rlat, d_rlon, d_wp,
        d_wb, n_rows, P->d_row_cell, d_row_w, d_bad);
    CTB_LAUNCH_CHECK();
  }
  unsigned long long bad = ~0ull;
  CTB_CUDA(cudaMemcpy(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost));
  if (bad != ~0ull) {
    if (bad_row) *bad_row = (int64_t)(bad >> 1);
    if (bad_axis) *bad_axis = (int32_t)(bad & 1);
    ctb_set_error("not all values found in index '%s' (weights row %lld)", (bad & 1) ? "lon" : "lat",
                  (long long)(bad >> 1));
    return CTB_ERR_LABEL_NOT_FOUND;
  }

  // stable sort of rows by region code (code -1 -> 0xffffffff sorts last)
  std::vector<uint32_t> h_keys(nr);
  for (int64_t k = 0; k < n_rows; ++k) h_keys[k] = (uint32_t)region_code[k];
  std::vector<int32_t> h_iota(nr);
  std::iota(h_iota.begin(), h_iota.end(), 0);
  CTB_CUDA(cudaMalloc(&d_keys, nr * sizeof(uint32_t)));
  CTB_CUDA(cudaMalloc(&d_keys_s, nr * sizeof(uint32_t)));
  CTB_CUDA(cudaMalloc(&d_rows, nr * sizeof(int32_t)));
  CTB_CUDA(cudaMalloc(&d_rows_s, nr * sizeof(int32_t)));
  CTB_CUDA(cudaMemcpy(d_keys, h_keys.data(), n_rows * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CTB_CUDA(cudaMemcpy(d_rows, h_iota.data(), n_rows * sizeof(int32_t), cudaMemcpyHostToDevice));
  if (n_rows > 0) {
    size_t tmp_bytes = 0;
    CTB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys_s, d_rows, d_rows_s,
                                             (int)n_rows));
    CTB_CUDA(cudaMalloc(&d_tmp, tmp_bytes));
    CTB_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys_s, d_rows, d_rows_s,
                                             (int)n_rows));
    g_ctb_launches.fetch_add(1);
  }
  int32_t* d_rp_all = nullptr;  // row pointers over ALL rows with a valid region
  CTB_CUDA(cudaMalloc(&d_rp_all, (R + 1) * sizeof(int32_t)));
  guard.v.push_back((void**)&d_rp_all);
  k0_rowptr_kernel<<<(R + 1 + 255) / 256, 256>>>(d_keys_s, n_rows, R, d_rp_all);
  CTB_LAUNCH_CHECK();
  CTB_CUDA(cudaMalloc(&P->d_den, std::max(R, 1) * sizeof(double)));
  if (R > 0) {
    k0_den_kernel<<<(R + 255) / 256, 256>>>(d_rp_all, d_rows_s, d_row_w, R, P->d_den);
    CTB_LAUNCH_CHECK();
  }

  // ---- bring the sorted structure to the host planner ----
  std::vector<int32_t> rp_all(R + 1), rows_s(nr);
  P->h_row_cell.resize(n_rows);
  P->h_row_w.resize(n_rows);
  P->h_den.resize(R);
  CTB_CUDA(cudaMemcpy(rp_all.data(), d_rp_all, (R + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CTB_CUDA(cudaMemcpy(rows_s.data(), d_rows_s, n_rows * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CTB_CUDA(cudaMemcpy(P->h_row_cell.data(), P->d_row_cell, n_rows * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CTB_CUDA(cudaMemcpy(P->h_row_w.data(), d_row_w, n_rows * sizeof(double), cudaMemcpyDeviceToHost));
  CTB_CUDA(cudaMemcpy(P->h_den.data(), P->d_den, R * sizeof(double), cudaMemcpyDeviceToHost));

  // kept CSR: drop rows whose weight is NaN or 0 -- they add nothing to the
  // numerator (NaN product is skipped; 0*x is 0 or NaN) and are already in den.
  std::vector<int32_t> row_ptr(R + 1, 0), col;
  std::vector<double> w;
  std::vector<uint32_t> gate;     // growing-season gate of every kept row's PHYSICAL gridcell
  const uint32_t* cell_gate = opts ? opts->cell_gate : nullptr;
  P->has_gate = cell_gate ? 1 : 0;
  col.reserve(n_rows);
  w.reserve(n_rows);
  gate.reserve(n_rows);
  int32_t max_rows = 0;
  for (int32_t r = 0; r < R; ++r) {
    for (int32_t k = rp_all[r]; k < rp_all[r + 1]; ++k) {
      const int32_t row = rows_s[k];
      const double ww = P->h_row_w[row];
      if (ww == ww && ww != 0.0) {
        col.push_back(P->h_row_cell[row]);
        w.push_back(ww);
        gate.push_back(cell_gate ? cell_gate[P->h_row_cell[row]] : CTB_GATE_ALWAYS);
      }
    }
    row_ptr[r + 1] = (int32_t)col.size();
    max_rows = std::max(max_rows, row_ptr[r + 1] - row_ptr[r]);
  }
  P->nnz = (int64_t)col.size();

  // region centroids (physical grid coordinates) order the regions along a Hilbert curve
  std::vector<double> cen_i(R, 0.0), cen_j(R, 0.0);
  for (int32_t r = 0; r < R; ++r) {
    for (int32_t k = row_ptr[r]; k < row_ptr[r + 1]; ++k) {
      cen_i[r] += col[k] / nlon_phys;
      cen_j[r] += col[k] % nlon_phys;
    }
    const int32_t n = row_ptr[r + 1] - row_ptr[r];
    if (n) { cen_i[r] /= n; cen_j[r] /= n; }
  }

  // ---- compact plans: renumber the referenced 4-cell pieces densely ----
  int64_t plan_ncell = ncell;
  P->compact = opts && opts->compact ? 1 : 0;
  if (P->compact) {
    std::vector<int32_t> cp;
    cp.reserve(col.size());
    for (int32_t c : col) cp.push_back(c / CTB_PIECE);
    std::sort(cp.begin(), cp.end());
    cp.erase(std::unique(cp.begin(), cp.end()), cp.end());
    // every run of consecutive pieces starts on a 64-byte boundary of the packed plane (4 pieces
    // of f32), so that ctb_host_pack can write whole cache lines with streaming stores
    std::vector<int32_t> packed_of(cp.size());
    int32_t cur = 0;
    for (size_t q = 0; q < cp.size();) {
      size_t e = q + 1;
      while (e < cp.size() && cp[e] == cp[e - 1] + 1) ++e;
      cur = (cur + 3) & ~3;
      P->h_pack_runs.push_back({cp[q], (int32_t)(e - q), cur});
      for (size_t k = q; k < e; ++k) packed_of[k] = cur + (int32_t)(k - q);
      cur += (int32_t)(e - q);
      q = e;
    }
    cur = (cur + 3) & ~3;
    for (auto& c : col) {
      const size_t k = (size_t)(std::lower_bound(cp.begin(), cp.end(), c / CTB_PIECE) - cp.begin());
      c = packed_of[k] * CTB_PIECE + c % CTB_PIECE;
    }
    plan_ncell = (int64_t)cur * CTB_PIECE;
    P->ncell = plan_ncell;   // what the kernels index
    // device copy for ctb_pull_pack: source piece of every packed piece
    std::vector<int32_t> pack_src((size_t)cur, -1);
    for (const auto& r : P->h_pack_runs)
      for (int32_t k = 0; k < r.n_pieces; ++k) pack_src[(size_t)r.packed_piece + k] = r.phys_piece + k;
    if (int rc_ = upload(&P->d_pack_src, pack_src)) return rc_;
  }

  // ---- staging bundles ----
  int32_t bytes_cd = opts && opts->stage_bytes_per_cell_day > 0 ? opts->stage_bytes_per_cell_day : 4;
  // shared memory of one CTA = CTB_TILE_STAGES tiles + CTB_META_SLOTS metadata slots; a
  // tile holds at most CTB_TILE_UNITS 16-byte units per day (register budget of the loads
  // in flight).  smem_budget_bytes (tests) shrinks the tile to force region splitting.
  const int32_t meta_cap = CTB_META_B_CAP;
  int32_t tile_cap = CTB_TILE_BYTES;
  if (opts && opts->smem_budget_bytes > 0) tile_cap = std::min(tile_cap, opts->smem_budget_bytes);
  BundleBuilder B;
  B.bytes_cd = bytes_cd;
  B.elem_bytes = opts && opts->elem_bytes == 8 ? 8 : 4;
  P->elem_bytes = B.elem_bytes;
  P->stage_bytes = bytes_cd;
  B.tile_cap = tile_cap;
  B.meta_cap = meta_cap;
  B.den = P->h_den.data();
  if (!B.fits_counts(2, 1, 8)) {
    ctb_set_error("ctb_plan_build: smem budget %d too small", tile_cap);
    return CTB_ERR_INVALID;
  }

  uint32_t hn = 1;
  while ((int32_t)hn < std::max(nlat_phys, nlon_phys)) hn <<= 1;
  std::vector<Region> regs;
  std::vector<int32_t> empty_regions;
  regs.reserve(R);
  for (int32_t r = 0; r < R; ++r) {
    if (row_ptr[r + 1] == row_ptr[r]) {
      // no kept rows: out = 0 / den (NaN when den == 0), written by the fix-up kernel
      // as a "split" region with an empty slot range
      empty_regions.push_back(r);
      continue;
    }
    regs.push_back({r, row_ptr[r], row_ptr[r + 1],
                    hilbert_xy2d(hn, (uint32_t)cen_j[r], (uint32_t)cen_i[r])});
  }
  std::stable_sort(regs.begin(), regs.end(),
                   [](const Region& a, const Region& b) { return a.hkey < b.hkey; });
  // the bundle sequence as a region permutation (regions without kept rows last): rows written in this
  // order keep the stores of one CTA inside a few pages (the fused peer-memory gather needs that)
  P->h_region_pos.assign(R, 0);
  {
    int32_t pos = 0;
    for (const Region& g : regs) P->h_region_pos[g.r] = pos++;
    for (int32_t r : empty_regions) P->h_region_pos[r] = pos++;
  }

  const int64_t npiece_grid = (plan_ncell + CTB_PIECE - 1) / CTB_PIECE;
  std::vector<int32_t> stamp(npiece_grid, -1);   // piece -> bundle generation that holds it
  std::vector<uint8_t> seen(npiece_grid, 0);     // piece referenced at all
  std::vector<uint8_t> cell_seen(plan_ncell, 0);
  int32_t gen = 0;
  std::vector<int32_t> split_region, split_slot_ptr{0};
  int32_t n_scratch = 0;
  std::vector<int32_t> newp;

  auto add_segment = [&](int32_t target, const int32_t* cols, const double* ws, const uint32_t* gs, int32_t n) {
    BundleBuilder::Seg s;
    s.target = target;
    s.cols.assign(cols, cols + n);
    s.ws.assign(ws, ws + n);
    s.gates.assign(gs, gs + n);
    for (int32_t k = 0; k < n; ++k) {
      const int32_t p = cols[k] / CTB_PIECE;
      if (stamp[p] != gen) { stamp[p] = gen; B.cur_pieces.push_back(p); }
    }
    B.add(std::move(s));
  };

  for (const Region& g : regs) {
    const int32_t n = g.e1 - g.e0;
    // distinct new pieces this region would add to the open bundle
    newp.clear();
    for (int32_t k = g.e0; k < g.e1; ++k) {
      const int32_t p = col[k] / CTB_PIECE;
      if (stamp[p] != gen) newp.push_back(p);
    }
    std::sort(newp.begin(), newp.end());
    newp.erase(std::unique(newp.begin(), newp.end()), newp.end());
    if (B.fits((int32_t)newp.size(), n)) {
      add_segment(g.r, &col[g.e0], &w[g.e0], &gate[g.e0], n);
      continue;
    }
    // does it fit an empty bundle?
    std::vector<int32_t> own;
    own.reserve(n);
    for (int32_t k = g.e0; k < g.e1; ++k) own.push_back(col[k] / CTB_PIECE);
    std::sort(own.begin(), own.end());
    own.erase(std::unique(own.begin(), own.end()), own.end());
    B.close();
    ++gen;
    if (B.fits((int32_t)own.size(), n)) {
      add_segment(g.r, &col[g.e0], &w[g.e0], &gate[g.e0], n);
      continue;
    }
    // split: order the region's rows by cell, cut into fragments that fit one tile
    std::vector<int32_t> idx(n);
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(),
                     [&](int a, int b) { return col[g.e0 + a] < col[g.e0 + b]; });
    std::vector<int32_t> fc;
    std::vector<double> fw;
    std::vector<uint32_t> fg;
    int32_t fpieces = 0, last_piece = -1;
    split_region.push_back(g.r);
    auto flush = [&]() {
      if (fc.empty()) return;
      add_segment(~n_scratch, fc.data(), fw.data(), fg.data(), (int32_t)fc.size());
      ++n_scratch;
      B.close();
      ++gen;
      fc.clear(); fw.clear(); fg.clear(); fpieces = 0; last_piece = -1;
    };
    for (int32_t q = 0; q < n; ++q) {
      const int32_t c = col[g.e0 + idx[q]];
      const int32_t p = c / CTB_PIECE;
      const int32_t np = fpieces + (p != last_piece ? 1 : 0);
      if (!fc.empty() && ((int32_t)fc.size() >= 65535 ||
                          !B.fits_counts(np, 1, BundleBuilder::pad((int32_t)fc.size() + 1, 4))))
        flush();
      if (p != last_piece) { ++fpieces; last_piece = p; }
      fc.push_back(c);
      fw.push_back(w[g.e0 + idx[q]]);
      fg.push_back(gate[g.e0 + idx[q]]);
    }
    flush();
    split_slot_ptr.push_back(n_scratch);
  }
  B.close();
  for (int32_t r : empty_regions) {
    split_region.push_back(r);
    split_slot_ptr.push_back(n_scratch);
  }

  int64_t U = 0, pieces_distinct = 0;
  for (int64_t k = 0; k < P->nnz; ++k) {
    if (!cell_seen[col[k]]) { cell_seen[col[k]] = 1; ++U; }
    if (!seen[col[k] / CTB_PIECE]) { seen[col[k] / CTB_PIECE] = 1; ++pieces_distinct; }
  }

  // ---- upload ----
  int rc;
  if ((rc = upload(&P->d_row_ptr, row_ptr))) return rc;
  if ((rc = upload(&P->d_col, col))) return rc;
  if ((rc = upload(&P->d_w, w))) return rc;
  if ((rc = upload(&P->d_gate, gate))) return rc;
  if ((rc = upload(&P->d_b_blob_off, B.b_blob_off))) return rc;
  if ((rc = upload(&P->d_blob, B.blob))) return rc;
  if ((rc = upload(&P->d_b_desc, B.desc))) return rc;
  if ((rc = upload(&P->d_unit_tab, B.unit_tab))) return rc;
  // {next unit, CTAs done} pairs of the streaming kernel: zero between launches (self re-arming)
  CTB_CUDA(cudaMalloc((void**)&P->d_work_counter, CTB_N_WORK_COUNTERS * sizeof(int)));
  CTB_CUDA(cudaMemset(P->d_work_counter, 0, CTB_N_WORK_COUNTERS * sizeof(int)));
  if ((rc = upload(&P->d_split_region, split_region))) return rc;
  if ((rc = upload(&P->d_split_slot_ptr, split_slot_ptr))) return rc;
  P->n_bundles = (int32_t)B.b_blob_off.size() - 1;
  P->n_segments = B.n_segments;
  P->n_split = (int32_t)split_region.size();
  P->n_scratch = n_scratch;

  ctb_plan_info& I = P->info;
  I.n_rows = n_rows; I.nnz = P->nnz; I.n_cells_distinct = U; I.n_cells_grid = ncell;
  I.n_regions = R; I.n_bundles = P->n_bundles; I.n_pieces = B.n_pieces_total;
  I.n_pieces_distinct = pieces_distinct; I.n_split_regions = P->n_split;
  I.n_scratch_slots = n_scratch; I.cap_cells = tile_cap / (CTB_S * bytes_cd); I.max_bundle_cells = B.max_cells;
  I.max_meta_bytes = B.max_meta;
  I.n_packed_cells = P->compact ? (int32_t)plan_ncell : 0;
  I.time_block = CTB_TB; I.max_region_rows = max_rows;
  I.n_quads = B.n_quads; I.n_quads_conflict = B.n_quads_conflict;
  CTB_CUDA(cudaDeviceSynchronize());
  return CTB_OK;
}

extern "C" int ctb_plan_build(const double* grid_lat, int32_t nlat, const int32_t* lat_phys,
                              int32_t nlat_phys, const double* grid_lon, int32_t nlon,
                              const int32_t* lon_phys, int32_t nlon_phys, const double* row_lat,
                              const double* row_lon, const int32_t* region_code,
                              const double* w_primary, const double* w_backup, int64_t n_rows,
                              int32_t n_regions, const ctb_plan_opts* opts, int device,
                              ctb_plan** out, int64_t* bad_row, int32_t* bad_axis) {
  if (!out || !grid_lat || !grid_lon || (n_rows > 0 && (!row_lat || !row_lon || !region_code ||
                                                        !w_primary || !w_backup))) {
    ctb_set_error("ctb_plan_build: null argument");
    return CTB_ERR_INVALID;
  }
  *out = nullptr;
  int prev = 0;
  CTB_CUDA(cudaGetDevice(&prev));
  CTB_CUDA(cudaSetDevice(device));
  ctb_plan* P = new ctb_plan();
  P->device = device;
  const int rc = plan_build_impl(grid_lat, nlat, lat_phys, nlat_phys, grid_lon, nlon, lon_phys,
                                 nlon_phys, row_lat, row_lon, region_code, w_primary, w_backup,
                                 n_rows, n_regions, opts, P, bad_row, bad_axis);
  cudaSetDevice(prev);
  if (rc != CTB_OK) {
    ctb_plan_free(P);
    return rc;
  }
  *out = P;
  return CTB_OK;
}

extern "C" int ctb_plan_get_info(const ctb_plan* plan, ctb_plan_info* info) {
  if (!plan || !info) { ctb_set_error("null argument"); return CTB_ERR_INVALID; }
  *info = plan->info;
  return CTB_OK;
}

extern "C" int ctb_plan_row_cells(const ctb_plan* plan, int32_t* out) {
  if (!plan || !out) { ctb_set_error("null argument"); return CTB_ERR_INVALID; }
  std::memcpy(out, plan->h_row_cell.data(), plan->h_row_cell.size() * sizeof(int32_t));
  return CTB_OK;
}

extern "C" int ctb_plan_den(const ctb_plan* plan, double* out) {
  if (!plan || !out) { ctb_set_error("null argument"); return CTB_ERR_INVALID; }
  std::memcpy(out, plan->h_den.data(), plan->h_den.size() * sizeof(double));
  return CTB_OK;
}

extern "C" int ctb_plan_region_order(const ctb_plan* plan, int32_t* out) {
  if (!plan || !out) { ctb_set_error("null argument"); return CTB_ERR_INVALID; }
  std::memcpy(out, plan->h_region_pos.data(), plan->h_region_pos.size() * sizeof(int32_t));
  return CTB_OK;
}

extern "C" int ctb_plan_row_weights(const ctb_plan* plan, double* out) {
  if (!plan || !out) { ctb_set_error("null argument"); return CTB_ERR_INVALID; }
  std::memcpy(out, plan->h_row_w.data(), plan->h_row_w.size() * sizeof(double));
  return CTB_OK;
}

// ---------------------------------------------------------------- host ingest ---
#include <atomic>
#include <thread>

extern "C" int ctb_host_pack(const ctb_plan* P, const void* x, int dtype, int64_t stride,
                             const int64_t* time_index, int64_t t_begin, int64_t T, void* dst,
                             int n_threads) {
  if (!P || !x || (!dst && T > 0) || T < 0 || !P->compact) {
    ctb_set_error("ctb_host_pack: needs a compact plan and non-null buffers");
    return CTB_ERR_INVALID;
  }
  if (dtype != CTB_F32 && dtype != CTB_F64) { ctb_set_error("dtype=%d unsupported", dtype); return CTB_ERR_INVALID; }
  const size_t es = dtype == CTB_F32 ? 4 : 8;
  const size_t piece_bytes = CTB_PIECE * es;
  const int64_t packed = P->ncell;   // cells per packed plane
  if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  n_threads = (int)std::min<int64_t>(n_threads, std::max<int64_t>(T, 1));
  const char* src = static_cast<const char*>(x);
  char* out = static_cast<char*>(dst);
  const bool nt = (reinterpret_cast<uintptr_t>(dst) & 63) == 0 && ((size_t)packed * es) % 64 == 0;
  // the last piece of a grid whose cell count is not a multiple of 4 ends past the plane: copy
  // what exists, zero-fill the rest (never read past the caller's buffer)
  const size_t plane_bytes = (size_t)P->nlat_phys * (size_t)P->nlon_phys * es;
  auto work = [&](int64_t d0, int64_t d1) {
    for (int64_t d = d0; d < d1; ++d) {
      const int64_t tp = time_index ? time_index[t_begin + d] : t_begin + d;
      const char* plane = src + (size_t)tp * stride * es;
      char* o = out + (size_t)d * packed * es;
      for (const auto& r : P->h_pack_runs) {
        char* q = o + (size_t)r.packed_piece * piece_bytes;
        const size_t s_off = (size_t)r.phys_piece * piece_bytes;
        const char* s = plane + s_off;
        const size_t n = (size_t)r.n_pieces * piece_bytes;
        if (s_off + n > plane_bytes) {   // ragged tail of the plane (at most one run per day)
          const size_t have = plane_bytes > s_off ? plane_bytes - s_off : 0;
          std::memcpy(q, s, have);
          std::memset(q + have, 0, n - have);
          if (nt) std::memset(q + n, 0, (64 - (n & 63)) & 63);
          continue;
        }
#if defined(__SSE2__)
        if (nt) {
          // runs start on 64-byte boundaries of the packed plane: write whole lines (the run, then
          // zeros up to the next boundary) with streaming stores -- no read-for-ownership of the
          // destination, which only the DMA engine will read
          size_t i = 0;
          for (; i < n; i += 16)
            _mm_stream_si128(reinterpret_cast<__m128i*>(q + i),
                             _mm_loadu_si128(reinterpret_cast<const __m128i*>(s + i)));
          for (; i & 63; i += 16) _mm_stream_si128(reinterpret_cast<__m128i*>(q + i), _mm_setzero_si128());
          continue;
        }
#endif
        std::memcpy(q, s, n);
      }
    }
#if defined(__SSE2__)
    if (nt) _mm_sfence();
#endif
  };
  if (n_threads == 1) { work(0, T); return CTB_OK; }
  // days are handed out one at a time: on a shared host a preempted core delays one day, not a
  // whole static share of the chunk
  std::atomic<int64_t> next{0};
  auto loop = [&]() {
    for (int64_t d; (d = next.fetch_add(1, std::memory_order_relaxed)) < T;) work(d, d + 1);
  };
  std::vector<std::thread> pool;
  for (int i = 1; i < n_threads; ++i) pool.emplace_back(loop);
  loop();   // the calling thread packs too
  for (auto& th : pool) th.join();
  return CTB_OK;
}


// ---------------------------------------------------------------- device ingest ---
// The same packing done by the GPU: the referenced 16-byte pieces of T day planes are read straight
// from a host array in pinned (device-accessible) memory over PCIe and written to a packed device
// buffer dst[T][n_packed_cells].  Only the referenced gridcells cross the bus and no host core
// touches the data -- what the ranks of a multi-GPU job need when they share the host's cores.
// Thread = one packed piece x 4 consecutive days (4 independent 16-byte loads in flight per
// thread); reads are contiguous along a run of referenced pieces, writes are fully coalesced.
#ifndef CTB_PULL_L2_HINT
#define CTB_PULL_L2_HINT ""      // experiments: ".L2::64B" / ".L2::256B" fetch-size hints (profiles/micro/r2_e2e_ingest.log)
#endif
namespace {
__global__ void __launch_bounds__(256) pull_pack_kernel(const uint4* __restrict__ src, int64_t stride16,
                                                        const int32_t* __restrict__ tix, int64_t t_begin, int T,
                                                        const int32_t* __restrict__ pack_src, int n_units,
                                                        int halves, uint4* __restrict__ dst) {
  const int64_t n_work = (int64_t)n_units * ((T + 3) / 4);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_work; i += (int64_t)gridDim.x * blockDim.x) {
    const int u = (int)(i % n_units);
    const int d0 = (int)(i / n_units) * 4;
    const int p = __ldg(pack_src + u / halves);
    if (p < 0) continue;                       // alignment padding of the packed plane: never read
    const int64_t so = (int64_t)p * halves + (u % halves);
    uint4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (d0 + k < T) {
        const int64_t tp = tix ? tix[t_begin + d0 + k] : t_begin + d0 + k;
        asm volatile("ld.global.nc.L1::no_allocate" CTB_PULL_L2_HINT ".v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(v[k].x), "=r"(v[k].y), "=r"(v[k].z), "=r"(v[k].w) : "l"(src + tp * stride16 + so));
      }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (d0 + k < T) dst[(int64_t)(d0 + k) * n_units + u] = v[k];
  }
}

// The launch shape of the pull kernels: one thread per unit of a packed plane and work row.  A unit is 16 bytes
// of a float source; of an int16 source it is one 4-cell piece, 8 bytes.
struct PullShape {
  int64_t es;        // bytes per source element
  int64_t stride16;  // the source's plane stride in units (16 bytes; 8 for int16)
  int halves;        // units per 4-cell piece
  int n_units;       // units per packed plane
  unsigned grid;
};

// Bytes per element of a float dtype, 0 for any other value
int64_t float_bytes(int dtype) { return dtype == CTB_F32 ? 4 : dtype == CTB_F64 ? 8 : 0; }

// The checks the pull entry points share, in this order: a compact plan, a source, 0 <= n_days < 2^31 and
// t_begin >= 0, a source element size es of 2, 4 or 8 (0: `dtype` is no float dtype), and source planes aligned
// to one unit on a grid of whole 4-cell pieces (a ragged last piece would be read past the plane).  Each entry
// checks its destinations itself.
int pull_check(const char* fn, const ctb_plan* P, const void* x, int dtype, int64_t es, int64_t stride,
               int64_t t_begin, int64_t n_days, int64_t rows, PullShape* sh) {
  if (!P || !P->compact) { ctb_set_error("%s: needs a compact plan", fn); return CTB_ERR_INVALID; }
  if (!x) { ctb_set_error("%s: the source is null", fn); return CTB_ERR_INVALID; }
  if (n_days < 0 || n_days >= (1ll << 31) || t_begin < 0) {
    ctb_set_error("%s: needs 0 <= T < 2^31 and t_begin >= 0, got T=%lld, t_begin=%lld", fn, (long long)n_days,
                  (long long)t_begin);
    return CTB_ERR_INVALID;
  }
  if (es == 0) {
    ctb_set_error("%s: dtype=%d unsupported", fn, dtype);
    return CTB_ERR_INVALID;
  }
  sh->es = es;
  const int64_t unit = es == 2 ? 8 : 16;
  if ((stride * sh->es) % unit != 0 || (uintptr_t)x % unit != 0 ||
      (int64_t)P->nlat_phys * P->nlon_phys % CTB_PIECE != 0) {
    ctb_set_error("%s: planes must be %d-byte aligned and hold a multiple of 4 gridcells", fn, (int)unit);
    return CTB_ERR_UNSUPPORTED;
  }
  sh->stride16 = stride * sh->es / unit;
  sh->halves = es == 2 ? 1 : (int)(sh->es / 4);
  sh->n_units = (int)(P->ncell / CTB_PIECE) * sh->halves;
  sh->grid = (unsigned)std::min<int64_t>(((int64_t)sh->n_units * rows + 255) / 256, 148 * 32);
  return CTB_OK;
}

// launch() enqueues the kernel on the plan's device; nothing is launched for zero days
template <typename F>
int pull_launch(const ctb_plan* P, int64_t n_days, F&& launch) {
  if (n_days == 0) return CTB_OK;
  CtbDeviceGuard guard(P->device);
  if (guard.err != cudaSuccess) { ctb_set_error("cudaSetDevice(%d) failed: %s", P->device, cudaGetErrorString(guard.err)); return CTB_ERR_CUDA; }
  if (int rc = launch()) return rc;
  CTB_LAUNCH_CHECK();
  return CTB_OK;
}
}  // namespace

extern "C" int ctb_pull_pack(const ctb_plan* P, const void* x, int dtype, int64_t stride,
                             const int32_t* time_index, int64_t t_begin, int64_t T, void* dst, void* stream) {
  PullShape sh;
  if (int rc = pull_check("ctb_pull_pack", P, x, dtype, float_bytes(dtype), stride, t_begin, T, (T + 3) / 4, &sh)) return rc;
  if (!dst && T > 0) { ctb_set_error("ctb_pull_pack: dst is null"); return CTB_ERR_INVALID; }
  return pull_launch(P, T, [&] {
    pull_pack_kernel<<<sh.grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint4*>(x), sh.stride16, time_index, t_begin, (int)T, P->d_pack_src, sh.n_units,
        sh.halves, static_cast<uint4*>(dst));
    return CTB_OK;
  });
}

// ---------------------------------------------------------------- sub-daily ingest ---
// Packing and the daily reduction in one read: day d of the packed planes reduces the steps
// s = day[t_begin + d] * S + h, h = 0..S-1, of a TIME_MAJOR source in device or pinned host memory.
// Mean: every step widened to fp64 and added in step order (plain adds), NaN steps skipped, the sum
// divided by the count (0/0: NaN for a day without values).  Min / max: NaN steps skipped, exact, in
// the source dtype; both come from the same loads.  Thread = one 16-byte unit of a packed piece x one
// day with 8 step loads in flight; a warp's loads are contiguous along a run of referenced pieces.
namespace {
__device__ __forceinline__ float ext_min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float ext_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double ext_min(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ double ext_max(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ void unit_get(const uint4& v, float (&e)[4]) {
  e[0] = __uint_as_float(v.x); e[1] = __uint_as_float(v.y); e[2] = __uint_as_float(v.z); e[3] = __uint_as_float(v.w);
}
__device__ __forceinline__ void unit_get(const uint4& v, double (&e)[2]) {
  e[0] = __hiloint2double((int)v.y, (int)v.x); e[1] = __hiloint2double((int)v.w, (int)v.z);
}
__device__ __forceinline__ uint4 unit_put(const float (&e)[4]) {
  return make_uint4(__float_as_uint(e[0]), __float_as_uint(e[1]), __float_as_uint(e[2]), __float_as_uint(e[3]));
}
__device__ __forceinline__ uint4 unit_put(const double (&e)[2]) {
  return make_uint4((unsigned)__double2loint(e[0]), (unsigned)__double2hiint(e[0]), (unsigned)__double2loint(e[1]),
                    (unsigned)__double2hiint(e[1]));
}

// Sources of the step loop: how one unit of a source piece is loaded and unpacked into C elements of type E.
// A float source: a unit is 16 bytes, C = 16 / sizeof(T) elements as stored.
template <typename T>
struct FloatSrc {
  using E = T;
  using V = uint4;
  static constexpr int C = 16 / sizeof(T);
  __device__ __forceinline__ void load(V& v, const V* p) const {
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  }
  __device__ __forceinline__ void get(const V& v, T (&e)[C]) const { unit_get(v, e); }
};

__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

// A CF-packed int16 source (netCDF short): a unit is one 4-cell piece, 8 bytes.  Raw value r decodes to NaN when
// it is a fill value, else to fl(fl(D(r) * scale) + offset) in D: two rounded operations, no contraction, which
// is numpy's r.astype(D) * D(scale) + D(offset) bit for bit.
template <typename D>
struct PackedI16Src {
  using E = D;
  using V = uint2;
  static constexpr int C = 4;
  D scale, offset;
  int fill[4];   // raw fill values; unused slots hold 0x10000, which no int16 equals
  __device__ __forceinline__ void load(V& v, const V* p) const {
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  }
  __device__ __forceinline__ void get(const V& v, D (&e)[4]) const {
    const int r[4] = {(int)(short)(v.x & 0xffff), (int)(short)(v.x >> 16), (int)(short)(v.y & 0xffff),
                      (int)(short)(v.y >> 16)};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const bool masked = r[c] == fill[0] || r[c] == fill[1] || r[c] == fill[2] || r[c] == fill[3];
      e[c] = masked ? (D)NAN : add_rn(mul_rn((D)r[c], scale), offset);
    }
  }
};

// The step loop of the sub-daily kernels.  Item = one unit u of a packed plane x one day d: step(e) gets the
// Src::C elements of each of the day's S steps, in step order, then item(d, u) stores the item's results and
// resets the kernel's accumulators for the next item.  Padding units call neither.  stride16 is the source's
// plane stride in units.
template <typename Src, typename Step, typename Item>
__device__ __forceinline__ void subdaily_step_loop(const Src& sp, const typename Src::V* src, int64_t stride16, int S,
                                                   const int32_t* day, int64_t t_begin, int n_days,
                                                   const int32_t* pack_src, int n_units, int halves, Step&& step,
                                                   Item&& item) {
  using T = typename Src::E;
  constexpr int C = Src::C;           // cells per unit
  constexpr int U = 8;                // step loads in flight
  const int64_t n_work = (int64_t)n_units * n_days;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_work; i += (int64_t)gridDim.x * blockDim.x) {
    const int u = (int)(i % n_units);
    const int d = (int)(i / n_units);
    const int p = __ldg(pack_src + u / halves);
    if (p < 0) continue;                       // alignment padding of the packed plane: never read
    const int64_t step0 = (int64_t)(day ? __ldg(day + t_begin + d) : t_begin + d) * S;
    const typename Src::V* s = src + step0 * stride16 + (int64_t)p * halves + (u % halves);
    for (int h0 = 0; h0 < S; h0 += U) {
      typename Src::V v[U];
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (h0 + k < S) sp.load(v[k], s + (int64_t)(h0 + k) * stride16);
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (h0 + k < S) {
          T e[C];
          sp.get(v[k], e);
          step(e);
        }
    }
    item(d, u);
  }
}

// Stores the C elements of one item to a plane of T at item index i: one 16-byte unit, or two (4 float64 cells)
template <typename T, int C>
__device__ __forceinline__ void item_put(uint4* dst, int64_t i, const T (&e)[C]) {
  if constexpr (C * sizeof(T) == 16) {
    dst[i] = unit_put(e);
  } else {
    dst[2 * i] = unit_put({e[0], e[1]});
    dst[2 * i + 1] = unit_put({e[2], e[3]});
  }
}

// Daily mean / min / max of the steps of one item: the body of subdaily_pack_kernel for a source Src
template <typename Src, bool MEAN, bool EXT>
__device__ __forceinline__ void subdaily_pack(const Src& sp, const typename Src::V* src, int64_t stride16, int S,
                                              const int32_t* day, int64_t t_begin, int n_days,
                                              const int32_t* pack_src, int n_units, int halves, double2* dst_mean,
                                              uint4* dst_min, uint4* dst_max) {
  using T = typename Src::E;
  constexpr int C = Src::C;
  double sum[C];
  int cnt[C];
  T mn[C], mx[C];
  auto reset = [&] {
#pragma unroll
    for (int c = 0; c < C; ++c) {
      sum[c] = 0.0;
      cnt[c] = 0;
      mn[c] = mx[c] = (T)NAN;
    }
  };
  reset();
  subdaily_step_loop(
      sp, src, stride16, S, day, t_begin, n_days, pack_src, n_units, halves,
      [&](const T (&e)[C]) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
          if (MEAN && e[c] == e[c]) { sum[c] = __dadd_rn(sum[c], (double)e[c]); ++cnt[c]; }
          if (EXT) { mn[c] = ext_min(mn[c], e[c]); mx[c] = ext_max(mx[c], e[c]); }
        }
      },
      [&](int d, int u) {
        if (MEAN) {
#pragma unroll
          for (int c = 0; c < C; c += 2)
            dst_mean[((int64_t)d * n_units + u) * (C / 2) + c / 2] =
                make_double2(__ddiv_rn(sum[c], (double)cnt[c]), __ddiv_rn(sum[c + 1], (double)cnt[c + 1]));
        }
        if (EXT) {
          if (dst_min) item_put(dst_min, (int64_t)d * n_units + u, mn);
          if (dst_max) item_put(dst_max, (int64_t)d * n_units + u, mx);
        }
        reset();
      });
}

template <typename T, bool MEAN, bool EXT>
__global__ void __launch_bounds__(256) subdaily_pack_kernel(
    const uint4* __restrict__ src, int64_t stride16, int S, const int32_t* __restrict__ day, int64_t t_begin,
    int n_days, const int32_t* __restrict__ pack_src, int n_units, int halves, double2* __restrict__ dst_mean,
    uint4* __restrict__ dst_min, uint4* __restrict__ dst_max) {
  subdaily_pack<FloatSrc<T>, MEAN, EXT>(FloatSrc<T>{}, src, stride16, S, day, t_begin, n_days, pack_src, n_units,
                                        halves, dst_mean, dst_min, dst_max);
}

// subdaily_pack_kernel of a CF-packed int16 source decoded to D; a unit of the source is a piece (halves = 1).
// (256, 2): without the bound ptxas spills 8 bytes around the division's slow path in <double, mean only>
template <typename D, bool MEAN, bool EXT>
__global__ void __launch_bounds__(256, 2) subdaily_pack_decode_kernel(
    const uint2* __restrict__ src, int64_t stride8, const PackedI16Src<D> dec, int S, const int32_t* __restrict__ day,
    int64_t t_begin, int n_days, const int32_t* __restrict__ pack_src, int n_units, double2* __restrict__ dst_mean,
    uint4* __restrict__ dst_min, uint4* __restrict__ dst_max) {
  subdaily_pack<PackedI16Src<D>, MEAN, EXT>(dec, src, stride8, S, day, t_begin, n_days, pack_src, n_units, 1,
                                            dst_mean, dst_min, dst_max);
}

// Decode-pack of daily int16 data: the step loop with one step per day, day_index as the time index, and the
// decoded values stored to packed planes of D
template <typename D>
__global__ void __launch_bounds__(256) pull_pack_decode_kernel(
    const uint2* __restrict__ src, int64_t stride8, const PackedI16Src<D> dec, const int32_t* __restrict__ tix,
    int64_t t_begin, int T, const int32_t* __restrict__ pack_src, int n_units, uint4* __restrict__ dst) {
  D y[4];
  subdaily_step_loop(
      dec, src, stride8, 1, tix, t_begin, T, pack_src, n_units, 1,
      [&](const D (&e)[4]) {
#pragma unroll
        for (int c = 0; c < 4; ++c) y[c] = e[c];
      },
      [&](int d, int u) { item_put(dst, (int64_t)d * n_units + u, y); });
}
}  // namespace

namespace {
// The CF decoding of an int16 source as the kernels take it.  CTB_ERR_INVALID for a null dec, a non-finite scale
// or offset, n_fill outside 0..4 or a dtype other than F32 / F64.
int decode_check(const char* fn, const ctb_decode* dec) {
  if (!dec) { ctb_set_error("%s: dec is null", fn); return CTB_ERR_INVALID; }
  if (!std::isfinite(dec->scale) || !std::isfinite(dec->offset) || dec->n_fill < 0 || dec->n_fill > 4 ||
      (dec->dtype != CTB_F32 && dec->dtype != CTB_F64)) {
    ctb_set_error("%s: dec needs a finite scale and offset, 0..4 fill values and dtype F32 or F64, got scale=%g, "
                  "offset=%g, n_fill=%d, dtype=%d", fn, dec->scale, dec->offset, dec->n_fill, dec->dtype);
    return CTB_ERR_INVALID;
  }
  return CTB_OK;
}

template <typename D>
PackedI16Src<D> decode_src(const ctb_decode& dec) {
  PackedI16Src<D> s;
  s.scale = (D)dec.scale;
  s.offset = (D)dec.offset;
  for (int k = 0; k < 4; ++k) s.fill[k] = k < dec.n_fill ? (int)dec.fill[k] : 0x10000;
  return s;
}

// Bytes per decoded element
int decoded_bytes(const ctb_decode& dec) { return dec.dtype == CTB_F32 ? 4 : 8; }

// ctb_pull_pack_daily (es = float_bytes(dtype)), and with es = 2 its CF-decoding counterpart for int16 sources
int pull_pack_daily(const char* fn, const ctb_plan* P, const void* x, int dtype, int64_t es, const ctb_decode* dec,
                    int64_t stride, int steps_per_day, const int32_t* day_index, int64_t t_begin, int64_t n_days,
                    int ops, void* dst_mean, void* dst_min, void* dst_max, void* stream) {
  PullShape sh;
  if (int rc = pull_check(fn, P, x, dtype, es, stride, t_begin, n_days, n_days, &sh)) return rc;
  if (es != 2) dec = nullptr;
  else if (int rc = decode_check(fn, dec)) return rc;
  if (steps_per_day < 1) {
    ctb_set_error("%s: steps_per_day=%d, needs >= 1", fn, steps_per_day);
    return CTB_ERR_INVALID;
  }
  if (ops == 0 || (ops & ~(CTB_DAILY_MEAN | CTB_DAILY_MIN | CTB_DAILY_MAX))) {
    ctb_set_error("%s: ops=%d, needs a non-empty subset of CTB_DAILY_MEAN|MIN|MAX", fn, ops);
    return CTB_ERR_INVALID;
  }
  if (((ops & CTB_DAILY_MEAN) && !dst_mean) || ((ops & CTB_DAILY_MIN) && !dst_min) ||
      ((ops & CTB_DAILY_MAX) && !dst_max)) {
    ctb_set_error("%s: every requested op needs a destination", fn);
    return CTB_ERR_INVALID;
  }
  if ((ops & CTB_DAILY_MEAN) && P->elem_bytes != 8) {
    ctb_set_error("%s: the mean plane is float64, the plan was built for %d-byte elements", fn, P->elem_bytes);
    return CTB_ERR_INVALID;
  }
  const int ext_bytes = dec ? decoded_bytes(*dec) : (int)sh.es;   // min / max planes: the source's (decoded) type
  if ((ops & (CTB_DAILY_MIN | CTB_DAILY_MAX)) && P->elem_bytes != ext_bytes) {
    ctb_set_error("%s: min/max planes have the source's %d-byte elements, the plan was built for %d-byte elements",
                  fn, ext_bytes, P->elem_bytes);
    return CTB_ERR_INVALID;
  }
  if ((uintptr_t)dst_mean % 16 != 0 || (uintptr_t)dst_min % 16 != 0 || (uintptr_t)dst_max % 16 != 0) {
    ctb_set_error("%s: destination planes must be 16-byte aligned", fn);
    return CTB_ERR_UNSUPPORTED;
  }
  const bool mean = ops & CTB_DAILY_MEAN, ext = ops & (CTB_DAILY_MIN | CTB_DAILY_MAX);
  uint4* dmin = (ops & CTB_DAILY_MIN) ? static_cast<uint4*>(dst_min) : nullptr;
  uint4* dmax = (ops & CTB_DAILY_MAX) ? static_cast<uint4*>(dst_max) : nullptr;
  auto go = [&](auto tag) {
    using T = decltype(tag);
    auto k = mean ? (ext ? subdaily_pack_kernel<T, true, true> : subdaily_pack_kernel<T, true, false>)
                  : subdaily_pack_kernel<T, false, true>;
    k<<<sh.grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(x), sh.stride16, steps_per_day, day_index,
                                                  t_begin, (int)n_days, P->d_pack_src, sh.n_units, sh.halves,
                                                  static_cast<double2*>(dst_mean), dmin, dmax);
    return CTB_OK;
  };
  auto go_decode = [&](auto tag) {
    using D = decltype(tag);
    auto k = mean ? (ext ? subdaily_pack_decode_kernel<D, true, true> : subdaily_pack_decode_kernel<D, true, false>)
                  : subdaily_pack_decode_kernel<D, false, true>;
    k<<<sh.grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint2*>(x), sh.stride16, decode_src<D>(*dec),
                                                  steps_per_day, day_index, t_begin, (int)n_days, P->d_pack_src,
                                                  sh.n_units, static_cast<double2*>(dst_mean), dmin, dmax);
    return CTB_OK;
  };
  return pull_launch(P, n_days, [&] {
    if (dec) return dec->dtype == CTB_F32 ? go_decode(float{}) : go_decode(double{});
    return dtype == CTB_F32 ? go(float{}) : go(double{});
  });
}
}  // namespace

extern "C" int ctb_pull_pack_daily(const ctb_plan* P, const void* x, int dtype, int64_t stride, int steps_per_day,
                                   const int32_t* day_index, int64_t t_begin, int64_t n_days, int ops,
                                   void* dst_mean, void* dst_min, void* dst_max, void* stream) {
  return pull_pack_daily("ctb_pull_pack_daily", P, x, dtype, float_bytes(dtype), nullptr, stride, steps_per_day, day_index, t_begin,
                         n_days, ops, dst_mean, dst_min, dst_max, stream);
}

extern "C" int ctb_pull_pack_daily_decode(const ctb_plan* P, const int16_t* x, int64_t stride, const ctb_decode* dec,
                                          int steps_per_day, const int32_t* day_index, int64_t t_begin,
                                          int64_t n_days, int ops, void* dst_mean, void* dst_min, void* dst_max,
                                          void* stream) {
  return pull_pack_daily("ctb_pull_pack_daily_decode", P, x, 0, 2, dec, stride, steps_per_day, day_index, t_begin,
                         n_days, ops, dst_mean, dst_min, dst_max, stream);
}

extern "C" int ctb_pull_pack_decode(const ctb_plan* P, const int16_t* x, int64_t stride, const ctb_decode* dec,
                                    const int32_t* time_index, int64_t t_begin, int64_t T, void* dst, void* stream) {
  const char* fn = "ctb_pull_pack_decode";
  PullShape sh;
  if (int rc = pull_check(fn, P, x, 0, 2, stride, t_begin, T, T, &sh)) return rc;
  if (int rc = decode_check(fn, dec)) return rc;
  if (!dst && T > 0) { ctb_set_error("%s: dst is null", fn); return CTB_ERR_INVALID; }
  if (P->elem_bytes != decoded_bytes(*dec)) {
    ctb_set_error("%s: the planes have %d-byte elements, the plan was built for %d-byte elements", fn,
                  decoded_bytes(*dec), P->elem_bytes);
    return CTB_ERR_INVALID;
  }
  if ((uintptr_t)dst % 16 != 0) { ctb_set_error("%s: dst must be 16-byte aligned", fn); return CTB_ERR_UNSUPPORTED; }
  auto go = [&](auto tag) {
    using D = decltype(tag);
    pull_pack_decode_kernel<D><<<sh.grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint2*>(static_cast<const void*>(x)), sh.stride16, decode_src<D>(*dec), time_index, t_begin,
        (int)T, P->d_pack_src, sh.n_units, static_cast<uint4*>(dst));
    return CTB_OK;
  };
  return pull_launch(P, T, [&] { return dec->dtype == CTB_F32 ? go(float{}) : go(double{}); });
}

// Per-step transforms of sub-daily sources, reduced to daily means in the same read: the step loop and the plane
// layout of subdaily_pack_kernel, with NOUT float64 planes of f_j averaged over the day's non-NaN steps.
// The threshold and edge decisions are those of the aggregation kernels (CtbTr packed by
// ctb_pack_transform): fp64 comparisons for double sources; for float sources the fp32 comparisons against
// up / dn, which decide every float -- infinities included -- as the fp64 rule does (NaN steps never get here).
//   EDD:  f = x > e ? x - e : 0                                    (= max(x - e, 0): x - e > 0 <=> x > e)
//   GDD:  f = x > lo ? (x >= hi ? hi - lo : x - lo) : 0           (= min(max(x - lo, 0), hi - lo): rounding
//         is monotone, so x < hi gives fl(x - lo) <= fl(hi - lo) and x >= hi the reverse; +inf gives hi - lo)
//   BINS: a count per bin (ctb_bins_in), divided by the count of valid steps
namespace {
struct StepDst {
  double2* p[CTB_MAX_OUT];
};

// (256, 2): at most 128 registers, which every instantiation fits (the largest uses 127); without the bound
// ptxas spills 8 bytes around the division's slow path in one of them
template <typename Src, int OP, int NOUT>
__device__ __forceinline__ void subdaily_steps(const Src& sp, const typename Src::V* src, int64_t stride16, int S,
                                               const int32_t* day, int64_t t_begin, int n_days,
                                               const int32_t* pack_src, int n_units, int halves, const CtbTr& tr,
                                               const StepDst& dst) {
  using T = typename Src::E;
  constexpr int C = Src::C;
  constexpr bool F32 = sizeof(T) == 4;
  double w[NOUT];                     // GDD: hi - lo of every pair
#pragma unroll
  for (int j = 0; j < NOUT; ++j) w[j] = OP == CTB_STEP_GDD ? tr.a[2 * j + 1] - tr.a[2 * j] : 0.0;
  double sum[C][NOUT];
  int hits[C][NOUT];
  int cnt[C];
  auto reset = [&] {
#pragma unroll
    for (int c = 0; c < C; ++c) {
      cnt[c] = 0;
#pragma unroll
      for (int j = 0; j < NOUT; ++j) {
        sum[c][j] = 0.0;
        hits[c][j] = 0;
      }
    }
  };
  reset();
  subdaily_step_loop(
      sp, src, stride16, S, day, t_begin, n_days, pack_src, n_units, halves,
      [&](const T (&e)[C]) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
          if (!(e[c] == e[c])) continue;   // NaN step: skipped
          ++cnt[c];
          const double x = (double)e[c];
          if constexpr (OP == CTB_STEP_BINS) {
            bool in[NOUT];
            if constexpr (F32) ctb_bins_in_f32<NOUT>(tr, e[c], in); else ctb_bins_in<NOUT>(tr, x, in);
#pragma unroll
            for (int j = 0; j < NOUT; ++j) hits[c][j] += in[j];
          } else if constexpr (OP == CTB_STEP_EDD) {
#pragma unroll
            for (int j = 0; j < NOUT; ++j) {
              const bool above = F32 ? (float)e[c] > tr.dn[j] : x > tr.a[j];
              sum[c][j] = __dadd_rn(sum[c][j], above ? __dsub_rn(x, tr.a[j]) : 0.0);
            }
          } else {
#pragma unroll
            for (int j = 0; j < NOUT; ++j) {
              const bool above = F32 ? (float)e[c] > tr.dn[2 * j] : x > tr.a[2 * j];
              const bool top = F32 ? (float)e[c] >= tr.up[2 * j + 1] : x >= tr.a[2 * j + 1];
              const double f = top ? w[j] : __dsub_rn(x, tr.a[2 * j]);
              sum[c][j] = __dadd_rn(sum[c][j], above ? f : 0.0);
            }
          }
        }
      },
      [&](int d, int u) {
#pragma unroll
        for (int j = 0; j < NOUT; ++j) {
#pragma unroll
          for (int c = 0; c < C; c += 2) {
            const double s0 = OP == CTB_STEP_BINS ? (double)hits[c][j] : sum[c][j];
            const double s1 = OP == CTB_STEP_BINS ? (double)hits[c + 1][j] : sum[c + 1][j];
            dst.p[j][((int64_t)d * n_units + u) * (C / 2) + c / 2] =
                make_double2(__ddiv_rn(s0, (double)cnt[c]), __ddiv_rn(s1, (double)cnt[c + 1]));
          }
        }
        reset();
      });
}

template <typename T, int OP, int NOUT>
__global__ void __launch_bounds__(256, 2) subdaily_steps_kernel(
    const uint4* __restrict__ src, int64_t stride16, int S, const int32_t* __restrict__ day, int64_t t_begin,
    int n_days, const int32_t* __restrict__ pack_src, int n_units, int halves, const CtbTr tr, StepDst dst) {
  subdaily_steps<FloatSrc<T>, OP, NOUT>(FloatSrc<T>{}, src, stride16, S, day, t_begin, n_days, pack_src, n_units,
                                        halves, tr, dst);
}

// subdaily_steps_kernel of a CF-packed int16 source decoded to D; a unit of the source is a piece (halves = 1)
template <typename D, int OP, int NOUT>
__global__ void __launch_bounds__(256, 2) subdaily_steps_decode_kernel(
    const uint2* __restrict__ src, int64_t stride8, const PackedI16Src<D> dec, int S, const int32_t* __restrict__ day,
    int64_t t_begin, int n_days, const int32_t* __restrict__ pack_src, int n_units, const CtbTr tr, StepDst dst) {
  subdaily_steps<PackedI16Src<D>, OP, NOUT>(dec, src, stride8, S, day, t_begin, n_days, pack_src, n_units, 1, tr,
                                            dst);
}
}  // namespace

namespace {
// ctb_pull_pack_daily_steps (es = float_bytes(dtype)), and with es = 2 its CF-decoding counterpart for int16 sources
int pull_pack_daily_steps(const char* fn, const ctb_plan* P, const void* x, int dtype, int64_t es,
                          const ctb_decode* dec, int64_t stride, int steps_per_day, const int32_t* day_index,
                          int64_t t_begin, int64_t n_days, int step_op, const double* params, int n_params, int n_out,
                          double* const* dst, void* stream) {
  PullShape sh;
  if (int rc = pull_check(fn, P, x, dtype, es, stride, t_begin, n_days, n_days, &sh)) return rc;
  if (es != 2) dec = nullptr;
  else if (int rc = decode_check(fn, dec)) return rc;
  if (steps_per_day < 1) {
    ctb_set_error("%s: steps_per_day=%d, needs >= 1", fn, steps_per_day);
    return CTB_ERR_INVALID;
  }
  if (step_op != CTB_STEP_EDD && step_op != CTB_STEP_GDD && step_op != CTB_STEP_BINS) {
    ctb_set_error("%s: step_op=%d, needs CTB_STEP_EDD, GDD or BINS", fn, step_op);
    return CTB_ERR_INVALID;
  }
  if (n_out < 1 || n_out > CTB_MAX_OUT) {
    ctb_set_error("%s: n_out=%d out of range 1..%d", fn, n_out, CTB_MAX_OUT);
    return CTB_ERR_INVALID;
  }
  const int need = step_op == CTB_STEP_EDD ? n_out : step_op == CTB_STEP_GDD ? 2 * n_out : n_out + 1;
  if (n_params != need || !params) {
    ctb_set_error("%s: step_op %d with n_out=%d needs %d params, got %d", fn, step_op, n_out,
                  need, n_params);
    return CTB_ERR_INVALID;
  }
  for (int j = 0; j < n_params && step_op != CTB_STEP_BINS; ++j) {
    if (!std::isfinite(params[j]) || (step_op == CTB_STEP_GDD && j % 2 == 1 && !(params[j - 1] < params[j]))) {
      ctb_set_error("%s: thresholds must be finite, with lo < hi in every GDD pair: "
                    "param %d is %g", fn, j, params[j]);
      return CTB_ERR_INVALID;
    }
  }
  CtbTr tr;
  int rc;
  if (step_op == CTB_STEP_BINS) {
    double b[CTB_MAX_OUT + 2] = {0.0};   // offset 0, then the edges
    std::copy(params, params + n_params, b + 1);
    rc = ctb_pack_transform(CTB_TR_BINS, b, n_params + 1, n_out, &tr);
  } else {
    rc = ctb_pack_transform(step_op == CTB_STEP_EDD ? CTB_TR_EDD : CTB_TR_GDD, params, n_params, n_out, &tr);
  }
  if (rc != CTB_OK) return rc;
  if (!dst) { ctb_set_error("%s: dst is null", fn); return CTB_ERR_INVALID; }
  StepDst planes{};
  for (int j = 0; j < n_out; ++j) {
    if (!dst[j]) { ctb_set_error("%s: dst[%d] is null", fn, j); return CTB_ERR_INVALID; }
    if ((uintptr_t)dst[j] % 16 != 0) {
      ctb_set_error("%s: dst[%d] is not 16-byte aligned", fn, j);
      return CTB_ERR_UNSUPPORTED;
    }
    planes.p[j] = reinterpret_cast<double2*>(dst[j]);
  }
  if (P->elem_bytes != 8) {
    ctb_set_error("%s: the planes are float64, the plan was built for %d-byte elements", fn,
                  P->elem_bytes);
    return CTB_ERR_INVALID;
  }
  auto go = [&](auto tag) {
    auto launch = [&](auto op, auto nout) {
      subdaily_steps_kernel<decltype(tag), op, nout><<<sh.grid, 256, 0, (cudaStream_t)stream>>>(
          static_cast<const uint4*>(x), sh.stride16, steps_per_day, day_index, t_begin, (int)n_days, P->d_pack_src,
          sh.n_units, sh.halves, tr, planes);
      return CTB_OK;
    };
    if (step_op == CTB_STEP_EDD) return ctb_dispatch_nout<CTB_STEP_EDD>(n_out, launch);
    if (step_op == CTB_STEP_GDD) return ctb_dispatch_nout<CTB_STEP_GDD>(n_out, launch);
    return ctb_dispatch_nout<CTB_STEP_BINS>(n_out, launch);
  };
  auto go_decode = [&](auto tag) {
    using D = decltype(tag);
    auto launch = [&](auto op, auto nout) {
      subdaily_steps_decode_kernel<D, op, nout><<<sh.grid, 256, 0, (cudaStream_t)stream>>>(
          static_cast<const uint2*>(x), sh.stride16, decode_src<D>(*dec), steps_per_day, day_index, t_begin,
          (int)n_days, P->d_pack_src, sh.n_units, tr, planes);
      return CTB_OK;
    };
    if (step_op == CTB_STEP_EDD) return ctb_dispatch_nout<CTB_STEP_EDD>(n_out, launch);
    if (step_op == CTB_STEP_GDD) return ctb_dispatch_nout<CTB_STEP_GDD>(n_out, launch);
    return ctb_dispatch_nout<CTB_STEP_BINS>(n_out, launch);
  };
  return pull_launch(P, n_days, [&] {
    if (dec) return dec->dtype == CTB_F32 ? go_decode(float{}) : go_decode(double{});
    return dtype == CTB_F32 ? go(float{}) : go(double{});
  });
}
}  // namespace

extern "C" int ctb_pull_pack_daily_steps(const ctb_plan* P, const void* x, int dtype, int64_t stride,
                                         int steps_per_day, const int32_t* day_index, int64_t t_begin,
                                         int64_t n_days, int step_op, const double* params, int n_params, int n_out,
                                         double* const* dst, void* stream) {
  return pull_pack_daily_steps("ctb_pull_pack_daily_steps", P, x, dtype, float_bytes(dtype), nullptr, stride,
                               steps_per_day, day_index, t_begin, n_days, step_op, params, n_params, n_out, dst,
                               stream);
}

extern "C" int ctb_pull_pack_daily_steps_decode(const ctb_plan* P, const int16_t* x, int64_t stride,
                                                const ctb_decode* dec, int steps_per_day, const int32_t* day_index,
                                                int64_t t_begin, int64_t n_days, int step_op, const double* params,
                                                int n_params, int n_out, double* const* dst, void* stream) {
  return pull_pack_daily_steps("ctb_pull_pack_daily_steps_decode", P, x, 0, 2, dec, stride, steps_per_day,
                               day_index, t_begin, n_days, step_op, params, n_params, n_out, dst, stream);
}

// ---------------------------------------------------------------------------
// Fingerprint of a host buffer for the plan cache's fast path: 8 independent polynomial lanes
// h_j = h_j * P + word (mod 2^64, P odd) over the 64-bit words j, j+8, ..., folded with a second
// multiplier.  Editing a word, or swapping two different words, changes the value; the length is mixed in.
extern "C" uint64_t ctb_fingerprint(const void* data, size_t nbytes) {
  const unsigned char* p = static_cast<const unsigned char*>(data);
  constexpr uint64_t P = 0x9E3779B97F4A7C15ull, Q = 0xC2B2AE3D27D4EB4Full;
  uint64_t h[8] = {1, 2, 3, 4, 5, 6, 7, 8};
  size_t n64 = nbytes / 64;
  for (size_t i = 0; i < n64; ++i, p += 64) {
    uint64_t w[8];
    std::memcpy(w, p, 64);
#pragma GCC unroll 8
    for (int j = 0; j < 8; ++j) h[j] = h[j] * P + w[j];
  }
  uint64_t tail[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::memcpy(tail, p, nbytes - n64 * 64);
  uint64_t r = (uint64_t)nbytes;
  for (int j = 0; j < 8; ++j) r = (r ^ (h[j] * P + tail[j])) * Q + (r >> 29);
  return r;
}
