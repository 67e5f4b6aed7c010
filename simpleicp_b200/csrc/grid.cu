// grid.cu — build the static uniform grid over a cloud (done ONCE per cloud; the reference
// rebuilds a kd-tree over the transformed movable cloud every iteration,
// python/simpleicp/corrpts.py:131 — here the cloud never moves, the queries do).
//
// Pipeline (all HBM-streaming, one pass each over n points or n_cells cells):
//   k_bbox        : min/max of x,y,z                (reads 24 n B)
//   k_cell_count  : cell id per point + histogram   (reads 24 n B, n atomics into L2)
//   scan          : exclusive prefix over cells     (reads/writes 4 n_cells B, 3 kernels)
//   k_scatter     : cell-sorted 32-byte records     (reads 28 n B, writes 32 n B)
#include <algorithm>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "ctx.cuh"

namespace sicp {

namespace {

constexpr int kScanItems = 4096;  // cells per scan block (256 threads x 16)

__global__ void __launch_bounds__(256) k_bbox(const double* __restrict__ xyz, long long n,
                                              unsigned long long* __restrict__ out) {
  double mn[3] = {kInf, kInf, kInf}, mx[3] = {-kInf, -kInf, -kInf};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      double v = xyz[3 * i + a];
      mn[a] = fmin(mn[a], v);
      mx[a] = fmax(mx[a], v);
    }
  }
  __shared__ double smn[8][3], smx[8][3];
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    mn[a] = warp_min(mn[a]);
    mx[a] = warp_max(mx[a]);
    if (lane == 0) {
      smn[w][a] = mn[a];
      smx[w][a] = mx[a];
    }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    int a = threadIdx.x;
    double lo = smn[0][a], hi = smx[0][a];
    for (int i = 1; i < 8; ++i) {
      lo = fmin(lo, smn[i][a]);
      hi = fmax(hi, smx[i][a]);
    }
    atomicMin(&out[a], f64_to_key(lo));
    atomicMax(&out[3 + a], f64_to_key(hi));
  }
}

__global__ void k_bbox_init(unsigned long long* out) {
  if (threadIdx.x < 3) out[threadIdx.x] = ~0ull;
  else if (threadIdx.x < 6) out[threadIdx.x] = 0ull;
}
__global__ void k_bbox_decode(const unsigned long long* in, double* out) {
  if (threadIdx.x < 6) out[threadIdx.x] = key_to_f64(in[threadIdx.x]);
}

struct GridParams {
  double ox, oy, oz, inv_h;
  int nx, ny, nz;
};

__global__ void __launch_bounds__(256) k_cell_count(const double* __restrict__ xyz, long long n,
                                                    GridParams g, uint32_t* __restrict__ cid,
                                                    uint32_t* __restrict__ count) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  int cx = cell_coord(xyz[3 * i + 0], g.ox, g.inv_h, g.nx);
  int cy = cell_coord(xyz[3 * i + 1], g.oy, g.inv_h, g.ny);
  int cz = cell_coord(xyz[3 * i + 2], g.oz, g.inv_h, g.nz);
  uint32_t c = (uint32_t)(((long long)cz * g.ny + cy) * g.nx + cx);
  cid[i] = c;
  atomicAdd(&count[c], 1u);
}

// ---- 3-kernel exclusive scan over uint32 (n up to 2^27) ------------------------------------
__global__ void __launch_bounds__(256) k_scan_reduce(const uint32_t* __restrict__ in, long long n,
                                                     uint32_t* __restrict__ block_sums,
                                                     unsigned int* __restrict__ n_nonzero) {
  long long base = (long long)blockIdx.x * kScanItems;
  uint32_t s = 0, nz = 0;
  for (int j = threadIdx.x; j < kScanItems; j += 256) {
    long long i = base + j;
    if (i < n) {
      uint32_t v = in[i];
      s += v;
      nz += (v != 0);
    }
  }
  __shared__ uint32_t sh[8], shz[8];
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    nz += __shfl_xor_sync(0xffffffffu, nz, o);
  }
  if ((threadIdx.x & 31) == 0) {
    sh[threadIdx.x >> 5] = s;
    shz[threadIdx.x >> 5] = nz;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0, tz = 0;
    for (int i = 0; i < 8; ++i) {
      t += sh[i];
      tz += shz[i];
    }
    block_sums[blockIdx.x] = t;
    if (tz) atomicAdd(n_nonzero, tz);
  }
}

__global__ void __launch_bounds__(1024) k_scan_blocksums(uint32_t* __restrict__ block_sums, int nb) {
  // single block, sequential chunks of 1024 with a running carry
  __shared__ uint32_t sh[1024];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += 1024) {
    int i = base + threadIdx.x;
    uint32_t v = (i < nb) ? block_sums[i] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      uint32_t t = (threadIdx.x >= o) ? sh[threadIdx.x - o] : 0;
      __syncthreads();
      sh[threadIdx.x] += t;
      __syncthreads();
    }
    uint32_t incl = sh[threadIdx.x];
    uint32_t c = carry;
    if (i < nb) block_sums[i] = c + incl - v;  // exclusive
    __syncthreads();
    if (threadIdx.x == 1023) carry = c + incl;
    __syncthreads();
  }
}

// Exclusive scan of one 4096-item block, fully coalesced: thread t moves uint4 number j*256 + t
// (j = 0..3), i.e. 16-byte accesses with unit stride across the warp in both directions; the
// four 256-wide slabs are scanned one after the other with a running carry.
__global__ void __launch_bounds__(256) k_scan_down(const uint32_t* __restrict__ in, long long n,
                                                   const uint32_t* __restrict__ block_offsets,
                                                   uint32_t* __restrict__ out) {
  const long long base = (long long)blockIdx.x * kScanItems;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __shared__ uint32_t wsum[8];
  __shared__ uint32_t carry_s;
  uint32_t carry = block_offsets[blockIdx.x];
  const bool vec_ok = (base + kScanItems <= n) && ((reinterpret_cast<uintptr_t>(in + base) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(out + base) & 15) == 0);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long long i0 = base + 4ll * (j * 256 + threadIdx.x);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (vec_ok) {
      v = *reinterpret_cast<const uint4*>(in + i0);
    } else {
      if (i0 + 0 < n) v.x = in[i0 + 0];
      if (i0 + 1 < n) v.y = in[i0 + 1];
      if (i0 + 2 < n) v.z = in[i0 + 2];
      if (i0 + 3 < n) v.w = in[i0 + 3];
    }
    const uint32_t s = v.x + v.y + v.z + v.w;
    uint32_t incl = s;
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    __syncthreads();  // wsum / carry_s of the previous slab have been consumed
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    uint32_t woff = 0, tot = 0;
    for (int i = 0; i < 8; ++i) {
      if (i < w) woff += wsum[i];
      tot += wsum[i];
    }
    uint32_t run = carry + woff + incl - s;
    uint4 o4;
    o4.x = run;
    o4.y = run + v.x;
    o4.z = o4.y + v.y;
    o4.w = o4.z + v.z;
    if (vec_ok) {
      *reinterpret_cast<uint4*>(out + i0) = o4;
    } else {
      if (i0 + 0 < n) out[i0 + 0] = o4.x;
      if (i0 + 1 < n) out[i0 + 1] = o4.y;
      if (i0 + 2 < n) out[i0 + 2] = o4.z;
      if (i0 + 3 < n) out[i0 + 3] = o4.w;
    }
    carry += tot;
  }
  (void)carry_s;
}

__global__ void k_scan_total(const uint32_t* __restrict__ in, long long n,
                             uint32_t* __restrict__ out) {
  // out[n] = out[n-1] + in[n-1]
  if (threadIdx.x == 0 && blockIdx.x == 0) out[n] = (n > 0) ? out[n - 1] + in[n - 1] : 0;
}

__global__ void __launch_bounds__(256) k_scatter(const double* __restrict__ xyz, long long n,
                                                 const uint32_t* __restrict__ cid,
                                                 const uint32_t* __restrict__ cell_start,
                                                 uint32_t* __restrict__ fill,
                                                 Rec* __restrict__ recs) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t c = cid[i];
  uint32_t pos = cell_start[c] + atomicAdd(&fill[c], 1u);
  Rec r;
  r.x = xyz[3 * i + 0];
  r.y = xyz[3 * i + 1];
  r.z = xyz[3 * i + 2];
  r.idx = i;
  recs[pos] = r;
}

// Cells hold their points in arrival order of the atomics; sort each cell by original index so
// the layout (and therefore every memory trace) is reproducible run to run.  Cells are tiny
// (target occupancy ~3), insertion sort by one thread per cell.
__global__ void __launch_bounds__(256) k_sort_cells(const uint32_t* __restrict__ cell_start,
                                                    long long n_cells, Rec* __restrict__ recs) {
  long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (c >= n_cells) return;
  uint32_t s = cell_start[c], e = cell_start[c + 1];
  for (uint32_t i = s + 1; i < e; ++i) {
    Rec r = recs[i];
    uint32_t j = i;
    while (j > s && recs[j - 1].idx > r.idx) {
      recs[j] = recs[j - 1];
      --j;
    }
    recs[j] = r;
  }
}

__global__ void __launch_bounds__(256) k_float4_copy(const double* __restrict__ xyz, long long n,
                                                     long long n_pad, double cx, double cy,
                                                     double cz, float4* __restrict__ out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  float4 v;
  if (i < n) {
    v.x = (float)(xyz[3 * i + 0] - cx);
    v.y = (float)(xyz[3 * i + 1] - cy);
    v.z = (float)(xyz[3 * i + 2] - cz);
    v.w = 0.f;
  } else {
    v.x = v.y = v.z = 3.0e18f;  // padding: never the nearest neighbour
    v.w = 0.f;
  }
  out[i] = v;
}

}  // namespace

void grid_build(Ctx& c, Grid& g, const double* xyz, long long n) {
  cudaStream_t st = c.stream;
  g.built = false;
  g.n = n;
  static const bool trace = std::getenv("SICP_TRACE_RUN") != nullptr;
  const auto tr0 = std::chrono::steady_clock::now();
  auto tr = [&](const char* what) {
    if (trace)
      fprintf(stderr, "[grid_build] %-12s t=%.1f us\n", what,
              std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tr0).count());
  };
  // ---- bounding box
  c.bbox_keys.reserve(16);
  c.ws.scal.reserve(256);
  k_bbox_init<<<1, 32, 0, st>>>(c.bbox_keys.p);
  int nb = (int)std::min<long long>((n + 255) / 256, (long long)c.num_sms * 8);
  k_bbox<<<std::max(nb, 1), 256, 0, st>>>(xyz, n, c.bbox_keys.p);
  k_bbox_decode<<<1, 32, 0, st>>>(c.bbox_keys.p, c.ws.scal.p);
  SICP_CUDA(cudaMemcpyAsync(c.scal_host, c.ws.scal.p, 6 * sizeof(double), cudaMemcpyDeviceToHost, st));
  tr("bbox queued");
  SICP_CUDA(cudaStreamSynchronize(st));
  tr("bbox synced");
  double lo[3], ext[3];
  for (int a = 0; a < 3; ++a) {
    lo[a] = c.scal_host[a];
    ext[a] = c.scal_host[3 + a] - c.scal_host[a];
    SICP_REQUIRE(isfinite(lo[a]) && isfinite(ext[a]), SICP_ERR_BAD_ARG,
                 "point cloud contains non-finite coordinates");
  }
  // ---- initial cell size: assume a 2-D manifold in 3-D (scans): h ~ sqrt(target * A / n) with A
  // the product of the two largest extents; refined below from the measured occupancy.
  double e[3] = {ext[0], ext[1], ext[2]};
  std::sort(e, e + 3);
  double emax = std::max(e[2], 1e-12);
  double area = std::max(e[2] * std::max(e[1], 1e-3 * emax), 1e-300);
  double h = sqrt(c.grid_target_occ * area / (double)std::max<long long>(n, 1));
  h = std::max(h, emax * 1e-6);
  const long long kMaxCells = 1ll << 25;  // 32 M cells (128 MB of cell_start)
  c.misc_counters.reserve(64);

  for (int attempt = 0; attempt < 4; ++attempt) {
    long long d[3];
    for (;;) {
      for (int a = 0; a < 3; ++a) d[a] = std::max<long long>(1, (long long)floor(ext[a] / h) + 1);
      if (d[0] * d[1] * d[2] <= kMaxCells) break;
      h *= 1.26;  // 2x fewer cells per step
    }
    g.h = h;
    for (int a = 0; a < 3; ++a) {
      g.o[a] = lo[a];
      g.dims[a] = (int)d[a];
    }
    g.n_cells = d[0] * d[1] * d[2];
    g.cell_start.reserve(g.n_cells + 1);
    g.fill.reserve(g.n_cells);
    g.cid.reserve(n);
    long long nsb = (g.n_cells + kScanItems - 1) / kScanItems;
    g.block_sums.reserve(nsb + 1);
    SICP_CUDA(cudaMemsetAsync(g.fill.p, 0, g.n_cells * sizeof(uint32_t), st));
    SICP_CUDA(cudaMemsetAsync(c.misc_counters.p, 0, 64 * sizeof(unsigned int), st));
    GridParams gp{g.o[0], g.o[1], g.o[2], 1.0 / h, g.dims[0], g.dims[1], g.dims[2]};
    k_cell_count<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(xyz, n, gp, g.cid.p, g.fill.p);
    k_scan_reduce<<<(unsigned)nsb, 256, 0, st>>>(g.fill.p, g.n_cells, g.block_sums.p, c.misc_counters.p);
    k_scan_blocksums<<<1, 1024, 0, st>>>(g.block_sums.p, (int)nsb);
    k_scan_down<<<(unsigned)nsb, 256, 0, st>>>(g.fill.p, g.n_cells, g.block_sums.p, g.cell_start.p);
    k_scan_total<<<1, 32, 0, st>>>(g.fill.p, g.n_cells, g.cell_start.p);
    c.tm.kernel_launches += 5;
    unsigned int* nocc_host = reinterpret_cast<unsigned int*>(c.scal_host + 16);
    SICP_CUDA(cudaMemcpyAsync(nocc_host, c.misc_counters.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    tr("count queued");
    SICP_CUDA(cudaStreamSynchronize(st));
    tr("count synced");
    const unsigned int nocc = *nocc_host;
    g.n_occupied = nocc;
    double occ = (double)n / (double)std::max<unsigned int>(nocc, 1u);
    // accept when within a factor 1.6 of the target, or when the cell cap binds
    if (attempt == 3 || (occ <= c.grid_target_occ * 1.6 && occ >= c.grid_target_occ / 1.6)) break;
    if (occ > c.grid_target_occ && d[0] * d[1] * d[2] * 2 > kMaxCells) break;  // cannot refine
    // occupancy of occupied cells scales ~ h^dim with dim in [2,3] for scan data; use 2.3
    double f = pow(c.grid_target_occ / occ, 1.0 / 2.3);
    f = std::min(std::max(f, 0.25), 4.0);
    h *= f;
  }
  g.recs.reserve(n);
  SICP_CUDA(cudaMemsetAsync(g.fill.p, 0, g.n_cells * sizeof(uint32_t), st));
  k_scatter<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(xyz, n, g.cid.p, g.cell_start.p, g.fill.p,
                                                        g.recs.p);
  // optional: order the records of every cell by original index (reproducible memory layout for
  // profiling; the search results never depend on it because ties are broken by index)
  if (c.grid_sort_cells)
    k_sort_cells<<<(unsigned)((g.n_cells + 255) / 256), 256, 0, st>>>(g.cell_start.p, g.n_cells,
                                                                     g.recs.p);
  SICP_CUDA(cudaGetLastError());
  tr("scatter queued");
  c.tm.kernel_launches += 5;  // bbox x3, scatter, sort_cells
  g.built = true;
}

// =============================================================================================
// Batched build: the grids of many (small) clouds in one segmented counting sort.
//   * all clouds share one record array (cloud c owns [rec_base, rec_base + n)) and one cell table
//     (cloud c owns [cell_base, cell_base + n_cells]); cell-table entries are GLOBAL record
//     positions, so one exclusive scan over the concatenated counters serves every cloud and the
//     end sentinel of a cloud is the first entry of the next;
//   * blockIdx.y selects the cloud in every per-point kernel;
//   * cell sizes follow the same rule as the single build (2-D manifold estimate, then refinement
//     from the measured occupancy); the host sees bounding boxes and occupancies of the whole
//     batch at once (three small read-backs per BATCH instead of three per cloud).
// Rec::idx is the index inside its own cloud.
// =============================================================================================
namespace {

__global__ void __launch_bounds__(256) k_bbox_batch(const CloudPlan* __restrict__ plans,
                                                    unsigned long long* __restrict__ keys) {
  const CloudPlan pl = plans[blockIdx.y];
  const double* __restrict__ xyz = pl.xyz;
  double mn[3] = {kInf, kInf, kInf}, mx[3] = {-kInf, -kInf, -kInf};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < pl.n;
       i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double v = xyz[3 * i + a];
      mn[a] = fmin(mn[a], v);
      mx[a] = fmax(mx[a], v);
    }
  }
  __shared__ double smn[8][3], smx[8][3];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    mn[a] = warp_min(mn[a]);
    mx[a] = warp_max(mx[a]);
    if (lane == 0) {
      smn[w][a] = mn[a];
      smx[w][a] = mx[a];
    }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int a = threadIdx.x;
    double lo = smn[0][a], hi = smx[0][a];
    for (int i = 1; i < 8; ++i) {
      lo = fmin(lo, smn[i][a]);
      hi = fmax(hi, smx[i][a]);
    }
    atomicMin(&keys[6 * blockIdx.y + a], f64_to_key(lo));
    atomicMax(&keys[6 * blockIdx.y + 3 + a], f64_to_key(hi));
  }
}

__global__ void k_bbox_batch_init(unsigned long long* keys, int n_clouds) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 6 * n_clouds) keys[i] = ((i % 6) < 3) ? ~0ull : 0ull;
}

__global__ void __launch_bounds__(256) k_cell_count_batch(const CloudPlan* __restrict__ plans,
                                                          uint32_t* __restrict__ cid,
                                                          uint32_t* __restrict__ count,
                                                          unsigned int* __restrict__ occ) {
  const CloudPlan pl = plans[blockIdx.y];
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  int first = 0;
  if (i < pl.n) {
    const int cx = cell_coord(pl.xyz[3 * i + 0], pl.ox, pl.inv_h, pl.nx);
    const int cy = cell_coord(pl.xyz[3 * i + 1], pl.oy, pl.inv_h, pl.ny);
    const int cz = cell_coord(pl.xyz[3 * i + 2], pl.oz, pl.inv_h, pl.nz);
    const uint32_t cell = (uint32_t)(((long long)cz * pl.ny + cy) * pl.nx + cx);
    cid[pl.rec_base + i] = cell;
    first = (atomicAdd(&count[pl.cell_base + cell], 1u) == 0u) ? 1 : 0;
  }
  // occupied cells of this cloud: ONE atomic per block (one per first touch serialised 30 000
  // same-address atomics per cloud: 113 us for 1.6 M points, ncu r2)
  const int n_first = __syncthreads_count(first);
  if (threadIdx.x == 0 && n_first) atomicAdd(&occ[blockIdx.y], (unsigned int)n_first);
}

__global__ void __launch_bounds__(256) k_scatter_batch(const CloudPlan* __restrict__ plans,
                                                       const uint32_t* __restrict__ cid,
                                                       const uint32_t* __restrict__ cell_start,
                                                       uint32_t* __restrict__ fill,
                                                       Rec* __restrict__ recs) {
  const CloudPlan pl = plans[blockIdx.y];
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= pl.n) return;
  const uint32_t cell = cid[pl.rec_base + i];
  const uint32_t pos = cell_start[pl.cell_base + cell] + atomicAdd(&fill[pl.cell_base + cell], 1u);
  Rec r;
  r.x = pl.xyz[3 * i + 0];
  r.y = pl.xyz[3 * i + 1];
  r.z = pl.xyz[3 * i + 2];
  r.idx = i;
  recs[pos] = r;
}

inline double host_key_to_f64(unsigned long long k) {
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  double v;
  std::memcpy(&v, &b, sizeof(v));
  return v;
}

}  // namespace

// The three-kernel scan plus the total: the batched grid build's cell table and the overlap
// filter's kept lists (nn.cu: batch_overlap_launch) both come out of one scan over a whole batch.
void scan_u32(Ctx& c, const uint32_t* in, long long n, DevBuf<uint32_t>& block_sums, uint32_t* out) {
  cudaStream_t st = c.stream;
  const long long nsb = (n + kScanItems - 1) / kScanItems;
  block_sums.reserve(nsb + 1);
  c.misc_counters.reserve(64);
  SICP_CUDA(cudaMemsetAsync(c.misc_counters.p + 16, 0, sizeof(unsigned int), st));  // the kernel's (unused here) nonzero counter
  k_scan_reduce<<<(unsigned)nsb, 256, 0, st>>>(in, n, block_sums.p, c.misc_counters.p + 16);
  k_scan_blocksums<<<1, 1024, 0, st>>>(block_sums.p, (int)nsb);
  k_scan_down<<<(unsigned)nsb, 256, 0, st>>>(in, n, block_sums.p, out);
  k_scan_total<<<1, 32, 0, st>>>(in, n, out);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 4;
}

void grid_build_batch(Ctx& c, Batch& b, BatchGrid& bg, const std::vector<BatchHostCloud>& clouds,
                      std::vector<GridView>& views, std::vector<double>& centres) {
  cudaStream_t st = c.stream;
  const int nc = (int)clouds.size();
  long long total_pts = 0, max_n = 0;
  for (const auto& cl : clouds) {
    total_pts = std::max(total_pts, cl.point_off + cl.n);
    max_n = std::max(max_n, cl.n);
  }
  SICP_REQUIRE(total_pts < (1ll << 32), SICP_ERR_BAD_ARG, "a batch is limited to 2^32 - 1 points in total");
  const size_t need_keys = (size_t)nc * 8;
  if (b.keys_cap < need_keys) {
    if (b.keys_host) cudaFreeHost(b.keys_host);
    SICP_CUDA(cudaMallocHost(&b.keys_host, need_keys * sizeof(unsigned long long)));
    b.keys_cap = need_keys;
  }
  b.bbox_keys.reserve((size_t)nc * 6);
  b.plans.reserve(nc);
  b.occ.reserve(nc);
  bg.cid.reserve(total_pts);
  bg.recs.reserve(total_pts);
  std::vector<CloudPlan> plans((size_t)nc);
  for (int i = 0; i < nc; ++i) {
    plans[(size_t)i] = CloudPlan{};
    plans[(size_t)i].xyz = clouds[(size_t)i].xyz_dev;
    plans[(size_t)i].n = clouds[(size_t)i].n;
    plans[(size_t)i].rec_base = clouds[(size_t)i].point_off;
  }
  auto upload_plans = [&]() {
    // pageable source: the runtime stages it before returning, `plans` may change afterwards
    SICP_CUDA(cudaMemcpyAsync(b.plans.p, plans.data(), sizeof(CloudPlan) * (size_t)nc, cudaMemcpyHostToDevice, st));
  };
  upload_plans();
  const unsigned bx = (unsigned)std::max<long long>(1, std::min<long long>((max_n + 255) / 256, 64));
  k_bbox_batch_init<<<(6 * nc + 255) / 256, 256, 0, st>>>(b.bbox_keys.p, nc);
  k_bbox_batch<<<dim3(bx, nc), 256, 0, st>>>(b.plans.p, b.bbox_keys.p);
  SICP_CUDA(cudaMemcpyAsync(b.keys_host, b.bbox_keys.p, sizeof(unsigned long long) * 6 * (size_t)nc,
                            cudaMemcpyDeviceToHost, st));
  SICP_CUDA(cudaStreamSynchronize(st));
  c.tm.kernel_launches += 2;

  std::vector<double> lo((size_t)nc * 3), ext((size_t)nc * 3), h((size_t)nc);
  for (int i = 0; i < nc; ++i) {
    double e[3];
    for (int a = 0; a < 3; ++a) {
      lo[(size_t)i * 3 + a] = host_key_to_f64(b.keys_host[6 * i + a]);
      ext[(size_t)i * 3 + a] = host_key_to_f64(b.keys_host[6 * i + 3 + a]) - lo[(size_t)i * 3 + a];
      SICP_REQUIRE(std::isfinite(lo[(size_t)i * 3 + a]) && std::isfinite(ext[(size_t)i * 3 + a]), SICP_ERR_BAD_ARG,
                   "point cloud contains non-finite coordinates");
      e[a] = ext[(size_t)i * 3 + a];
    }
    std::sort(e, e + 3);
    const double emax = std::max(e[2], 1e-12);
    const double area = std::max(e[2] * std::max(e[1], 1e-3 * emax), 1e-300);
    h[(size_t)i] = std::max(sqrt(c.grid_target_occ * area / (double)std::max<long long>(plans[(size_t)i].n, 1)), emax * 1e-6);
  }
  // per-cloud cell cap: generous for scans (a 2-D manifold in a 3-D box), bounded for the batch
  auto cap_of = [&](long long n) { return std::min<long long>(1ll << 25, std::max<long long>(4096, 32 * n)); };
  long long total_cells = 0;
  std::vector<char> final_h((size_t)nc, 0);
  for (int attempt = 0; attempt < 4; ++attempt) {
    total_cells = 0;
    for (int i = 0; i < nc; ++i) {
      CloudPlan& pl = plans[(size_t)i];
      long long d[3];
      for (;;) {
        for (int a = 0; a < 3; ++a) d[a] = std::max<long long>(1, (long long)floor(ext[(size_t)i * 3 + a] / h[(size_t)i]) + 1);
        if (d[0] * d[1] * d[2] <= cap_of(pl.n)) break;
        h[(size_t)i] *= 1.26;
        final_h[(size_t)i] = 1;  // the cap binds: no further refinement
      }
      pl.ox = lo[(size_t)i * 3 + 0];
      pl.oy = lo[(size_t)i * 3 + 1];
      pl.oz = lo[(size_t)i * 3 + 2];
      pl.h = h[(size_t)i];
      pl.inv_h = 1.0 / h[(size_t)i];
      pl.nx = (int)d[0];
      pl.ny = (int)d[1];
      pl.nz = (int)d[2];
      pl.cell_base = total_cells;
      total_cells += d[0] * d[1] * d[2];
    }
    SICP_REQUIRE(total_cells < (1ll << 31), SICP_ERR_BAD_ARG, "batch needs too many grid cells: use smaller batches");
    upload_plans();
    bg.cell_table.reserve(total_cells + 1);
    bg.fill.reserve(total_cells + 1);
    SICP_CUDA(cudaMemsetAsync(bg.fill.p, 0, (size_t)total_cells * sizeof(uint32_t), st));
    SICP_CUDA(cudaMemsetAsync(b.occ.p, 0, (size_t)nc * sizeof(unsigned int), st));
    k_cell_count_batch<<<dim3((unsigned)((max_n + 255) / 256), nc), 256, 0, st>>>(b.plans.p, bg.cid.p, bg.fill.p, b.occ.p);
    c.tm.kernel_launches += 1;
    unsigned int* occ_host = reinterpret_cast<unsigned int*>(b.keys_host);
    SICP_CUDA(cudaMemcpyAsync(occ_host, b.occ.p, sizeof(unsigned int) * (size_t)nc, cudaMemcpyDeviceToHost, st));
    SICP_CUDA(cudaStreamSynchronize(st));
    bool again = false;
    for (int i = 0; i < nc && attempt < 3; ++i) {
      if (final_h[(size_t)i]) continue;
      const double occ = (double)plans[(size_t)i].n / (double)std::max<unsigned int>(occ_host[i], 1u);
      if (occ <= c.grid_target_occ * 1.6 && occ >= c.grid_target_occ / 1.6) {
        final_h[(size_t)i] = 1;
        continue;
      }
      double f = pow(c.grid_target_occ / occ, 1.0 / 2.3);
      f = std::min(std::max(f, 0.25), 4.0);
      h[(size_t)i] *= f;
      again = true;
    }
    if (!again) break;
  }
  // exclusive scan of the concatenated counters -> global record positions
  scan_u32(c, bg.fill.p, total_cells, bg.block_sums, bg.cell_table.p);
  SICP_CUDA(cudaMemsetAsync(bg.fill.p, 0, (size_t)total_cells * sizeof(uint32_t), st));
  k_scatter_batch<<<dim3((unsigned)((max_n + 255) / 256), nc), 256, 0, st>>>(b.plans.p, bg.cid.p, bg.cell_table.p, bg.fill.p, bg.recs.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
  views.resize((size_t)nc);
  centres.resize((size_t)nc * 3);
  for (int i = 0; i < nc; ++i) {
    const CloudPlan& pl = plans[(size_t)i];
    GridView v;
    v.recs = bg.recs.p;
    v.cell_start = bg.cell_table.p + pl.cell_base;
    v.ox = pl.ox;
    v.oy = pl.oy;
    v.oz = pl.oz;
    v.h = pl.h;
    v.inv_h = pl.inv_h;
    v.nx = pl.nx;
    v.ny = pl.ny;
    v.nz = pl.nz;
    v.n_points = total_pts;  // positions in the shared record array are global
    views[(size_t)i] = v;
    centres[(size_t)i * 3 + 0] = pl.ox + 0.5 * pl.nx * pl.h;
    centres[(size_t)i * 3 + 1] = pl.oy + 0.5 * pl.ny * pl.h;
    centres[(size_t)i * 3 + 2] = pl.oz + 0.5 * pl.nz * pl.h;
  }
}

void make_float4_copy(Ctx& c) {
  // centred float4 copy of the movable cloud in caller order (TMA brute-force engine)
  const GridView v = c.gmov.view();
  double hi[3] = {v.ox + v.nx * v.h, v.oy + v.ny * v.h, v.oz + v.nz * v.h};
  c.mov_center[0] = 0.5 * (v.ox + hi[0]);
  c.mov_center[1] = 0.5 * (v.oy + hi[1]);
  c.mov_center[2] = 0.5 * (v.oz + hi[2]);
  c.mov_radius = 0.5 * std::max(hi[0] - v.ox, std::max(hi[1] - v.oy, hi[2] - v.oz));
  long long n_pad = ((c.n_mov + kBfTile - 1) / kBfTile) * kBfTile;
  c.mov_f4.reserve(n_pad);
  k_float4_copy<<<(unsigned)((n_pad + 255) / 256), 256, 0, c.stream>>>(
      c.mov_xyz.p, c.n_mov, n_pad, c.mov_center[0], c.mov_center[1], c.mov_center[2], c.mov_f4.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

}  // namespace sicp
