// nn.cu — nearest-neighbour correspondence search (reference: CorrPts.match,
// python/simpleicp/corrpts.py:124-137 + 195-211, and PointCloud.select_in_range,
// python/simpleicp/pointcloud.py:149-171).
//
// The reference transforms the whole movable cloud by H, rebuilds a kd-tree and queries it with
// the selected fixed points.  Rigid maps preserve distances, so here the K queries are moved by
// H^-1 instead and searched in a STATIC structure over the original movable cloud; only the
// matched point is moved by H for the point-to-plane distance.
//
// Two exact engines:
//   grid  : uniform-grid search in float64, 3x3x3 block then shell-by-shell ring expansion until
//           the best distance is provably <= the distance to every unexplored cell.
//   brute : tiled exhaustive search.  float4 tiles of the (centred, float32) cloud are staged
//           into shared memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier, 4-stage ring),
//           lanes split the tile, float32 distances act as a FILTER with a rigorous error margin,
//           every candidate that passes is re-evaluated in float64 from the original
//           coordinates, and the per-lane winners are combined with a warp-shuffle min-reduction.
// Ties are broken towards the lower original index in both.
#include <algorithm>

#include "ctx.cuh"

namespace sicp {

namespace {

// ------------------------------------------------------------------------------------------
// grid engine
// ------------------------------------------------------------------------------------------
// bpos follows the winner's position in the cell-sorted record array: the record holds the
// original coordinates, so whoever needs the matched point afterwards re-reads that (cache-hot)
// record instead of gathering mov_xyz[bidx] from a cold line.
__device__ __forceinline__ void consider(const Rec& r, uint32_t pos, double qx, double qy, double qz,
                                         double& best, long long& bidx, uint32_t& bpos) {
  const double dx = r.x - qx, dy = r.y - qy, dz = r.z - qz;
  const double d2 = dx * dx + dy * dy + dz * dz;
  if (d2 < best || (d2 == best && r.idx < bidx)) {
    best = d2;
    bidx = r.idx;
    bpos = pos;
  }
}

// Scan the records [s, e).  The search is latency-bound, so four 32-byte records (LDG.E.256
// each) are requested before the first one is used; the tail re-reads the last record instead
// of branching (a duplicate never changes the result: same distance, same index).
__device__ __forceinline__ void scan_range(const Rec* __restrict__ recs, uint32_t s, uint32_t e,
                                           double qx, double qy, double qz, double& best,
                                           long long& bidx, uint32_t& bpos) {
  for (uint32_t i = s; i < e; i += 4) {
    const uint32_t last = e - 1;
    const uint32_t i1 = min(i + 1, last), i2 = min(i + 2, last), i3 = min(i + 3, last);
    const Rec r0 = recs[i];
    const Rec r1 = recs[i1];
    const Rec r2 = recs[i2];
    const Rec r3 = recs[i3];
    consider(r0, i, qx, qy, qz, best, bidx, bpos);
    consider(r1, i1, qx, qy, qz, best, bidx, bpos);
    consider(r2, i2, qx, qy, qz, best, bidx, bpos);
    consider(r3, i3, qx, qy, qz, best, bidx, bpos);
  }
}

// Returns true when (best, bidx) is proven to be the nearest neighbour.
// cap2 >= 0: the caller only needs to know on which side of cap2 the squared nearest-neighbour
// distance lies (overlap filter, PointCloud.select_in_range): the search may stop as soon as any
// point closer than the bound is found, or once every unexplored cell is farther than the bound.
__device__ bool grid_nn(const GridView& g, double qx, double qy, double qz, int rmax, double cap2,
                        double& best, long long& bidx) {
  const int cx = cell_coord(qx, g.ox, g.inv_h, g.nx);
  const int cy = cell_coord(qy, g.oy, g.inv_h, g.ny);
  const int cz = cell_coord(qz, g.oz, g.inv_h, g.nz);
  best = kInf;
  bidx = -1;
  uint32_t bpos = 0;
  const uint32_t* __restrict__ cs = g.cell_start;
  for (int r = 1;; ++r) {
    const int x0 = cx - r, x1 = cx + r, y0 = cy - r, y1 = cy + r, z0 = cz - r, z1 = cz + r;
    const int xa = max(x0, 0), xb = min(x1, g.nx - 1);
    const int za = max(z0, 0), zb = min(z1, g.nz - 1);
    const int ya = max(y0, 0), yb = min(y1, g.ny - 1);
    for (int z = za; z <= zb; ++z) {
      for (int y = ya; y <= yb; ++y) {
        const long long row = ((long long)z * g.ny + y) * g.nx;
        const bool full = (r == 1) || z == z0 || z == z1 || y == y0 || y == y1;
        if (full) {
          scan_range(g.recs, cs[row + xa], cs[row + xb + 1], qx, qy, qz, best, bidx, bpos);
        } else {
          if (x0 >= 0) scan_range(g.recs, cs[row + x0], cs[row + x0 + 1], qx, qy, qz, best, bidx, bpos);
          if (x1 < g.nx) scan_range(g.recs, cs[row + x1], cs[row + x1 + 1], qx, qy, qz, best, bidx, bpos);
        }
      }
    }
    // distance from the query to the nearest face behind which unexplored cells remain
    double guard = kInf;
    if (x0 > 0) guard = fmin(guard, qx - (g.ox + x0 * g.h));
    if (x1 < g.nx - 1) guard = fmin(guard, (g.ox + (x1 + 1) * g.h) - qx);
    if (y0 > 0) guard = fmin(guard, qy - (g.oy + y0 * g.h));
    if (y1 < g.ny - 1) guard = fmin(guard, (g.oy + (y1 + 1) * g.h) - qy);
    if (z0 > 0) guard = fmin(guard, qz - (g.oz + z0 * g.h));
    if (z1 < g.nz - 1) guard = fmin(guard, (g.oz + (z1 + 1) * g.h) - qz);
    if (guard >= kInf) return true;  // the block covers the whole grid
    guard -= 1e-9 * g.h;             // cell assignment of points rounds at the 1e-13 level
    if (guard > 0.0 && best <= guard * guard) return true;
    if (cap2 >= 0.0 && (best < cap2 || (guard > 0.0 && guard * guard >= cap2))) return true;
    if (r >= rmax) return false;
  }
}

// signed point-to-plane distance exactly as the reference evaluates it (corrpts.py:198-209):
// (dx*nx + dy*ny) + dz*nz with the float32 normal promoted to float64, no fused multiply-add.
__device__ __forceinline__ double plane_distance(const Rigid& T, const double* __restrict__ mov_xyz,
                                                 long long j, double px, double py, double pz,
                                                 float4 nrm) {
  double tx, ty, tz;
  rigid_apply(T, mov_xyz[3 * j + 0], mov_xyz[3 * j + 1], mov_xyz[3 * j + 2], tx, ty, tz);
  const double dx = tx - px, dy = ty - py, dz = tz - pz;
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, (double)nrm.x), __dmul_rn(dy, (double)nrm.y)),
                   __dmul_rn(dz, (double)nrm.z));
}

__device__ __forceinline__ double plane_distance_rec(const Rigid& T, const Rec& m, double px, double py,
                                                     double pz, float4 nrm) {
  double tx, ty, tz;
  rigid_apply(T, m.x, m.y, m.z, tx, ty, tz);
  const double dx = tx - px, dy = ty - py, dz = tz - pz;
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, (double)nrm.x), __dmul_rn(dy, (double)nrm.y)),
                   __dmul_rn(dz, (double)nrm.z));
}

// Feed the predictor histogram of the reject kernel (reject_solve.cuh: lh_bin): one spread-out
// atomic per planarity survivor instead of a separate pass over the distances later.
// Feed the predictor histogram of the reject kernel (reject_solve.cuh: lh_bin): one spread-out
// atomic per member of the statistics set instead of a separate pass over the distances later.
// The value the atomic returns is the correspondence's rank inside its bin: it doubles as the
// slot of a per-bin index store, so that the reject/solve kernel can read the members of the few
// bins that hold its order statistics directly (no scan, no gather pass, no barrier).
__device__ __forceinline__ void lin_hist_add(const DevState* st, unsigned int* lin_hist,
                                             float planarity, double d, unsigned int* binstore,
                                             int bin_cap, long long qi) {
  if (lin_hist != nullptr && st->pred_valid && (double)planarity >= st->pred_minpl) {
    const int b = lh_bin(d, st->pred_med, st->pred_mad);
    const unsigned int slot = atomicAdd(&lin_hist[b], 1u);
    if (binstore != nullptr && b < LH_BINS && slot < (unsigned int)bin_cap)
      binstore[(size_t)b * bin_cap + slot] = (unsigned int)qi;
  }
}

// Epilogue data of one correspondence for the fused reject/solve kernel: the matched movable
// point in caller coordinates (so the moment pass streams it instead of chasing nn_idx ->
// mov_xyz) and the histogram code.
struct CorrOut {
  unsigned int* binstore;  // LH_BINS x bin_cap correspondence numbers, may be null
  int bin_cap;
  double* m_xyz;           // K x 3, may be null
  // Warm start (may be null): position, in the cell-sorted record array, of the neighbour each
  // query found in the PREVIOUS iteration of this registration.  Its distance to the moved query
  // is a valid upper bound from the first instruction on, so most of the 27 cells of ring 1 are
  // pruned by their distance bound before their cell-table entries are even requested.  The
  // result is unchanged (any point is a valid bound; ties still go to the lower index).
  uint32_t* nn_pos;
  int warm;              // nn_pos holds positions of the previous iteration
  int sphere;            // finish a search inside the sphere of the first known point (option "sphere_scan")
  // Movable-side attributes (null = the reference's default run, pc_mov without normals):
  // mov_nrm[j] = (nx, ny, nz, planarity) of movable point j in ITS OWN frame, NaN where not
  // estimated.  q_eff[i] receives the fixed normal with an "effective planarity" that carries
  // both movable-side tests to the reject kernels (effective_planarity below).
  const float4* mov_nrm;
  float4* q_eff;
  double cos_max;        // cos of the largest accepted angle between the normals; < 0: no angle test
};
// CorrPts.reject_wrt_planarity's second branch (corrpts.py:157-162: a correspondence also needs
// planarity >= min_planarity on the MOVABLE side when pc_mov carries the column; NaN, i.e. "not
// estimated", fails the comparison) and the hook the reference leaves unimplemented
// (reject_wrt_to_angle_between_normals, corrpts.py:190-193; called after the distance rejection,
// simpleicp.py:207).  Both are folded into one float per correspondence:
//   |w| = min(planarity_fix, planarity_mov)   (NaN if either is NaN): both planarity tests are
//         |w| >= min_planarity, and the median / MAD population is the set that passes them;
//   sign(w) = 1 if the angle between the fixed normal and the ROTATED movable normal exceeds the
//         limit (normals are axes: the angle is taken modulo their sign): such a correspondence
//         takes part in the median / MAD like in the reference's call order, and is dropped after it.
__device__ __forceinline__ float effective_planarity(const CorrOut& co, const Rigid& T, long long qi,
                                                     long long midx, const float4& nr) {
  if (co.mov_nrm == nullptr) return nr.w;
  const float4 m = co.mov_nrm[midx];
  float w = (m.w >= nr.w) ? nr.w : ((m.w < nr.w) ? m.w : __int_as_float(0x7fc00000));
  if (co.cos_max >= 0.0) {
    const double rx = T.r[0] * (double)m.x + T.r[1] * (double)m.y + T.r[2] * (double)m.z;
    const double ry = T.r[3] * (double)m.x + T.r[4] * (double)m.y + T.r[5] * (double)m.z;
    const double rz = T.r[6] * (double)m.x + T.r[7] * (double)m.y + T.r[8] * (double)m.z;
    const double c = fabs(rx * (double)nr.x + ry * (double)nr.y + rz * (double)nr.z);
    if (!(c >= co.cos_max)) w = __int_as_float(__float_as_int(w) | 0x80000000);
  }
  co.q_eff[qi] = make_float4(nr.x, nr.y, nr.z, w);
  return fabsf(w);
}
__device__ __forceinline__ void store_matched(const CorrOut& co, long long qi, double x, double y, double z) {
  if (co.m_xyz) {
    co.m_xyz[3 * qi + 0] = x;
    co.m_xyz[3 * qi + 1] = y;
    co.m_xyz[3 * qi + 2] = z;
  }
}

__global__ void __launch_bounds__(128)
    k_match_grid(GridView g, const DevState* __restrict__ st, const double* __restrict__ q_xyz,
                 const float4* __restrict__ q_nrm, const double* __restrict__ mov_xyz, long long K,
                 int rmax, int with_distance, long long* __restrict__ nn_idx,
                 double* __restrict__ out, unsigned int* __restrict__ unresolved,
                 unsigned int* __restrict__ lin_hist, double cap2, CorrOut co) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K || st->stop) return;
  const Rigid Tinv = st->Tinv;
  const double px = q_xyz[3 * i + 0], py = q_xyz[3 * i + 1], pz = q_xyz[3 * i + 2];
  double qx, qy, qz;
  rigid_apply(Tinv, px, py, pz, qx, qy, qz);
  double best;
  long long bidx;
  const bool ok = grid_nn(g, qx, qy, qz, rmax, cap2, best, bidx);
  if (!ok) {
    const unsigned int slot = atomicAdd(&unresolved[K], 1u);
    unresolved[slot] = (unsigned int)i;
    return;
  }
  nn_idx[i] = bidx;
  if (with_distance) {
    const float4 nr = q_nrm[i];
    const double d = plane_distance(st->T, mov_xyz, bidx, px, py, pz, nr);
    out[i] = d;
    lin_hist_add(st, lin_hist, effective_planarity(co, st->T, i, bidx, nr), d, co.binstore, co.bin_cap, i);
    store_matched(co, i, mov_xyz[3 * bidx + 0], mov_xyz[3 * bidx + 1], mov_xyz[3 * bidx + 2]);
  } else {
    out[i] = best;
  }
}

// Cooperative variant: MG lanes share one query.  In ring 1 every lane owns one of the 9 grid
// rows (x-contiguous cell triples), so the 9 dependent chains cell_start -> records run side by
// side instead of back to back; the winners are combined with a shuffle min-reduction inside the
// 16-lane group.  Later rings deal their (2r+1)^2 rows round-robin over the lanes.  The search is
// latency-bound (a handful of 32-byte L2 sectors per query), so what counts is how many of
// those loads are in flight — with one thread per query a K = 1000 search took 27 us.
template <int MG>
__device__ __forceinline__ void match_coop_body(
    const GridView& g, const DevState* __restrict__ st, const double* __restrict__ q_xyz,
    const float4* __restrict__ q_nrm, const double* __restrict__ mov_xyz, long long K, int rmax,
    int with_distance, long long* __restrict__ nn_idx, double* __restrict__ out,
    unsigned int* __restrict__ unresolved, unsigned int* __restrict__ lin_hist, double cap2,
    const CorrOut& co, const long long gt) {
  const long long qi = gt / MG;
  const int sub = threadIdx.x & (MG - 1);
  pdl_launch_dependents();
  if (qi >= K) return;  // a whole group leaves together
  // the query's coordinates do not depend on the previous kernel: on their way before the wait
  const double px = q_xyz[3 * qi + 0], py = q_xyz[3 * qi + 1], pz = q_xyz[3 * qi + 2];
  pdl_wait();
  if (st->stop) return;
  const unsigned int gmask = (MG == 32) ? 0xffffffffu : (((1u << MG) - 1u) << ((threadIdx.x & 31) & ~(MG - 1)));
  const Rigid Tinv = st->Tinv;
  double qx, qy, qz;
  rigid_apply(Tinv, px, py, pz, qx, qy, qz);
  const int cx = cell_coord(qx, g.ox, g.inv_h, g.nx);
  const int cy = cell_coord(qy, g.oy, g.inv_h, g.ny);
  const int cz = cell_coord(qz, g.oz, g.inv_h, g.nz);
  const uint32_t* __restrict__ cs = g.cell_start;
  // the normal is only needed at the very end: start its (cold) line on the way now
  if (with_distance && sub == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(q_nrm + qi));
  double best = kInf;
  long long bidx = -1;
  uint32_t bpos = 0;
  bool resolved = false;
  if (co.warm) {
    const uint32_t p = co.nn_pos[qi];
    if ((long long)p < g.n_points) consider(g.recs[p], p, qx, qy, qz, best, bidx, bpos);
  }
  // Sphere scan: once ANY point is known (its squared distance is `best`), the nearest neighbour
  // lies inside the sphere of that radius around the query, i.e. in the cells of the box
  // [q - R, q + R] clipped to the grid; each x-row of the box is pruned by its distance to the
  // query and narrowed to the chord of the sphere.  With a good bound (the previous iteration's
  // neighbour) that is 1-4 rows of 1-2 cells instead of the 27 cells of ring 1; for a query
  // outside the cloud's box (partial overlap) it is the small cap of the sphere that reaches into
  // the grid instead of rings expanding through empty space.  rs = radius of the cube of cells
  // already scanned around the query's cell (0: none).  Returns false (nothing done) when the box
  // is too large to be worth it: the bound is poor, another ring will improve it.
  // The row bounds are evaluated in float, in CELL units, with margins that keep every bound on
  // the safe side (a row is only skipped / narrowed when it certainly holds nothing nearer than
  // `best`); the distances themselves stay float64.  (Per-row float64 bounds, a float64 sqrt, two
  // float64 floor conversions and an integer division were half of the first iteration's
  // instructions, profiles/r2_README.md.)
  const float fqx = (float)((qx - g.ox) * g.inv_h), fqy = (float)((qy - g.oy) * g.inv_h),
              fqz = (float)((qz - g.oz) * g.inv_h);
  // float32 error of a cell coordinate (a query may lie far outside the grid) + cell faces vs the
  // floor() that assigned the points
  const float marg = 1e-3f + 4e-7f * fmaxf(fmaxf(fabsf(fqx), fabsf(fqy)),
                                           fmaxf(fabsf(fqz), (float)max(g.nx, max(g.ny, g.nz))));
  const double inv_h2 = g.inv_h * g.inv_h;
  auto sphere_scan = [&](const int rs, const int max_rows) -> bool {
    const float Rc = sqrtf(__double2float_ru(best * inv_h2)) * (1.0f + 1e-6f) + marg;  // radius in cells, rounded up
    const int ya = min(max(__float2int_rd(fqy - Rc), 0), g.ny - 1), yb = min(max(__float2int_rd(fqy + Rc), 0), g.ny - 1);
    const int za = min(max(__float2int_rd(fqz - Rc), 0), g.nz - 1), zb = min(max(__float2int_rd(fqz + Rc), 0), g.nz - 1);
    const int nyb = yb - ya + 1;
    const long long rows = (long long)nyb * (zb - za + 1);
    if (rows > max_rows) return false;
    // (yr, zr) walk the box with stride MG, kept incrementally (no division per row)
    int zr = sub / nyb, yr = sub - zr * nyb;
    float limc = __double2float_ru(best * (1.0 + 1e-12) * inv_h2);  // strictly farther rows only: ties are still visited
    double best_seen = best;
    for (int t = sub; t < (int)rows; t += MG, yr += MG) {
      while (yr >= nyb) {
        yr -= nyb;
        ++zr;
      }
      const int yy = ya + yr, zz = za + zr;
      if (best != best_seen) {
        best_seen = best;
        limc = __double2float_ru(best * (1.0 + 1e-12) * inv_h2);
      }
      const float by = fmaxf(fabsf(fqy - ((float)yy + 0.5f)) - 0.5f - marg, 0.0f);
      const float bz = fmaxf(fabsf(fqz - ((float)zz + 0.5f)) - 0.5f - marg, 0.0f);
      const float lb = (by * by + bz * bz) * (1.0f - 1e-6f);  // rounded down
      if (lb > limc) continue;
      const float xr = sqrtf(limc - lb) * (1.0f + 1e-6f) + marg;
      const int xs = max(__float2int_rd(fqx - xr), 0), xe = min(__float2int_rd(fqx + xr), g.nx - 1);
      if (xs > xe) continue;  // the chord lies outside the grid
      const uint32_t row = ((uint32_t)zz * (uint32_t)g.ny + (uint32_t)yy) * (uint32_t)g.nx;  // < 2^25 cells
      if (rs > 0 && abs(yy - cy) <= rs && abs(zz - cz) <= rs) {
        // cells cx - rs .. cx + rs of this row were scanned by the rings
        const int le = min(xe, cx - rs - 1), rb = max(xs, cx + rs + 1);
        if (xs <= le) scan_range(g.recs, cs[row + xs], cs[row + le + 1], qx, qy, qz, best, bidx, bpos);
        if (rb <= xe) scan_range(g.recs, cs[row + rb], cs[row + xe + 1], qx, qy, qz, best, bidx, bpos);
      } else {
        scan_range(g.recs, cs[row + xs], cs[row + xe + 1], qx, qy, qz, best, bidx, bpos);
      }
    }
#pragma unroll
    for (int o = MG / 2; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(gmask, best, o, MG);
      const long long oi = __shfl_xor_sync(gmask, bidx, o, MG);
      const uint32_t op = __shfl_xor_sync(gmask, bpos, o, MG);
      if (od < best || (od == best && oi >= 0 && (bidx < 0 || oi < bidx))) {
        best = od;
        bidx = oi;
        bpos = op;
      }
    }
    return true;
  };
  const bool use_sphere = (cap2 < 0.0) && co.sphere;
  // Warm start: finish inside the sphere of the previous neighbour right away when that sphere
  // is small (the steady state: 1-4 rows).  After a large update of the transform (second
  // iteration of a registration) the old neighbour is a poor bound — several cells — while the
  // true one is almost surely in the query's own row: ring 1 first, it prunes with the bound it
  // has and leaves a much smaller sphere to the scan after it.
  if (use_sphere && best < kInf && sphere_scan(0, 4 * MG)) resolved = true;
  for (int r = 1; !resolved; ++r) {
    const int x0 = cx - r, x1 = cx + r;
    const int xa = max(x0, 0), xb = min(x1, g.nx - 1);
    if (r == 1) {
      // Ring 1 in two steps.  (1) the query's own x-row, one cell per lane; (2) the eight
      // neighbouring rows, each skipped (or narrowed in x) when the distance from the query to
      // the row / cell already exceeds the best distance of step 1 — the nearest neighbour
      // is usually in the own row, so most of the 27 cells are never read.
      // (Requesting every cell-table entry step 2 might need before step 1's records — to shorten
      // the chain of dependent round trips — was measured 10 % SLOWER: the kernel is bound by
      // issue slots as much as by latency, and 8 extra loads per lane cost more than the round
      // trip they save; profiles/README.md.)
      constexpr int NR = (8 + MG - 1) / MG;  // rows per lane in step 2
      // distances from the query to the faces of its own cell (>= 0 up to rounding)
      const double fxl = fmax(qx - (g.ox + cx * g.h), 0.0), fxh = fmax((g.ox + (cx + 1) * g.h) - qx, 0.0);
      const double fyl = fmax(qy - (g.oy + cy * g.h), 0.0), fyh = fmax((g.oy + (cy + 1) * g.h) - qy, 0.0);
      const double fzl = fmax(qz - (g.oz + cz * g.h), 0.0), fzh = fmax((g.oz + (cz + 1) * g.h) - qz, 0.0);
#pragma unroll
      for (int t = sub; t < 3 || t == sub; t += MG) {  // one pass for MG >= 4, two for MG = 2
        const int x = cx - 1 + t;
        bool own = t < 3 && x >= 0 && x < g.nx;
        // with a warm-start bound the two side cells of the own row are usually out of reach
        const double bx = (t == 0) ? fxl : ((t == 2) ? fxh : 0.0);
        if (bx * bx > best * (1.0 + 1e-12)) own = false;
        const long long row0 = ((long long)cz * g.ny + cy) * g.nx;
        const uint32_t os = own ? cs[row0 + x] : 0u, oe = own ? cs[row0 + x + 1] : 0u;
        scan_range(g.recs, os, oe, qx, qy, qz, best, bidx, bpos);
        if (MG >= 3) break;
      }
#pragma unroll
      for (int o = MG / 2; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(gmask, best, o, MG);
        const long long oi = __shfl_xor_sync(gmask, bidx, o, MG);
        const uint32_t op = __shfl_xor_sync(gmask, bpos, o, MG);
        if (od < best || (od == best && oi >= 0 && (bidx < 0 || oi < bidx))) {
          best = od;
          bidx = oi;
          bpos = op;
        }
      }
      const double lim = best * (1.0 + 1e-12);  // strictly farther only: ties are still visited
      uint32_t rs[NR], re[NR];
#pragma unroll
      for (int u = 0; u < NR; ++u) {
        rs[u] = re[u] = 0;
        const int t = sub + u * MG;
        if (t >= 8) continue;
        const int tt = t + (t >= 4 ? 1 : 0);  // 0..8 without the centre (4)
        const int dz = tt / 3 - 1, dy = tt % 3 - 1;
        const int y = cy + dy, z = cz + dz;
        if (y < 0 || y >= g.ny || z < 0 || z >= g.nz) continue;
        const double by = (dy < 0) ? fyl : ((dy > 0) ? fyh : 0.0);
        const double bz = (dz < 0) ? fzl : ((dz > 0) ? fzh : 0.0);
        const double lb = by * by + bz * bz;
        if (lb > lim) continue;
        int xs = xa, xe = xb;
        if (x0 >= 0 && lb + fxl * fxl > lim) xs = cx;
        if (x1 < g.nx && lb + fxh * fxh > lim) xe = cx;
        const long long row = ((long long)z * g.ny + y) * g.nx;
        rs[u] = cs[row + xs];
        re[u] = cs[row + xe + 1];
      }
#pragma unroll
      for (int u = 0; u < NR; ++u) scan_range(g.recs, rs[u], re[u], qx, qy, qz, best, bidx, bpos);
    } else {
      const int side = 2 * r + 1, items = side * side;
      // (dy, dz) walk the (2r+1)^2 rows with stride MG; kept incrementally — two integer
      // divisions by the run-time `side` per row were a third of the instructions of this loop
      int dzr = sub / side, dyr = sub - dzr * side;
      for (int t = sub; t < items; t += MG, dyr += MG) {
        while (dyr >= side) {
          dyr -= side;
          ++dzr;
        }
        const int dz = dzr - r, dy = dyr - r;
        const int y = cy + dy, z = cz + dz;
        if (y < 0 || y >= g.ny || z < 0 || z >= g.nz) continue;
        const long long row = ((long long)z * g.ny + y) * g.nx;
        const bool full = dy == -r || dy == r || dz == -r || dz == r;
        if (full) {
          scan_range(g.recs, cs[row + xa], cs[row + xb + 1], qx, qy, qz, best, bidx, bpos);
        } else {
          if (x0 >= 0) scan_range(g.recs, cs[row + x0], cs[row + x0 + 1], qx, qy, qz, best, bidx, bpos);
          if (x1 < g.nx) scan_range(g.recs, cs[row + x1], cs[row + x1 + 1], qx, qy, qz, best, bidx, bpos);
        }
      }
    }
    // min-reduction of (d2, idx) over the 16 lanes of the group; every lane ends with the result
#pragma unroll
    for (int o = MG / 2; o > 0; o >>= 1) {
      const double od = __shfl_xor_sync(gmask, best, o, MG);
      const long long oi = __shfl_xor_sync(gmask, bidx, o, MG);
      const uint32_t op = __shfl_xor_sync(gmask, bpos, o, MG);
      if (od < best || (od == best && oi >= 0 && (bidx < 0 || oi < bidx))) {
        best = od;
        bidx = oi;
        bpos = op;
      }
    }
    const int y0 = cy - r, y1 = cy + r, z0 = cz - r, z1 = cz + r;
    double guard = kInf;
    if (x0 > 0) guard = fmin(guard, qx - (g.ox + x0 * g.h));
    if (x1 < g.nx - 1) guard = fmin(guard, (g.ox + (x1 + 1) * g.h) - qx);
    if (y0 > 0) guard = fmin(guard, qy - (g.oy + y0 * g.h));
    if (y1 < g.ny - 1) guard = fmin(guard, (g.oy + (y1 + 1) * g.h) - qy);
    if (z0 > 0) guard = fmin(guard, qz - (g.oz + z0 * g.h));
    if (z1 < g.nz - 1) guard = fmin(guard, (g.oz + (z1 + 1) * g.h) - qz);
    if (guard >= kInf) {
      resolved = true;
      break;
    }
    guard -= 1e-9 * g.h;
    if (guard > 0.0 && best <= guard * guard) {
      resolved = true;
      break;
    }
    if (cap2 >= 0.0 && (best < cap2 || (guard > 0.0 && guard * guard >= cap2))) {
      resolved = true;  // overlap filter: the side of the bound is decided (see grid_nn)
      break;
    }
    // Nothing within the 27 cells (first iteration of a registration: the clouds are still apart
    // by several cells, typically along the surface normal).  A cube grown ring by ring meets a
    // sheet-like surface with a whole FACE at once — hundreds of candidates at ring r, thousands
    // of cell-table reads before it.  Probe outwards along the three axes instead (six cells per
    // step): a surface at distance D crosses one of the axes within sqrt(3) D, the first point
    // found bounds the search, and the sphere scan below finishes it.
    if (use_sphere && r == 1 && best == kInf) {
      // The y and z probes read three x-neighbouring cells (one contiguous record range, the same
      // two cell-table loads): a sheet sampled at ~3 points per cell has holes, and a probe that
      // slips through one runs on until another axis meets the surface ten times farther out —
      // 5 % of the queries of the C3 pair, i.e. a third of the warps, with single-cell probes.
      // The lanes only vote per step; the (distance, index, position) reduction runs once, after
      // the step that found something.
      for (int s2 = 2; s2 <= 96; ++s2) {
        bool any_inside = false;
        for (int t = sub; t < 6; t += MG) {
          const int axis = t >> 1, off = (t & 1) ? s2 : -s2;
          const int x = cx + (axis == 0 ? off : 0), y = cy + (axis == 1 ? off : 0), z = cz + (axis == 2 ? off : 0);
          if (x < 0 || x >= g.nx || y < 0 || y >= g.ny || z < 0 || z >= g.nz) continue;
          any_inside = true;
          const long long row = ((long long)z * g.ny + y) * g.nx;
          const int xl = (axis == 0) ? x : max(x - 1, 0), xh = (axis == 0) ? x : min(x + 1, g.nx - 1);
          scan_range(g.recs, cs[row + xl], cs[row + xh + 1], qx, qy, qz, best, bidx, bpos);
        }
        const bool found = __any_sync(gmask, best < kInf);
        const bool inside = __any_sync(gmask, any_inside);
        if (found) {
#pragma unroll
          for (int o = MG / 2; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(gmask, best, o, MG);
            const long long oi = __shfl_xor_sync(gmask, bidx, o, MG);
            const uint32_t op = __shfl_xor_sync(gmask, bpos, o, MG);
            if (od < best || (od == best && oi >= 0 && (bidx < 0 || oi < bidx))) {
              best = od;
              bidx = oi;
              bpos = op;
            }
          }
          break;
        }
        if (!inside) break;
      }
    }
    // a point is known now: finish inside its sphere instead of growing the cube ring by ring
    // (best is uniform across the group after the reduction, so the whole group takes one branch)
    if (use_sphere && best < kInf && sphere_scan(r, 64 * MG)) {  // ~15 instructions per pruned row: cheaper than the next rings up to there
      resolved = true;
      break;
    }
    if (r >= rmax) break;
  }
  if (sub != 0) return;
  if (co.nn_pos) co.nn_pos[qi] = resolved ? bpos : 0xffffffffu;
  if (!resolved) {
    const unsigned int slot = atomicAdd(&unresolved[K], 1u);
    unresolved[slot] = (unsigned int)qi;
    return;
  }
  nn_idx[qi] = bidx;
  if (with_distance) {
    const float4 nr = q_nrm[qi];
    // the winner's record was read a moment ago by a lane of this warp: same coordinates as
    // mov_xyz[bidx], but from L1/L2 instead of a cold line
    const Rec m = g.recs[bpos];
    const double d = plane_distance_rec(st->T, m, px, py, pz, nr);
    out[qi] = d;
    lin_hist_add(st, lin_hist, effective_planarity(co, st->T, qi, bidx, nr), d, co.binstore, co.bin_cap, qi);
    store_matched(co, qi, m.x, m.y, m.z);
  } else {
    out[qi] = best;
  }
}

template <int MG>
__global__ void __launch_bounds__(128)
    k_match_grid_coop(GridView g, const DevState* __restrict__ st, const double* __restrict__ q_xyz,
                      const float4* __restrict__ q_nrm, const double* __restrict__ mov_xyz,
                      long long K, int rmax, int with_distance, long long* __restrict__ nn_idx,
                      double* __restrict__ out, unsigned int* __restrict__ unresolved,
                      unsigned int* __restrict__ lin_hist, double cap2, CorrOut co) {
  match_coop_body<MG>(g, st, q_xyz, q_nrm, mov_xyz, K, rmax, with_distance, nn_idx, out, unresolved,
                      lin_hist, cap2, co, blockIdx.x * (long long)blockDim.x + threadIdx.x);
}

// Batched form: blockIdx.y is the pair, everything else comes from its descriptor.  The ring
// expansion runs to completion (no brute-force hand-over inside a batch).
struct BatchMatchArgs {
  const PairDev* pairs;
  const DevState* state;
  const double* q_xyz;
  const float4* q_nrm;
  long long* nn_idx;
  double* dist;
  unsigned int* lin_hist;
  unsigned int* binstore;
  int bin_cap;
  double* m_xyz;
  uint32_t* nn_pos;
  int warm;
  int sphere;
};
template <int MG>
__global__ void __launch_bounds__(128) k_match_batch(BatchMatchArgs a) {
  const PairDev pd = a.pairs[blockIdx.y];
  const long long gt = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (gt / MG >= pd.K) return;
  const long long q = pd.q_off;
  const CorrOut co{a.binstore + (size_t)blockIdx.y * LH_BINS * a.bin_cap, a.bin_cap, a.m_xyz + 3 * q, a.nn_pos + q, a.warm, a.sphere,
                   nullptr, nullptr, -1.0};
  match_coop_body<MG>(pd.gmov, a.state + blockIdx.y, a.q_xyz + 3 * q, a.q_nrm + q, nullptr, pd.K, 1 << 30, 1,
                      a.nn_idx + q, a.dist + q, nullptr, a.lin_hist + (size_t)blockIdx.y * (LH_BINS + 2), -1.0,
                      co, gt);
}

// Overlap filter of a batch (PointCloud.select_in_range, pointcloud.py:149-171): every fixed point
// of every pair is a query, read in place from the concatenated clouds.  The grid is flat over the
// batch's fixed points (pairs are ragged: a grid sized by the largest pair would idle most blocks);
// a query group finds its pair by bisection of the offsets.  The search only decides on which side
// of cap2 = max_overlap_distance^2 the nearest distance lies (grid_nn); without a brute-force
// hand-over a query far outside the movable box still ends once every unexplored cell lies beyond
// the bound, after about max_overlap_distance / h rings.
struct BatchOverlapArgs {
  const PairDev* pairs;
  const long long* fix_off;  // n_pairs + 1
  int n_pairs;
  const DevState* state;
  const double* fix_xyz;
  long long total;
  long long* nn;
  double* d2;
  uint32_t* flag;
  double cap2;
};
template <int MG>
__global__ void __launch_bounds__(128) k_overlap_batch(BatchOverlapArgs a) {
  const long long gt = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long g = gt / MG;
  if (g >= a.total) return;  // a whole group leaves together
  int lo = 0, hi = a.n_pairs - 1;  // the last pair that starts at or before g
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (a.fix_off[mid] <= g) lo = mid;
    else hi = mid - 1;
  }
  const long long f = a.fix_off[lo];
  const GridView gv = a.pairs[lo].gmov;
  const CorrOut co{nullptr, 0, nullptr, nullptr, 0, 0, nullptr, nullptr, -1.0};
  match_coop_body<MG>(gv, a.state + lo, a.fix_xyz + 3 * f, nullptr, nullptr, a.fix_off[lo + 1] - f, 1 << 30, 0,
                      a.nn + f, a.d2 + f, nullptr, nullptr, a.cap2, co, (g - f) * MG + (gt & (MG - 1)));
  // lane 0 of the group stored the distance above
  if ((threadIdx.x & (MG - 1)) == 0) a.flag[g] = (a.d2[g] < a.cap2) ? 1u : 0u;  // strict, as cKDTree's bound
}

// kept list: position scan[g] of the batch-wide list holds g
__global__ void __launch_bounds__(256)
    k_overlap_compact(const uint32_t* __restrict__ flag, const uint32_t* __restrict__ scan, long long total,
                      uint32_t* __restrict__ kept) {
  const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (g < total && flag[g]) kept[scan[g]] = (uint32_t)g;
}

// per pair: m = kept count, its list starts at scan[fix_off]; K = min(correspondences, m).  A pair
// that keeps nothing gets K = 0 and a raised stop flag, so every later kernel leaves it alone.
__global__ void k_overlap_pairs(PairDev* __restrict__ pairs, DevState* __restrict__ state,
                                const long long* __restrict__ fix_off, const uint32_t* __restrict__ scan,
                                int n_pairs, long long correspondences) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  const long long s0 = scan[fix_off[i]], m = (long long)scan[fix_off[i + 1]] - s0;
  pairs[i].n_cand = m;
  pairs[i].kept_off = s0;
  pairs[i].K = min(correspondences, m);
  if (m == 0) state[i].stop = 2;
}

// ------------------------------------------------------------------------------------------
// brute-force engine (TMA staged)
// ------------------------------------------------------------------------------------------
constexpr int BF_TILE = kBfTile;  // float4 points per stage = 32 KB
constexpr int BF_STAGES = 3;    // 96 KB of shared memory in flight per block, two blocks per SM
constexpr int BF_THREADS = 256; // 8 warps
constexpr int BF_QPW = 8;       // queries per warp
constexpr int BF_QPB = BF_QPW * (BF_THREADS / 32);

struct BfPartial {
  double d2;
  long long idx;
};

// float32 filter margin.  Centred float32 coordinates carry a per-coordinate error
// eta <= 2^-23 (|a|_inf + R) * 1.5 (a = centred query, R = cloud half-extent); the float32
// squared distance then differs from the true one by at most e(d) = 4 eta sqrt(d) + 1e-6 d +
// 4 eta^2.  A point is re-evaluated in float64 iff d32 <= best32 + 2.5 e(best32), which the
// true nearest neighbour always satisfies.  The threshold is evaluated in float32 with its
// constants rounded up (cA = 10 eta, cC = 10 eta^2, 4e-6 >= 2.5e-6 + rounding).
__device__ __forceinline__ float bf_threshold(float best32, float cA, float cC) {
  return fmaf(cA, sqrtf(best32), fmaf(4.0e-6f, best32, best32)) + cC;
}

__global__ void __launch_bounds__(BF_THREADS, 2)
    k_bf_nn(const float4* __restrict__ mov_f4, const double* __restrict__ mov_xyz, long long n_mov,
            long long n_pad, double cx, double cy, double cz, double radius,
            const DevState* __restrict__ st,
            const double* __restrict__ q_xyz, const unsigned int* __restrict__ qlist,
            const unsigned int* __restrict__ qcount_ptr, long long q_total, int tiles_per_chunk,
            BfPartial* __restrict__ partials) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float4* tiles = reinterpret_cast<float4*>(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)BF_STAGES * BF_TILE * sizeof(float4));
  uint64_t* empty = full + BF_STAGES;
  double* q64 = reinterpret_cast<double*>(empty + BF_STAGES);  // BF_QPB x 3

  const long long nq = qlist ? (long long)(*qcount_ptr) : q_total;
  const long long n_groups = (nq + BF_QPB - 1) / BF_QPB;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long n_tiles = n_pad / BF_TILE;
  const long long tile0 = (long long)blockIdx.y * tiles_per_chunk;
  const long long tile1 = min(tile0 + tiles_per_chunk, n_tiles);
  if (tile0 >= tile1 || n_groups == 0 || st->stop) return;
  const int my_tiles = (int)(tile1 - tile0);
  const Rigid Tinv = st->Tinv;

  if (threadIdx.x == 0) {
    for (int s = 0; s < BF_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], BF_THREADS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  uint32_t it_base = 0;  // tiles consumed so far by this block (across query groups)
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    // ---- queries of this warp: move into the movable frame, centre, round to float32
    float ax[BF_QPW], ay[BF_QPW], az[BF_QPW], best32[BF_QPW], thr[BF_QPW], cA[BF_QPW], cC[BF_QPW];
    double best64[BF_QPW];
    int bidx[BF_QPW];
#pragma unroll
    for (int k = 0; k < BF_QPW; ++k) {
      const long long qi = grp * BF_QPB + warp * BF_QPW + k;
      double mx = 0, my = 0, mz = 0;
      if (qi < nq) {
        const long long q = qlist ? (long long)qlist[qi] : qi;
        rigid_apply(Tinv, q_xyz[3 * q + 0], q_xyz[3 * q + 1], q_xyz[3 * q + 2], mx, my, mz);
      }
      if (lane == 0) {
        q64[(warp * BF_QPW + k) * 3 + 0] = mx;
        q64[(warp * BF_QPW + k) * 3 + 1] = my;
        q64[(warp * BF_QPW + k) * 3 + 2] = mz;
      }
      const double a0 = mx - cx, a1 = my - cy, a2 = mz - cz;
      ax[k] = (float)a0;
      ay[k] = (float)a1;
      az[k] = (float)a2;
      const double eta = 1.1920929e-7 * (fmax(fabs(a0), fmax(fabs(a1), fabs(a2))) + radius) * 1.5;
      cA[k] = nextafterf((float)(10.0 * eta), 3.0e38f);
      cC[k] = nextafterf((float)(10.0 * eta * eta), 3.0e38f);
      best32[k] = 3.0e38f;
      thr[k] = 3.0e38f;
      best64[k] = kInf;
      bidx[k] = -1;
    }
    __syncwarp();

    // ---- producer prologue: fill the ring
    if (threadIdx.x == 0) {
      for (int t = 0; t < min(BF_STAGES, my_tiles); ++t) {
        const uint32_t g_it = it_base + t;
        const int s = g_it % BF_STAGES;
        if (g_it >= BF_STAGES) mbar_wait(&empty[s], ((g_it / BF_STAGES) - 1) & 1);
        mbar_expect_tx(&full[s], BF_TILE * sizeof(float4));
        tma_load_1d(tiles + (size_t)s * BF_TILE, mov_f4 + (tile0 + t) * BF_TILE,
                    BF_TILE * sizeof(float4), &full[s]);
      }
    }

    for (int t = 0; t < my_tiles; ++t) {
      const uint32_t g_it = it_base + t;
      const int s = g_it % BF_STAGES;
      mbar_wait(&full[s], (g_it / BF_STAGES) & 1);
      const float4* __restrict__ tp = tiles + (size_t)s * BF_TILE;
      const long long base = (tile0 + t) * BF_TILE;
      unsigned int improved = 0;  // bit k: this lane lowered best32[k] in this tile
#pragma unroll 2
      for (int j = lane; j < BF_TILE; j += 32) {
        const float4 p = tp[j];  // conflict-free LDS.128
        float dk[BF_QPW];
        bool hit = false;
#pragma unroll
        for (int k = 0; k < BF_QPW; ++k) {
          const float dx = p.x - ax[k], dy = p.y - ay[k], dz = p.z - az[k];
          dk[k] = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
          hit = hit || (dk[k] <= thr[k]);
        }
        if (__builtin_expect(hit, 0)) {
          // rare: exact float64 re-evaluation from the original coordinates
          const long long gi = base + j;
          if (gi < n_mov) {
            const double gx = mov_xyz[3 * gi + 0], gy = mov_xyz[3 * gi + 1], gz = mov_xyz[3 * gi + 2];
#pragma unroll
            for (int k = 0; k < BF_QPW; ++k) {
              if (dk[k] <= thr[k]) {
                const double* qq = &q64[(warp * BF_QPW + k) * 3];
                const double ex = gx - qq[0], ey = gy - qq[1], ez = gz - qq[2];
                const double d64 = ex * ex + ey * ey + ez * ez;
                if (d64 < best64[k] || (d64 == best64[k] && (int)gi < bidx[k])) {
                  best64[k] = d64;
                  bidx[k] = (int)gi;
                }
                if (dk[k] < best32[k]) {
                  best32[k] = dk[k];
                  thr[k] = bf_threshold(dk[k], cA[k], cC[k]);
                  improved |= 1u << k;
                }
              }
            }
          }
        }
      }
      // share the float32 bound across the warp, but only for the queries some lane improved in
      // this tile (after the first tiles that is almost never)
      unsigned int any = improved;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) any |= __shfl_xor_sync(0xffffffffu, any, o);
      if (any) {
#pragma unroll
        for (int k = 0; k < BF_QPW; ++k) {
          if (any & (1u << k)) {
            float m = best32[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (m < best32[k]) {
              best32[k] = m;
              thr[k] = bf_threshold(m, cA[k], cC[k]);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
      // producer: refill this stage with tile t + BF_STAGES once every warp has released it
      if (threadIdx.x == 0 && t + BF_STAGES < my_tiles) {
        mbar_wait(&empty[s], (g_it / BF_STAGES) & 1);
        mbar_expect_tx(&full[s], BF_TILE * sizeof(float4));
        tma_load_1d(tiles + (size_t)s * BF_TILE, mov_f4 + (tile0 + t + BF_STAGES) * BF_TILE,
                    BF_TILE * sizeof(float4), &full[s]);
      }
    }
    it_base += my_tiles;

    // ---- warp-shuffle lexicographic min-reduction of (d64, idx) over the lanes
#pragma unroll
    for (int k = 0; k < BF_QPW; ++k) {
      double d = best64[k];
      int ix = bidx[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, d, o);
        const int oi = __shfl_xor_sync(0xffffffffu, ix, o);
        if (od < d || (od == d && oi >= 0 && (ix < 0 || oi < ix))) {
          d = od;
          ix = oi;
        }
      }
      const long long qi = grp * BF_QPB + warp * BF_QPW + k;
      if (lane == 0 && qi < nq) {
        BfPartial pr;
        pr.d2 = d;
        pr.idx = ix;
        partials[(long long)blockIdx.y * q_total + qi] = pr;
      }
    }
    __syncthreads();  // q64 is reused by the next group
  }
}

__global__ void __launch_bounds__(128)
    k_bf_finalize(const BfPartial* __restrict__ partials, int n_chunks, long long q_total,
                  const unsigned int* __restrict__ qlist, const unsigned int* __restrict__ qcount_ptr,
                  const DevState* __restrict__ st, const double* __restrict__ q_xyz,
                  const float4* __restrict__ q_nrm,
                  const double* __restrict__ mov_xyz, int with_distance,
                  long long* __restrict__ nn_idx, double* __restrict__ out,
                  unsigned int* __restrict__ lin_hist, CorrOut co) {
  const long long nq = qlist ? (long long)(*qcount_ptr) : q_total;
  const long long qi = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (qi >= nq || st->stop) return;
  const Rigid T = st->T;
  double d = kInf;
  long long ix = -1;
  for (int c = 0; c < n_chunks; ++c) {
    const BfPartial p = partials[(long long)c * q_total + qi];
    if (p.idx >= 0 && (p.d2 < d || (p.d2 == d && p.idx < ix) || ix < 0)) {
      d = p.d2;
      ix = p.idx;
    }
  }
  const long long q = qlist ? (long long)qlist[qi] : qi;
  nn_idx[q] = ix;
  if (with_distance) {
    const float4 nr = q_nrm[q];
    const double dd = plane_distance(T, mov_xyz, ix, q_xyz[3 * q + 0], q_xyz[3 * q + 1], q_xyz[3 * q + 2], nr);
    out[q] = dd;
    lin_hist_add(st, lin_hist, effective_planarity(co, T, q, ix, nr), dd, co.binstore, co.bin_cap, q);
    store_matched(co, q, mov_xyz[3 * ix + 0], mov_xyz[3 * ix + 1], mov_xyz[3 * ix + 2]);
  } else {
    out[q] = d;
  }
}

__global__ void __launch_bounds__(256)
    k_gather_queries(const double* __restrict__ fix_xyz, const long long* __restrict__ sel,
                     long long K, double* __restrict__ q_xyz) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K) return;
  const long long j = sel[i];
  q_xyz[3 * i + 0] = fix_xyz[3 * j + 0];
  q_xyz[3 * i + 1] = fix_xyz[3 * j + 1];
  q_xyz[3 * i + 2] = fix_xyz[3 * j + 2];
}

constexpr size_t kBfSmem =
    (size_t)BF_STAGES * BF_TILE * sizeof(float4) + 2 * BF_STAGES * sizeof(uint64_t) +
    (size_t)BF_QPB * 3 * sizeof(double);

}  // namespace

void gather_queries_launch(Ctx& c) {
  c.unresolved_clean = false;  // another K: the counter lives at another address
  c.q_xyz.reserve(3 * std::max<long long>(c.K, 1));
  k_gather_queries<<<(unsigned)((c.K + 255) / 256), 256, 0, c.stream>>>(c.fix_xyz.p, c.sel_idx.p,
                                                                       c.K, c.q_xyz.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

// Slots per histogram bin of the per-bin index store: a few times the mean count of a bin that
// matters (the statistics set spreads over ~2500 of the 4096 bins), so that a distribution which
// narrows several-fold between two iterations still fits; a bin that overflows just sends that
// iteration through the general kernel.
int bin_cap_for(long long K) {
  long long cap = 32;
  while (cap < K / 192 && cap < 2048) cap *= 2;
  return (int)cap;
}
static void reserve_binstore(Ctx& c) {
  c.bin_cap = bin_cap_for(c.K);
  c.binstore.reserve((size_t)LH_BINS * c.bin_cap);
}

// Brute-force pass over either the unresolved list (qlist != nullptr) or all K queries.
static void bf_launch(Ctx& c, bool with_distance, double* out, bool whole_set) {
  if (with_distance) {
    reserve_binstore(c);
    c.m_xyz.reserve(3 * std::max<long long>(c.K, 1));
  }
  // the attribute belongs to the (device-specific) function handle: once per context, not per process
  if (!c.bf_attr_set) {
    SICP_CUDA(cudaFuncSetAttribute(k_bf_nn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBfSmem));
    c.bf_attr_set = true;
  }
  const long long n_tiles = (c.n_mov + BF_TILE - 1) / BF_TILE;
  SICP_REQUIRE(c.mov_f4.cap >= (size_t)n_tiles * BF_TILE, SICP_ERR_STATE,
               "float4 copy not padded to the brute-force tile");
  const long long q_total = c.K;
  // grid: x = query groups (grid-stride), y = point chunks
  long long groups_hint = whole_set ? (c.K + BF_QPB - 1) / BF_QPB : 4;
  int gx = (int)std::min<long long>(std::max<long long>(groups_hint, 1), 4096);
  long long want_blocks = 2ll * c.num_sms;
  int n_chunks = (int)std::min<long long>(std::max<long long>(want_blocks / gx, 1), n_tiles);
  int tiles_per_chunk = (int)((n_tiles + n_chunks - 1) / n_chunks);
  n_chunks = (int)((n_tiles + tiles_per_chunk - 1) / tiles_per_chunk);
  c.bf_scratch.reserve((size_t)n_chunks * q_total * sizeof(BfPartial));
  BfPartial* partials = reinterpret_cast<BfPartial*>(c.bf_scratch.p);
  const unsigned int* qlist = whole_set ? nullptr : c.unresolved.p;
  const unsigned int* qcount = whole_set ? nullptr : c.unresolved.p + c.K;
  dim3 grid(gx, n_chunks);
  k_bf_nn<<<grid, BF_THREADS, kBfSmem, c.stream>>>(
      c.mov_f4.p, c.mov_xyz.p, c.n_mov, n_tiles * BF_TILE, c.mov_center[0], c.mov_center[1],
      c.mov_center[2], c.mov_radius, c.dev_state.p, c.q_xyz.p, qlist, qcount, q_total,
      tiles_per_chunk,
      partials);
  k_bf_finalize<<<(unsigned)((q_total + 127) / 128), 128, 0, c.stream>>>(
      partials, n_chunks, q_total, qlist, qcount, c.dev_state.p, c.q_xyz.p, c.q_nrm.p, c.mov_xyz.p,
      with_distance ? 1 : 0, c.nn_idx.p, out, with_distance ? c.lin_hist.p : nullptr,
      with_distance ? CorrOut{c.binstore.p, c.bin_cap, c.m_xyz.p, nullptr, 0, 0, mov_attr_nrm(c), mov_attr_eff(c), c.mov_cos_max}
                    : CorrOut{nullptr, 0, nullptr, nullptr, 0, 0, nullptr, nullptr, -1.0});
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 2;
}

namespace {
// per pair: sel[i] = rint(linspace(0, n_fix - 1, K)) (PointCloud.select_n_points, k_select_n in
// capi.cu) and the gather of the selected fixed points, in one launch for the whole batch.  With
// the overlap filter (kept != null) the linspace runs over the pair's kept list instead:
// sel[i] = kept[rint(linspace(0, m - 1, K))[i]], m = the pair's kept count.
__global__ void __launch_bounds__(256)
    k_select_gather_batch(const PairDev* __restrict__ pairs, const double* __restrict__ fix_xyz, int away,
                          const uint32_t* __restrict__ kept, long long* __restrict__ sel, double* __restrict__ q_xyz) {
  const PairDev pd = pairs[blockIdx.y];
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= pd.K) return;
  const long long m = pd.n_cand, n = pd.K;
  long long j = i;
  if (n < m) {
    const double step = (n > 1) ? (double)(m - 1) / (double)(n - 1) : 0.0;
    const double y = (i == n - 1 && n > 1) ? (double)(m - 1) : (double)i * step;
    j = (long long)(away ? round(y) : rint(y));
  }
  if (kept) j = (long long)kept[pd.kept_off + j] - pd.fix_off;
  sel[pd.q_off + i] = j;
  const double* __restrict__ src = fix_xyz + 3 * (pd.fix_off + j);
  double* __restrict__ dst = q_xyz + 3 * (pd.q_off + i);
  dst[0] = src[0];
  dst[1] = src[1];
  dst[2] = src[2];
}
}  // namespace

void batch_select_gather_launch(Ctx& c, Batch& b, long long correspondences, int round_away, bool overlap) {
  (void)correspondences;
  k_select_gather_batch<<<dim3((unsigned)((b.Kmax + 255) / 256), b.n_pairs), 256, 0, c.stream>>>(
      b.pairs.p, b.fix_xyz.p, round_away, overlap ? b.ov_kept.p : nullptr, b.sel_idx.p, b.q_xyz.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

void batch_overlap_launch(Ctx& c, Batch& b, long long correspondences, double max_dist) {
  const long long total = b.total_fix;
  b.ov_nn.reserve(total);
  b.ov_d2.reserve(total);
  b.ov_flag.reserve(total);
  b.ov_scan.reserve(total + 1);
  b.ov_kept.reserve(total);
  BatchOverlapArgs a;
  a.pairs = b.pairs.p;
  a.fix_off = b.fix_off.p;
  a.n_pairs = b.n_pairs;
  a.state = b.state.p;
  a.fix_xyz = b.fix_xyz.p;
  a.total = total;
  a.nn = b.ov_nn.p;
  a.d2 = b.ov_d2.p;
  a.flag = b.ov_flag.p;
  a.cap2 = max_dist * max_dist;
  // lanes per query: 16 while few queries are in flight, else 8 (with 4 or 2 lanes the search body
  // spills a few registers in this kernel)
  const int mg = (total <= 16384) ? 16 : 8;
  const unsigned blocks = (unsigned)((total * mg + 127) / 128);
  if (mg == 8) k_overlap_batch<8><<<blocks, 128, 0, c.stream>>>(a);
  else k_overlap_batch<16><<<blocks, 128, 0, c.stream>>>(a);
  SICP_CUDA(cudaGetLastError());
  scan_u32(c, b.ov_flag.p, total, b.ov_block_sums, b.ov_scan.p);
  k_overlap_compact<<<(unsigned)((total + 255) / 256), 256, 0, c.stream>>>(b.ov_flag.p, b.ov_scan.p, total, b.ov_kept.p);
  k_overlap_pairs<<<(b.n_pairs + 127) / 128, 128, 0, c.stream>>>(b.pairs.p, b.state.p, b.fix_off.p, b.ov_scan.p,
                                                                  b.n_pairs, correspondences);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 3;
}

void batch_match_launch(Ctx& c, Batch& b, bool warm) {
  BatchMatchArgs a;
  a.pairs = b.pairs.p;
  a.state = b.state.p;
  a.q_xyz = b.q_xyz.p;
  a.q_nrm = b.q_nrm.p;
  a.nn_idx = b.nn_idx.p;
  a.dist = b.dist.p;
  a.lin_hist = b.lin_hist.p;
  a.binstore = b.binstore.p;
  a.bin_cap = b.bin_cap;
  a.m_xyz = b.m_xyz.p;
  a.nn_pos = b.nn_pos.p;
  a.warm = warm ? 1 : 0;
  a.sphere = c.sphere_scan;
  // lanes per query as in the single-pair launch, by the number of queries in flight
  const long long total = b.Kmax * b.n_pairs;
  int mg = c.match_group;
  if (mg == 0 || mg == 1) mg = (total <= 16384) ? 16 : ((total <= 65536) ? 8 : 4);
  const dim3 grid((unsigned)((b.Kmax * mg + 127) / 128), b.n_pairs);
  // programmatically dependent on the previous iteration's k_rs_batch (both kernels wait before
  // they touch anything the other writes; the pair descriptors are static)
  const bool pdl = c.pdl != 0;
  if (mg == 2) launch_kernel(k_match_batch<2>, grid, dim3(128), 0, c.stream, pdl, a);
  else if (mg == 4) launch_kernel(k_match_batch<4>, grid, dim3(128), 0, c.stream, pdl, a);
  else if (mg == 8) launch_kernel(k_match_batch<8>, grid, dim3(128), 0, c.stream, pdl, a);
  else launch_kernel(k_match_batch<16>, grid, dim3(128), 0, c.stream, pdl, a);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

void match_launch(Ctx& c, bool with_distance, double* out_d2, cudaEvent_t mid, bool allow_bf, double cap2, bool in_loop) {
  const long long K = c.K;
  // predictor histogram for the reject kernel: zero it if an earlier match filled it and no
  // reject consumed it (the reject kernel itself leaves it zeroed)
  c.lin_hist.reserve(LH_BINS + 2);
  if (with_distance && (c.lin_hist_pending || !c.lin_hist_init)) {
    SICP_CUDA(cudaMemsetAsync(c.lin_hist.p, 0, (LH_BINS + 2) * sizeof(unsigned int), c.stream));
    c.lin_hist_init = true;
  }
  unsigned int* lh = with_distance ? c.lin_hist.p : nullptr;
  c.nn_idx.reserve(K);
  c.dist.reserve(K);
  c.unresolved.reserve(K + 1);
  reserve_binstore(c);
  c.m_xyz.reserve(3 * std::max<long long>(K, 1));
  c.nn_pos.reserve(std::max<long long>(K, 1));
  const bool warm = with_distance && c.warm_start && c.nn_pos_valid && c.nn_pos_K == K;
  const CorrOut co = with_distance ? CorrOut{c.binstore.p, c.bin_cap, c.m_xyz.p, c.nn_pos.p, warm ? 1 : 0, c.sphere_scan,
                                             mov_attr_nrm(c), mov_attr_eff(c), c.mov_cos_max}
                                   : CorrOut{nullptr, 0, nullptr, nullptr, 0, 0, nullptr, nullptr, -1.0};
  if (with_distance) {
    c.nn_pos_valid = (c.nn_engine != SICP_NN_BRUTE) && c.match_group != 1;
    c.nn_pos_K = K;
  }
  double* out = with_distance ? c.dist.p : out_d2;
  if (c.nn_engine == SICP_NN_BRUTE) {
    bf_launch(c, with_distance, out, true);
    if (mid) SICP_CUDA(cudaEventRecord(mid, c.stream));
    if (with_distance) c.lin_hist_pending = true;
    return;
  }
  if (!(in_loop && c.unresolved_clean))
    SICP_CUDA(cudaMemsetAsync(c.unresolved.p + K, 0, sizeof(unsigned int), c.stream));
  c.unresolved_clean = false;  // the caller's reject/solve launch declares it clean again
  const bool pdl = in_loop && c.pdl;
  const bool use_bf = (c.nn_engine == SICP_NN_AUTO) && allow_bf;
  const int rmax = use_bf ? c.grid_max_rings : (1 << 30);
  if (c.match_group == 1) {
    k_match_grid<<<(unsigned)((K + 127) / 128), 128, 0, c.stream>>>(
        c.gmov.view(), c.dev_state.p, c.q_xyz.p, c.q_nrm.p, c.mov_xyz.p, K, rmax,
        with_distance ? 1 : 0, c.nn_idx.p, out, c.unresolved.p, lh, cap2, co);
  } else {
    // lanes per query: 16 while the search is latency-bound (few queries), fewer once there are
    // enough queries to fill the machine and issue slots become the limit
    int mg = c.match_group;
    if (mg == 0) mg = (K <= 16384) ? 16 : ((K <= 65536) ? 8 : 4);
    const long long threads = K * mg;
    const unsigned blocks = (unsigned)((threads + 127) / 128);
#define SICP_LAUNCH_COOP(N)                                                                          \
  launch_kernel(k_match_grid_coop<N>, dim3(blocks), dim3(128), 0, c.stream, pdl, c.gmov.view(),       \
                c.dev_state.p, c.q_xyz.p, c.q_nrm.p, c.mov_xyz.p, K, rmax, with_distance ? 1 : 0, \
                c.nn_idx.p, out, c.unresolved.p, lh, cap2, co)
    if (mg == 2) SICP_LAUNCH_COOP(2);
    else if (mg == 4) SICP_LAUNCH_COOP(4);
    else if (mg == 8) SICP_LAUNCH_COOP(8);
    else SICP_LAUNCH_COOP(16);
#undef SICP_LAUNCH_COOP
  }
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
  if (mid) SICP_CUDA(cudaEventRecord(mid, c.stream));
  if (use_bf) bf_launch(c, with_distance, out, false);
  if (with_distance) c.lin_hist_pending = true;
}

}  // namespace sicp
