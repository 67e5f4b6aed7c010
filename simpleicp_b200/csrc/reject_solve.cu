// reject_solve.cu — one kernel for everything between the match and the next match:
//
//   CorrPts.reject_wrt_planarity                    python/simpleicp/corrpts.py:139-163
//   CorrPts.reject_wrt_point_to_plane_distances     python/simpleicp/corrpts.py:165-188
//   SimpleICPOptimization.estimate_parameters       python/simpleicp/optimization.py:65-124
//   SimpleICPOptimization.estimate_parameter_uncertainties          optimization.py:126-170
//   SimpleICP.__check_convergence_criteria          python/simpleicp/simpleicp.py:355-379
//
// Phases (grid-wide barriers between them; a single block for K <= 4096, a cooperative grid of
// one block per SM otherwise):
//   A  median of d over the planarity survivors   : MSB-first radix select on order-preserving
//      64-bit keys, 11-bit digits, early exit to an in-block bitonic sort once <= 2048 candidates
//      remain.  NumPy semantics: mean of the two middle elements for even n.
//   B  MAD = median(|d - median|) the same way (raw MAD, no 1.4826: corrpts.py:186).
//   C  keep = |d - median| <= 3 MAD; accumulate, over the kept correspondences, the 13 x 13
//      moment matrix M = sum phi phi^T of phi = [n (x) (p', 1), -n.q'] (73 distinct sums).  The
//      residual of EVERY rigid transform is phi . theta(x), so one pass over the data suffices
//      and the non-linear least squares runs on M alone.
//   D  block 0 / warp 0: Levenberg-Marquardt on the exact Euler model to convergence, with the
//      reference's fixed (weight inf) / observed (0 < weight < inf) / free parameter handling.
//   E  residuals at the solution (direct float64 evaluation, reference operation order), their
//      mean / population std, parameter sigmas, stop rule, per-iteration record.
#include <cooperative_groups.h>

#include <algorithm>

#include "ctx.cuh"
#include "reject_solve.cuh"

namespace cg = cooperative_groups;

namespace sicp {

namespace {

constexpr int RS_THREADS = 384;  // 12 warps = 3 accumulation roles x 4 warps
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_BINS = 2048;
constexpr int RS_LEVELS = 6;
constexpr int RS_CAP = 2048;       // candidate buffer (last two slots carry the selected keys)
constexpr int RS_NACC = 26;           // accumulators per role
constexpr int RS_NPART = 3 * RS_NACC; // partial sums per block in phase C

__device__ __constant__ int kShift[RS_LEVELS] = {53, 42, 31, 20, 9, 0};
__device__ __constant__ int kWidth[RS_LEVELS] = {11, 11, 11, 11, 11, 9};

struct Shared {
  unsigned int hist[LH_BINS];  // radix histogram (first RS_BINS) or prefix sums of the predictor histogram
  int lh_i[8];
  unsigned long long sortbuf[RS_CAP];
  double red[RS_WARPS][RS_NACC];
  unsigned int scan_tmp[RS_WARPS];
  // select state (identical in every block)
  unsigned long long prefix;
  unsigned int k;
  unsigned int cnt;
  unsigned int below;
  unsigned int total;
  double bc[8];  // broadcast scalars
  // LM workspace
  double M[13][13];
  double J[13][6];
  double th[13];
  double th_in[13];  // theta of the transform the distances were evaluated at (re-centred model)
  double B[13][7];
  double A[36];
  double g[6];
  double F;
  double tot[RS_NPART];
  double Ak[36];
  double gk[6];
  double delta[6];
  double cholL[21];  // factor published for the per-parameter sigma solves
  int spd;
  unsigned long long stamp[2];
  // in-block refinement of the selected radix bin
  unsigned int h256[256];
  unsigned int rank_acc[RS_THREADS];  // rank_select: partial ranks per candidate
  unsigned long long small[64];
  unsigned long long sel_above;
  unsigned int small_n;
};

// Grid-wide barrier for the cooperative launch (all blocks co-resident).  Hand-written instead of
// cooperative_groups' grid.sync() so that waiting blocks BACK OFF (__nanosleep): while block 0
// runs its serial phases the other 147 blocks would otherwise hammer one L2 line with polling
// loads and slow exactly the block everybody is waiting for.  bar[0] = arrival count,
// bar[1] = generation.  The fence after the wait also invalidates this SM's L1 (gpu-scope
// fence), so data written by other blocks before the barrier is re-read from L2.
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int gen = *(volatile unsigned int*)(bar + 1);
    const unsigned int old = atomicAdd(bar, 1u);
    if (old == nblocks - 1u) {
      *(volatile unsigned int*)bar = 0u;
      __threadfence();
      atomicAdd(bar + 1, 1u);
    } else {
      unsigned int ns = 32;
      while (*(volatile unsigned int*)(bar + 1) == gen) {
        __nanosleep(ns);
        if (ns < 256) ns *= 2;
      }
    }
    __threadfence();
  }
  __syncthreads();
}

template <bool MULTI>
__device__ __forceinline__ void gsync(unsigned int* bar) {
  if (MULTI)
    grid_barrier(bar, gridDim.x);
  else
    __syncthreads();
}

// Find the bin holding rank k in hist (n_bins <= RS_BINS); writes s.k (rank inside the bin),
// s.cnt (bin count), returns the bin through s.below (count below) and the return value.
__device__ __noinline__ unsigned int find_bin(Shared& s, const unsigned int* __restrict__ ghist, int n_bins,
                                 unsigned int k, unsigned int* total_out) {
  // each thread owns a contiguous chunk of 6 bins (384 * 6 = 2304 >= 2048)
  constexpr int PER = (RS_BINS + RS_THREADS - 1) / RS_THREADS;
  const int b0 = threadIdx.x * PER;
  unsigned int v[PER];
  unsigned int sum = 0;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int b = b0 + j;
    v[j] = (b < n_bins) ? ghist[b] : 0u;
    sum += v[j];
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned int incl = sum;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s.scan_tmp[w] = incl;
  __syncthreads();
  unsigned int woff = 0, total = 0;
  for (int i = 0; i < RS_WARPS; ++i) {
    if (i < w) woff += s.scan_tmp[i];
    total += s.scan_tmp[i];
  }
  unsigned int run = woff + incl - sum;  // exclusive prefix of this thread's chunk
  if (k >= run && k < run + sum) {
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      if (k < run + v[j]) {
        s.below = run;
        s.cnt = v[j];
        s.k = k - run;
        s.bc[7] = (double)(b0 + j);
        break;
      }
      run += v[j];
    }
  }
  __syncthreads();
  if (total_out) *total_out = total;
  return (unsigned int)s.bc[7];
}

// In-block refinement: keys[0..cnt) agree on every bit above `shift`; find the k-th smallest
// (0-based) and its successor (`above` when the k-th is the largest).  8-bit radix passes over
// the shared-memory candidates (__syncthreads only) until <= 32 remain, then one warp ranks
// them.  Duplicates are handled (all 64 bits fixed -> every remaining candidate is equal).
__device__ __noinline__ void block_select(Shared& s, const unsigned long long* keys, int cnt, unsigned int k,
                             int shift, unsigned long long above, unsigned long long& klo,
                             unsigned long long& khi) {
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned long long lowmask = (shift >= 64) ? ~0ull : ((1ull << shift) - 1ull);
  unsigned long long prefix = 0;
  int bits = shift;
  unsigned int n = (unsigned int)cnt;
  if (tid == 0) s.sel_above = above;
  __syncthreads();
  while (n > 32u && bits > 0) {
    const int w = min(8, bits), sh = bits - w;
    if (tid < 256) s.h256[tid] = 0;
    __syncthreads();
    for (int t = tid; t < cnt; t += RS_THREADS) {
      const unsigned long long low = keys[t] & lowmask;
      if (bits == shift || (low >> bits) == prefix)
        atomicAdd(&s.h256[(unsigned int)(low >> sh) & ((1u << w) - 1u)], 1u);
    }
    __syncthreads();
    if (tid < 32) {
      unsigned int v[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = s.h256[lane * 8 + j];
        sum += v[j];
      }
      unsigned int incl = sum;
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t2 = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t2;
      }
      unsigned int run = incl - sum;
      if (k >= run && k < run + sum) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (k < run + v[j]) {
            s.k = k - run;
            s.cnt = v[j];
            s.bc[7] = (double)(lane * 8 + j);
            break;
          }
          run += v[j];
        }
      }
    }
    __syncthreads();
    const unsigned int bin = (unsigned int)s.bc[7];
    k = s.k;
    n = s.cnt;
    if (k + 1u >= n) {
      // the successor may lie outside the chosen bin: smallest active key with a larger digit
      unsigned long long mymin = ~0ull;
      for (int t = tid; t < cnt; t += RS_THREADS) {
        const unsigned long long low = keys[t] & lowmask;
        if ((bits == shift || (low >> bits) == prefix) &&
            ((unsigned int)(low >> sh) & ((1u << w) - 1u)) > bin)
          mymin = min(mymin, keys[t]);
      }
      for (int o = 16; o > 0; o >>= 1) mymin = min(mymin, __shfl_xor_sync(0xffffffffu, mymin, o));
      if (lane == 0 && mymin != ~0ull) atomicMin(&s.sel_above, mymin);
    }
    prefix = (prefix << w) | bin;
    bits = sh;
    __syncthreads();
  }
  if (tid == 0) s.small_n = 0;
  __syncthreads();
  if (n > 32u) {
    // all low bits fixed and still more than 32 candidates: they are all the same key
    for (int t = tid; t < cnt; t += RS_THREADS)
      if (((keys[t] & lowmask) >> bits) == prefix) s.small[0] = keys[t];
    __syncthreads();
    klo = s.small[0];
    khi = (k + 1u < n) ? klo : s.sel_above;
    __syncthreads();
    return;
  }
  for (int t = tid; t < cnt; t += RS_THREADS) {
    const unsigned long long low = keys[t] & lowmask;
    if (bits == shift || (low >> bits) == prefix) s.small[atomicAdd(&s.small_n, 1u)] = keys[t];
  }
  __syncthreads();
  if (tid < 32) {
    const unsigned long long key = (lane < (int)n) ? s.small[lane] : ~0ull;
    unsigned int r = 0;
    for (unsigned int j = 0; j < n; ++j) {
      const unsigned long long kj = s.small[j];
      r += (kj < key || (kj == key && (int)j < lane)) ? 1u : 0u;
    }
    if (lane < (int)n && r == k) s.sortbuf[RS_CAP - 2] = key;
    if (lane < (int)n && r == k + 1u) s.sortbuf[RS_CAP - 1] = key;
  }
  __syncthreads();
  klo = s.sortbuf[RS_CAP - 2];
  khi = (k + 1u < n) ? s.sortbuf[RS_CAP - 1] : s.sel_above;
  __syncthreads();
}

// Median of {keyfn(i) : i in S1} with NumPy semantics.  SEL = 0: keys of d; SEL = 1: keys of
// |d - center|.  Result broadcast through s.bc[0] (lower middle) and s.bc[1] (upper middle).
template <bool MULTI, int SEL>
__device__ void radix_median(Shared& s, const RSArgs& a, RSWork wk, double center,
                             unsigned int& n1_out, const int bid = blockIdx.x, const int G = gridDim.x) {
  const long long K = a.K;
  const double minpl = a.stat_minpl;
  unsigned int* ghist_base = wk.hist + (size_t)SEL * RS_LEVELS * RS_BINS;
  unsigned long long prefix = 0;
  unsigned int k = 0, cnt = 0, n1 = 0;
  bool even = false;
  int level = 0;
  for (;; ++level) {
    const int shift = kShift[level], width = kWidth[level];
    const int n_bins = 1 << width;
    for (int b = threadIdx.x; b < RS_BINS; b += RS_THREADS) s.hist[b] = 0;
    __syncthreads();
    for (long long i = bid * (long long)RS_THREADS + threadIdx.x; i < K;
         i += (long long)G * RS_THREADS) {
      if (pl_stat(a.q_nrm[i].w, a.pl_signed) >= minpl) {
        const double v = (SEL == 0) ? a.dist[i] : fabs(a.dist[i] - center);
        const unsigned long long key = f64_to_key(v);
        if (level == 0 || (key >> kShift[level - 1]) == prefix)
          atomicAdd(&s.hist[(unsigned int)(key >> shift) & (n_bins - 1)], 1u);
      }
    }
    __syncthreads();
    unsigned int* gh = ghist_base + (size_t)level * RS_BINS;
    if (MULTI) {
      for (int b = threadIdx.x; b < n_bins; b += RS_THREADS)
        if (s.hist[b]) atomicAdd(&gh[b], s.hist[b]);
      gsync<MULTI>(wk.barrier);
    }
    const unsigned int* src = MULTI ? gh : s.hist;
    unsigned int total = 0;
    if (level == 0) {
      // total = |S1| decides the ranks
      find_bin(s, src, n_bins, 0u, &total);
      n1 = total;
      if (n1 == 0) {
        n1_out = 0;
        return;
      }
      k = (n1 - 1) >> 1;
      even = ((n1 & 1u) == 0u);
    }
    const unsigned int bin = find_bin(s, src, n_bins, k, nullptr);
    k = s.k;
    cnt = s.cnt;
    prefix = (prefix << width) | bin;
    __syncthreads();
    if (cnt <= RS_CAP - 2 || level == RS_LEVELS - 1) break;
  }
  if (bid == 0 && threadIdx.x == 0) {
    wk.phase_t[10 + SEL * 4] = global_timer_ns();
    wk.phase_t[24 + SEL] = (unsigned long long)(level + 1);
    wk.phase_t[26 + SEL] = (unsigned long long)cnt;
  }
  // ---- gather the candidates of the selected bin; track the smallest key above it
  const int shift = kShift[level];
  unsigned long long* cand = wk.cand + (size_t)SEL * RS_CAP;
  unsigned int* ccount = wk.counters + SEL;
  unsigned long long* gmin = wk.minkey + SEL;
  const bool gather = (cnt <= RS_CAP - 2);
  unsigned long long mymin = ~0ull;
  if (!MULTI) {
    if (threadIdx.x == 0) s.total = 0;
    __syncthreads();
  }
  for (long long i = bid * (long long)RS_THREADS + threadIdx.x; i < K;
       i += (long long)G * RS_THREADS) {
    if (pl_stat(a.q_nrm[i].w, a.pl_signed) >= minpl) {
      const double v = (SEL == 0) ? a.dist[i] : fabs(a.dist[i] - center);
      const unsigned long long key = f64_to_key(v);
      const unsigned long long top = key >> shift;
      if (top == prefix) {
        if (gather) {
          if (MULTI)
            cand[atomicAdd(ccount, 1u)] = key;
          else
            s.sortbuf[atomicAdd(&s.total, 1u)] = key;
        }
      } else if (top > prefix) {
        mymin = min(mymin, key);
      }
    }
  }
  // block-min of mymin
  for (int o = 16; o > 0; o >>= 1) mymin = min(mymin, __shfl_xor_sync(0xffffffffu, mymin, o));
  __shared__ unsigned long long wmin[RS_WARPS];
  if ((threadIdx.x & 31) == 0) wmin[threadIdx.x >> 5] = mymin;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long m = wmin[0];
    for (int i = 1; i < RS_WARPS; ++i) m = min(m, wmin[i]);
    if (MULTI) {
      if (m != ~0ull) atomicMin(gmin, m);
    } else {
      wmin[0] = m;
    }
  }
  gsync<MULTI>(wk.barrier);
  if (bid == 0 && threadIdx.x == 0) wk.phase_t[11 + SEL * 4] = global_timer_ns();
  const unsigned long long above = MULTI ? *gmin : wmin[0];
  unsigned long long klo, khi;
  if (gather) {
    if (MULTI) {
      for (int t = threadIdx.x; t < (int)cnt; t += RS_THREADS) s.sortbuf[t] = cand[t];
      __syncthreads();
    }
    block_select(s, s.sortbuf, (int)cnt, k, shift, above, klo, khi);
  } else {
    // only reachable when all 64 key bits are fixed: every candidate equals the prefix
    klo = prefix;
    khi = (k + 1 < cnt) ? prefix : above;
  }
  __syncthreads();
  if (bid == 0 && threadIdx.x == 0) wk.phase_t[12 + SEL * 4] = global_timer_ns();
  if (threadIdx.x == 0) {
    s.bc[0] = key_to_f64(klo);
    s.bc[1] = even ? key_to_f64(khi) : key_to_f64(klo);
  }
  __syncthreads();
  n1_out = n1;
}

// theta of an affine map p -> A p + b in the centred frame: [rows of A with b'_a after each, 1],
// b' = A c_m + b - c_f.  Lanes 0..12 return their entry.
__device__ __forceinline__ double theta_entry(const Rigid& T, const double* cm, const double* cf, int e) {
  if (e >= 12) return 1.0;
  const int r = e >> 2, c = e & 3;
  if (c < 3) return T.r[r * 3 + c];
  return T.r[r * 3 + 0] * cm[0] + T.r[r * 3 + 1] * cm[1] + T.r[r * 3 + 2] * cm[2] + T.t[r] - cf[r];
}

// --- Levenberg-Marquardt on the 13 x 13 moment matrix (warp 0 of block 0) -------------------
// Re-centred linear model.  With T_in the transform the match evaluated the distances d_i at,
//   r_i(T) = n_i . (T p_i - q_i) = d_i + n_i . ((A - A_in) u_i + (b' - b'_in)),   u_i = p_i - c_m,
// i.e. r_i = phi_i . theta with phi_i = [n_i (x) (u_i, 1), d_i] and
//   theta(x) = [R(alpha) row-wise with t'_a after each row, 1] - [theta(T_in), 0],  t' = R c_m + t - c_f.
// M = sum phi phi^T.  Near the solution theta is (tiny, ..., tiny, 1): sum r^2 = theta^T M theta is
// dominated by sum d^2 and carries no cancellation (the un-centred form phi = [.., -n.q'] loses
// (|q'| / |r|)^2 ~ 1e9 on millimetre residuals over metre-sized clouds).
// Everything here is a serial dependency chain executed by ONE warp while the rest of the grid
// waits at a barrier, so the code is organised to keep that chain short: the three sincos run on
// three lanes, the matrix products are spread over the lanes, and the 6 x 6 factorisation is a
// fully unrolled register Cholesky (one rsqrt per pivot, no division, no local memory).
__device__ __noinline__ void moment_products(Shared& s, int lane);
__device__ __noinline__ void lm_eval(Shared& s, const double* x, const double* cm, const double* cf, int lane) {
  double sn = 0.0, cs = 1.0;
  if (lane < 3) sincos(x[lane], &sn, &cs);
  const double s1 = __shfl_sync(0xffffffffu, sn, 0), c1 = __shfl_sync(0xffffffffu, cs, 0);
  const double s2 = __shfl_sync(0xffffffffu, sn, 1), c2 = __shfl_sync(0xffffffffu, cs, 1);
  const double s3 = __shfl_sync(0xffffffffu, sn, 2), c3 = __shfl_sync(0xffffffffu, cs, 2);
  if (lane == 0) {
    double R[9], D[3][9];
    R[0] = c2 * c3; R[1] = -c2 * s3; R[2] = s2;
    R[3] = c1 * s3 + s1 * s2 * c3; R[4] = c1 * c3 - s1 * s2 * s3; R[5] = -s1 * c2;
    R[6] = s1 * s3 - c1 * s2 * c3; R[7] = s1 * c3 + c1 * s2 * s3; R[8] = c1 * c2;
    // d/d alpha1
    D[0][0] = 0; D[0][1] = 0; D[0][2] = 0;
    D[0][3] = -R[6]; D[0][4] = -R[7]; D[0][5] = -R[8];
    D[0][6] = R[3]; D[0][7] = R[4]; D[0][8] = R[5];
    // d/d alpha2
    D[1][0] = -s2 * c3; D[1][1] = s2 * s3; D[1][2] = c2;
    D[1][3] = s1 * c2 * c3; D[1][4] = -s1 * c2 * s3; D[1][5] = s1 * s2;
    D[1][6] = -c1 * c2 * c3; D[1][7] = c1 * c2 * s3; D[1][8] = -c1 * s2;
    // d/d alpha3
    D[2][0] = -c2 * s3; D[2][1] = -c2 * c3; D[2][2] = 0;
    D[2][3] = c1 * c3 - s1 * s2 * s3; D[2][4] = -c1 * s3 - s1 * s2 * c3; D[2][5] = 0;
    D[2][6] = s1 * c3 + c1 * s2 * s3; D[2][7] = -s1 * s3 + c1 * s2 * c3; D[2][8] = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        s.th[a * 4 + b] = R[a * 3 + b] - s.th_in[a * 4 + b];
#pragma unroll
        for (int k = 0; k < 3; ++k) s.J[a * 4 + b][k] = D[k][a * 3 + b];
#pragma unroll
        for (int k = 3; k < 6; ++k) s.J[a * 4 + b][k] = 0.0;
      }
      s.th[a * 4 + 3] = (R[a * 3 + 0] * cm[0] + R[a * 3 + 1] * cm[1] + R[a * 3 + 2] * cm[2] + x[3 + a] - cf[a]) -
                        s.th_in[a * 4 + 3];
#pragma unroll
      for (int k = 0; k < 3; ++k)
        s.J[a * 4 + 3][k] = D[k][a * 3 + 0] * cm[0] + D[k][a * 3 + 1] * cm[1] + D[k][a * 3 + 2] * cm[2];
#pragma unroll
      for (int k = 3; k < 6; ++k) s.J[a * 4 + 3][k] = (k - 3 == a) ? 1.0 : 0.0;
    }
    s.th[12] = 1.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) s.J[12][k] = 0.0;
  }
  __syncwarp();
  moment_products(s, lane);
}

// A = J^T M J, g = J^T M theta, F = theta^T M theta from s.J / s.th (one warp).
__device__ __noinline__ void moment_products(Shared& s, int lane) {
  for (int e = lane; e < 91; e += 32) {
    const int r = e / 7, c = e % 7;
    double acc = 0.0;
#pragma unroll
    for (int m = 0; m < 13; ++m) acc = fma(s.M[r][m], (c < 6) ? s.J[m][c] : s.th[m], acc);
    s.B[r][c] = acc;
  }
  __syncwarp();
  for (int e = lane; e < 43; e += 32) {
    double acc = 0.0;
    if (e < 36) {
      const int i = e / 6, j = e % 6;
#pragma unroll
      for (int m = 0; m < 13; ++m) acc = fma(s.J[m][i], s.B[m][j], acc);
      s.A[e] = acc;
    } else if (e < 42) {
      const int i = e - 36;
#pragma unroll
      for (int m = 0; m < 13; ++m) acc = fma(s.J[m][i], s.B[m][6], acc);
      s.g[i] = acc;
    } else {
#pragma unroll
      for (int m = 0; m < 13; ++m) acc = fma(s.th[m], s.B[m][6], acc);
      s.F = acc;
    }
  }
  __syncwarp();
}

// Warp-cooperative Cholesky of the AUGMENTED 7 x 7 system [[A, b], [b^T, 1]]: lane t < 28 owns
// entry (ri, cj) of the lower triangle, t = ri (ri + 1) / 2 + cj; rows 0..5 are A, row 6 is the
// right-hand side, so the factorisation leaves the forward substitution L y = b in row 6.  Every
// step is a handful of shuffles and one FMA per lane, nothing is indexed dynamically and a lane
// holds ONE matrix value: the earlier single-lane register version needed the whole matrix plus
// its factor live at once, overflowed the kernel's 168-register budget and ran out of local
// memory (4.3 us per solve).  All 32 lanes must call these functions converged.
__device__ __forceinline__ void tri_coords(int lane, int& ri, int& cj) {
  const int t = min(lane, 27);
  int i = 0;
#pragma unroll
  for (int r = 1; r < 7; ++r)
    if (t >= r * (r + 1) / 2) i = r;
  ri = i;
  cj = t - i * (i + 1) / 2;
}

// In: val = this lane's entry of the augmented matrix.  Out: its entry of the factor L (the
// diagonal holds sqrt(d_j)); inv[j] = 1 / sqrt(d_j) in every lane; returns false when a pivot is
// not positive (uniform across the warp).
__device__ __forceinline__ bool warp_chol7_factor(double& val, int ri, int cj, double (&inv)[6]) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const double d = __shfl_sync(0xffffffffu, val, j * (j + 1) / 2 + j);
    ok = ok && (d > 0.0) && isfinite(d);
    const double r = rsqrt(d);
    inv[j] = r;
    if (cj == j) val *= r;
    const double lij = __shfl_sync(0xffffffffu, val, ri * (ri + 1) / 2 + j);
    const double lkj = __shfl_sync(0xffffffffu, val, cj * (cj + 1) / 2 + j);
    if (cj > j) val = fma(-lij, lkj, val);
  }
  return ok;
}

// Back substitution L^T x = y on the factored lanes; returns x[lane] in lanes 0..5.
__device__ __forceinline__ double warp_chol7_backsolve(double val, int lane, int ri, int cj,
                                                       const double (&inv)[6]) {
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    if (ri == 6 && cj == i) val *= inv[i];
    const double xi = __shfl_sync(0xffffffffu, val, 21 + i);
    const double lik = __shfl_sync(0xffffffffu, val, i * (i + 1) / 2 + min(cj, i));
    if (ri == 6 && cj < i) val = fma(-lik, xi, val);
  }
  return __shfl_sync(0xffffffffu, val, 21 + min(lane, 5));
}

struct LmOut {
  double x[6];
  int iters;
  int ok;
};

// s.Ak / s.gk hold the unweighted J^T M J and J^T M theta at the current x.
__device__ void lm_solve(Shared& s, const RSArgs& a, double w, const double* x0, const double* cm,
                         const double* cf, LmOut& out, int lane) {
  double x[6], xn[6];
  bool fre[6], obsd[6];
  int nf = 0;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    x[j] = x0[j];
    fre[j] = isfinite(a.wobs[j]);
    obsd[j] = fre[j] && a.wobs[j] > 0.0;
    nf += fre[j] ? 1 : 0;
  }
  const double w2 = w * w;
  int ri, cj;
  tri_coords(lane, ri, cj);
  auto obs_cost = [&](const double* xx) {
    double c = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j)
      if (obsd[j]) {
        const double r = a.wobs[j] * (xx[j] - a.obs[j]);
        c += r * r;
      }
    return c;
  };
  auto keep_eval = [&]() {
    for (int e = lane; e < 42; e += 32) {
      if (e < 36) s.Ak[e] = s.A[e];
      else s.gk[e - 36] = s.g[e - 36];
    }
    __syncwarp();
  };
  lm_eval(s, x, cm, cf, lane);
  keep_eval();
  if (lane == 0) s.stamp[0] = global_timer_ns();
  double F = w2 * s.F + obs_cost(x);
  double lambda = 0.0, rel_prev = 0.0;
  int it = 0, ok = 1;
  for (it = 0; it < 40 && nf > 0; ++it) {
    {
      // weighted Gauss-Newton system; fixed parameters become identity rows (delta = 0)
      double val;
      const double wi = a.wobs[min(ri, 5)], wj = a.wobs[min(cj, 5)];
      const bool fj = isfinite(wj);
      double xj = 0.0;
#pragma unroll
      for (int k = 0; k < 6; ++k)
        if (k == cj) xj = x[k];
      if (ri < 6) {
        if (!(isfinite(wi) && fj)) {
          val = (ri == cj) ? 1.0 : 0.0;
        } else {
          val = w2 * s.Ak[ri * 6 + cj];
          if (ri == cj) {
            if (wi > 0.0) val += wi * wi;
            val *= (1.0 + lambda);
          }
        }
      } else if (cj < 6) {
        double gi = fj ? w2 * s.gk[cj] : 0.0;
        if (fj && wj > 0.0) gi += wj * wj * (xj - a.obs[cj]);
        val = -gi;
      } else {
        val = 1.0;
      }
      double inv[6];
      const bool spd = warp_chol7_factor(val, ri, cj, inv);
      const double sol = warp_chol7_backsolve(val, lane, ri, cj, inv);
      if (lane < 6) s.delta[lane] = sol;
      if (lane == 0) {
        s.spd = spd ? 1 : 0;
        if (it == 0) s.stamp[1] = global_timer_ns();
      }
    }
    __syncwarp();
    if (!s.spd) {
      lambda = fmax(lambda * 10.0, 1e-6);
      if (lambda > 1e10) {
        ok = 0;
        break;
      }
      __syncwarp();
      continue;
    }
    double rel = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const double dj = fre[j] ? s.delta[j] : 0.0;
      xn[j] = x[j] + dj;
      rel = fmax(rel, fabs(dj) / fmax(fabs(x[j]), 1e-3));
    }
    __syncwarp();
    // Gauss-Newton contracts linearly with a rate rho << 1 on these small-residual problems;
    // rho is estimated from consecutive steps (prior 1e-2 for the first one).  Once the error
    // predicted to remain AFTER taking this step, rel * rho / (1 - rho), is below 3e-10 the step
    // is taken and the loop ends without another evaluation (the reference's own solver stops
    // at ftol = xtol = 1e-8).
    const double rho = (rel_prev > 0.0) ? fmin(fmax(rel / rel_prev, 1e-6), 0.5) : 1e-2;
    const double remaining = rel * rho / (1.0 - rho);
    rel_prev = rel;
    if ((rel < 1e-9 || remaining < 3e-10) && lambda == 0.0) {
#pragma unroll
      for (int j = 0; j < 6; ++j) x[j] = xn[j];
      ++it;
      break;
    }
    lm_eval(s, xn, cm, cf, lane);
    const double Fn = w2 * s.F + obs_cost(xn);
    // Inside the basin (small undamped steps) plain Gauss-Newton is used: the cost, evaluated
    // through the moment matrix, carries cancellation noise of ~1e-9 relative, too coarse to
    // accept or reject steps that change it by less.  Far from it the cost test guards the step.
    const bool in_basin = (lambda == 0.0 && rel < 1e-3);
    if (in_basin || Fn <= F * (1.0 + 1e-10) + 1e-300) {
#pragma unroll
      for (int j = 0; j < 6; ++j) x[j] = xn[j];
      keep_eval();
      F = Fn;
      lambda = (lambda > 1e-9) ? lambda * 0.1 : 0.0;
    } else {
      lambda = fmax(lambda * 10.0, 1e-4);
      if (lambda > 1e10) break;
    }
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) out.x[j] = x[j];
  out.iters = it;
  out.ok = ok;
}

// Linearised variant: ONE solve of A x = l (c++/src/corrpts.cpp:113-156) expressed on the moment
// matrix.  With p2 = R_c u + c_f (u = movable point minus its centre, c_f = T_c c_m) the
// reference's row is r(x) = n . ((I + [alpha]x) p2 + t - q), i.e. theta(x) = theta0 + J x with
//   theta0 = [R_c rows, 0 after each row, 1],
//   d theta / d alpha_k = [e_k x (columns of R_c), (e_k x c_f)],   d theta / d t_k = e_k in slot 4a+3,
// so A^T A = J^T M J and A^T l = -J^T M theta0.  The centring only conditions the sums; x is the
// reference's x.  Returns x in s.delta and the pivot check in s.spd (warp 0 of block 0).
__device__ void lin_solve(Shared& s, const Rigid& Tc, const double* cf, int lane) {
  for (int e = lane; e < 13 * 6; e += 32) {
    const int r = e / 6, k = e % 6;
    double v = 0.0;
    if (r < 12) {
      const int a = r / 4, b = r % 4;
      if (k < 3) {
        if (a != k) {
          const bool neg = (a == (k + 1) % 3);
          const int c = neg ? (k + 2) % 3 : (k + 1) % 3;  // e_k x v: component a takes -/+ v[c]
          const double vc = (b < 3) ? Tc.r[c * 3 + b] : cf[c];
          v = neg ? -vc : vc;
        }
      } else if (b == 3 && k - 3 == a) {
        v = 1.0;
      }
    }
    s.J[r][k] = v;
  }
  if (lane < 13) {
    const int a = lane / 4, b = lane % 4;
    (void)a;
    (void)b;
    s.th[lane] = (lane == 12) ? 1.0 : 0.0;  // re-centred model: theta(x) - theta(T_c) = J x
  }
  __syncwarp();
  moment_products(s, lane);
  int ri, cj;
  tri_coords(lane, ri, cj);
  double val = 1.0;
  if (ri < 6) val = s.A[ri * 6 + cj];
  else if (cj < 6) val = -s.g[cj];
  double inv[6];
  const bool spd = warp_chol7_factor(val, ri, cj, inv);
  const double sol = warp_chol7_backsolve(val, lane, ri, cj, inv);
  if (lane < 6) s.delta[lane] = sol;
  if (lane == 0) s.spd = spd ? 1 : 0;
  __syncwarp();
}

// sigma of the free parameters: Cxx = s0^2 (A^T P A)^-1 in the reference's formulation
// (optimization.py:147-160): N = w * sum a a^T + diag(w_obs), vPv = w sum r^2 + sum w_obs dx^2.
// Called by a full warp: lane j < 6 produces sigma[j] (one column of the inverse each).
__device__ void uncertainties(Shared& s, const RSArgs& a, const double* An, double w,
                              const double* x, double sum_r2, long long n_kept, int lane,
                              double* sigma) {
  int nf = 0, nobs = 0;
  double vPv = w * sum_r2;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const bool fj = isfinite(a.wobs[j]);
    nf += fj ? 1 : 0;
    if (fj && a.wobs[j] > 0.0) {
      ++nobs;
      vPv += a.wobs[j] * (x[j] - a.obs[j]) * (x[j] - a.obs[j]);
    }
  }
  const double s02 = vPv / (double)(n_kept + nobs - nf);
  int ri, cj;
  tri_coords(lane, ri, cj);
  const double wi = a.wobs[min(ri, 5)], wj = a.wobs[min(cj, 5)];
  double val = (ri == cj) ? 1.0 : 0.0;
  if (ri < 6 && isfinite(wi) && isfinite(wj)) {
    val = w * An[ri * 6 + cj];
    if (ri == cj && wi > 0.0) val += wi;
  } else if (ri == 6 && cj < 6) {
    val = 0.0;
  }
  double inv[6];
  const bool ok = warp_chol7_factor(val, ri, cj, inv);
  // (N^-1)_jj = |L^-1 e_j|^2: lane j forward-substitutes its own unit vector against the factor,
  // which the owning lanes publish through shared memory.
  double* L = s.cholL;
  if (lane < 21) L[lane] = val;
  __syncwarp();
  if (lane < 6) {
    double y[6], acc = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      double v = (i == lane) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < i; ++k) v = fma(-L[i * (i + 1) / 2 + k], y[k], v);
      y[i] = v * inv[i];
      acc = fma(y[i], y[i], acc);
    }
    sigma[lane] = (ok && isfinite(a.wobs[lane])) ? sqrt(s02 * acc) : nan("");
  }
  __syncwarp();
}

// Median and MAD from the predictor histogram the match kernel filled (reject_solve.cuh:
// lh_bin): LH_BINS linear bins centred on the previous median, +-4 previous MADs wide.
//   * the bins holding the two middle ranks give the median candidates;
//   * with med somewhere in those bins, an element delta bins away has |d - med| inside
//     ((delta-1) w, (delta+g+1) w), so cumulative symmetric counts N_in(t) bracket the MAD ranks:
//     everything closer than t_lo - g bins is certainly below the MAD (counted, not gathered),
//     everything farther than t_hi + g + 1 bins certainly above; the bins in between are the
//     MAD candidates.
// One gather pass + one grid barrier then yields both order statistics exactly (same values as
// the radix path).  Returns false — before touching global state — when the prediction does not
// bracket the ranks (first iteration, large change, too many candidates): the caller falls back.
template <bool MULTI>
__device__ bool predicted_median_mad(Shared& s, const RSArgs& a, RSWork wk, const DevState* st,
                                     unsigned int& n1_out, double& median, double& mad) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double pm = st->pred_med, pd = st->pred_mad;
  constexpr int PER = (LH_BINS + RS_THREADS - 1) / RS_THREADS;
  const int b0 = tid * PER;
  unsigned int v[PER], sum = 0;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int b = b0 + j;
    v[j] = (b < LH_BINS) ? wk.lin_hist[b] : 0u;
    sum += v[j];
  }
  unsigned int incl = sum;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s.scan_tmp[warp] = incl;
  __syncthreads();
  unsigned int woff = 0, total_in = 0;
  for (int i = 0; i < RS_WARPS; ++i) {
    if (i < warp) woff += s.scan_tmp[i];
    total_in += s.scan_tmp[i];
  }
  {
    unsigned int run = woff + incl - sum;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      run += v[j];
      if (b0 + j < LH_BINS) s.hist[b0 + j] = run;  // inclusive prefix sums
    }
  }
  if (tid == 0) {
    s.lh_i[0] = -1;
    s.lh_i[1] = -1;
    s.lh_i[2] = LH_BINS + 1;  // t_hi (min over t)
    s.lh_i[3] = -1;           // t_lo (max over t)
  }
  __syncthreads();
  const unsigned int* P = s.hist;
  const unsigned int under = wk.lin_hist[LH_BINS], over = wk.lin_hist[LH_BINS + 1];
  const unsigned int n1 = under + total_in + over;
  n1_out = n1;
  if (n1 == 0) return true;
  const unsigned int k = (n1 - 1) >> 1;
  const bool even = ((n1 & 1u) == 0u);
  const unsigned int k2 = k + (even ? 1u : 0u);
  if (k < under || k2 >= under + total_in) return false;
  const unsigned int r = k - under, r2 = k2 - under;
  // bins of the two middle ranks: first b with P[b] > r
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int b = b0 + j;
    if (b < LH_BINS) {
      const unsigned int pb = P[b], pa = (b > 0) ? P[b - 1] : 0u;
      if (pa <= r && r < pb) s.lh_i[0] = b;
      if (pa <= r2 && r2 < pb) s.lh_i[1] = b;
    }
  }
  __syncthreads();
  const int bm = s.lh_i[0], bm2 = s.lh_i[1];
  if (bm < 0 || bm2 < bm) return false;
  const int g = bm2 - bm;
  if (g > 4) return false;
  const unsigned int below_m = (bm > 0) ? P[bm - 1] : 0u;
  const unsigned int cnt_med = P[bm2] - below_m;
  if (cnt_med > (unsigned int)(RS_CAP - 2)) return false;
  const unsigned int kA = r - below_m;
  auto Nin = [&](int t) -> unsigned int {
    const int hi = min(bm2 + t, LH_BINS - 1), lo = bm - t - 1;
    return P[hi] - ((lo >= 0) ? P[lo] : 0u);
  };
  int tmin = LH_BINS + 1, tmax = -1;
  for (int t = tid; t <= LH_BINS; t += RS_THREADS) {
    const unsigned int nin = Nin(t);
    if (nin >= k2 + 1u) tmin = min(tmin, t);
    if (nin <= k) tmax = max(tmax, t);
  }
  for (int o = 16; o > 0; o >>= 1) {
    tmin = min(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
    tmax = max(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
  }
  if (lane == 0) {
    atomicMin(&s.lh_i[2], tmin);
    atomicMax(&s.lh_i[3], tmax);
  }
  __syncthreads();
  const int t_hi = s.lh_i[2], t_lo = s.lh_i[3];
  if (t_hi > LH_BINS) return false;
  const int e_lo = max(t_lo - g, 0), e_hi = t_hi + g + 1;
  if (bm - e_hi < 0 || bm2 + e_hi > LH_BINS - 1) return false;  // candidates must be regular bins
  const unsigned int n_inner = (t_lo - g - 1 >= 0) ? Nin(t_lo - g - 1) : 0u;
  const unsigned int cnt_edge = Nin(e_hi) - n_inner;
  if (cnt_edge > (unsigned int)(RS_CAP - 2) || k < n_inner || k2 - n_inner >= cnt_edge) return false;
  const unsigned int kM = k - n_inner;
  __syncthreads();

  // ---- the one gather pass
  unsigned long long* cand_med = wk.cand;
  unsigned long long* cand_edge = wk.cand + RS_CAP;
  for (long long i = blockIdx.x * (long long)RS_THREADS + tid; i < a.K; i += (long long)gridDim.x * RS_THREADS) {
    if (pl_stat(a.q_nrm[i].w, a.pl_signed) >= a.stat_minpl) {
      const double d = a.dist[i];
      const int b = lh_bin(d, pm, pd);
      if (b < LH_BINS) {
        const int delta = (b < bm) ? (bm - b) : ((b > bm2) ? (b - bm2) : 0);
        if (delta == 0) cand_med[atomicAdd(&wk.counters[0], 1u)] = f64_to_key(d);
        if (delta >= e_lo && delta <= e_hi)
          cand_edge[atomicAdd(&wk.counters[1], 1u)] = (unsigned long long)__double_as_longlong(d);
      }
    }
  }
  gsync<MULTI>(wk.barrier);
  if (blockIdx.x == 0 && tid == 0) {
    wk.phase_t[10] = global_timer_ns();
    wk.phase_t[24] = 0;
    wk.phase_t[25] = 0;
    wk.phase_t[26] = cnt_med;
    wk.phase_t[27] = cnt_edge;
  }
  unsigned long long klo, khi;
  for (int t = tid; t < (int)cnt_med; t += RS_THREADS) s.sortbuf[t] = cand_med[t];
  __syncthreads();
  block_select(s, s.sortbuf, (int)cnt_med, kA, 64, ~0ull, klo, khi);
  median = even ? (a.variant ? key_to_f64(khi) : 0.5 * (key_to_f64(klo) + key_to_f64(khi))) : key_to_f64(klo);
  __syncthreads();
  for (int t = tid; t < (int)cnt_edge; t += RS_THREADS)
    s.sortbuf[t] = f64_to_key(fabs(__longlong_as_double((long long)cand_edge[t]) - median));
  __syncthreads();
  block_select(s, s.sortbuf, (int)cnt_edge, kM, 64, ~0ull, klo, khi);
  mad = even ? (a.variant ? key_to_f64(khi) : 0.5 * (key_to_f64(klo) + key_to_f64(khi))) : key_to_f64(klo);
  __syncthreads();
  return true;
}

template <bool MULTI>
__global__ void __launch_bounds__(RS_THREADS, 1) k_reject_solve(RSArgs a, RSWork wk) {
  __shared__ Shared s;
  DevState* st = a.state;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long K = a.K;
  const int G = gridDim.x;

  // zero the other parity's workspace for the next launch (nobody is using it)
  {
    unsigned int* oh = wk.hist_other;
    const long long nz = 2ll * RS_LEVELS * RS_BINS;
    for (long long i = blockIdx.x * (long long)RS_THREADS + tid; i < nz; i += (long long)G * RS_THREADS) oh[i] = 0;
    if (blockIdx.x == 0 && tid < 2) {
      wk.counters_other[tid] = 0;
      wk.minkey_other[tid] = ~0ull;
    }
  }
  if (st->stop) {  // a previous iteration already met the stop rule
    for (int i = blockIdx.x * RS_THREADS + tid; i < LH_BINS + 2; i += G * RS_THREADS) wk.lin_hist[i] = 0;
    return;
  }
#define RS_STAMP(i) do { if (blockIdx.x == 0 && tid == 0) wk.phase_t[i] = global_timer_ns(); } while (0)
  RS_STAMP(0);

  // ---- A + B: median and MAD of the planarity survivors
  unsigned int n1 = 0;
  double median = 0.0, mad = 0.0;
  bool fast = false;
  if (a.hist_expected && st->pred_valid && st->pred_minpl == a.stat_minpl && st->pred_mad > 0.0)
    fast = predicted_median_mad<MULTI>(s, a, wk, st, n1, median, mad);
  sicp_iter_record* rec = a.rec;
  if (!fast) {
    __syncthreads();
    radix_median<MULTI, 0>(s, a, wk, 0.0, n1);
    if (n1 != 0) {
      median = a.variant ? s.bc[1] : 0.5 * (s.bc[0] + s.bc[1]);
      __syncthreads();
      RS_STAMP(1);
      unsigned int n1b = 0;
      radix_median<MULTI, 1>(s, a, wk, median, n1b);
      mad = a.variant ? s.bc[1] : 0.5 * (s.bc[0] + s.bc[1]);
    }
  }
  if (n1 == 0) {
    for (int i = blockIdx.x * RS_THREADS + tid; i < LH_BINS + 2; i += G * RS_THREADS) wk.lin_hist[i] = 0;
    if (blockIdx.x == 0 && tid == 0) {
      rec->n_kept = 0;
      rec->median = rec->mad = nan("");
      st->n_kept = 0;
    }
    return;
  }
  // python: |d - med| <= 3 mad (corrpts.py:176-188); linearised: not > 3 (1.4826 mad) (corrpts.cpp:61-66)
  const double lim = a.variant ? 3.0 * (1.4826 * mad) : 3.0 * mad;
  __syncthreads();
  if (fast) RS_STAMP(1);
  RS_STAMP(2);
  if (blockIdx.x == 0 && tid == 0) wk.phase_t[28] = fast ? 1 : 0;
  // the predictor histogram has been consumed (or was not usable): leave it zeroed for the next match
  for (int i = blockIdx.x * RS_THREADS + tid; i < LH_BINS + 2; i += G * RS_THREADS) wk.lin_hist[i] = 0;

  // ---- C: keep flags + moment accumulation
  const Rigid Tin = st->T;
  double cm[3] = {a.cm[0], a.cm[1], a.cm[2]}, cf[3];
  rigid_apply(Tin, cm[0], cm[1], cm[2], cf[0], cf[1], cf[2]);
  {
    const int role = warp % 3, sub = (warp / 3) * 32 + lane;  // 128 threads per role
    double acc[RS_NACC];
#pragma unroll
    for (int j = 0; j < RS_NACC; ++j) acc[j] = 0.0;
    const long long chunk = (K + G - 1) / G;
    const long long i0 = blockIdx.x * chunk, i1 = min(i0 + chunk, K);
    const float4* __restrict__ qn = a.q_nrm;
    const double* __restrict__ dd = a.dist;
    const long long* __restrict__ nn = a.nn_idx;
    const double* __restrict__ mv = a.mov_xyz;
    const double* __restrict__ qx = a.q_xyz;
    auto accumulate = [&](const float4 nr, const double d, const double p0, const double p1,
                          const double p2, const double f0, const double f1, const double f2) {
      const double u0 = p0 - cm[0], u1 = p1 - cm[1], u2 = p2 - cm[2];
      (void)f0;
      (void)f1;
      (void)f2;
      const double n0 = (double)nr.x, n1d = (double)nr.y, n2 = (double)nr.z;
      const double sc = d;  // re-centred model: the scalar entry of phi is the distance itself
      double na, nb, nv;
      if (role == 0) {
        na = n0 * n0; nb = n0 * n1d; nv = n0;
      } else if (role == 1) {
        na = n0 * n2; nb = n1d * n1d; nv = n1d;
      } else {
        na = n1d * n2; nb = n2 * n2; nv = n2;
      }
      const double U[10] = {u0 * u0, u0 * u1, u0 * u2, u0, u1 * u1, u1 * u2, u1, u2 * u2, u2, 1.0};
#pragma unroll
      for (int t = 0; t < 10; ++t) {
        acc[t] = fma(na, U[t], acc[t]);
        acc[10 + t] = fma(nb, U[t], acc[10 + t]);
      }
      const double sn = sc * nv;
      acc[20] = fma(sn, u0, acc[20]);
      acc[21] = fma(sn, u1, acc[21]);
      acc[22] = fma(sn, u2, acc[22]);
      acc[23] += sn;
      if (role == 0) {
        acc[24] = fma(sc, sc, acc[24]);
        acc[25] += 1.0;
      } else if (role == 1) {
        acc[24] += d;
        acc[25] = fma(d, d, acc[25]);
      }
    };
    // two elements per trip so that both dependent gather chains (nn_idx -> mov_xyz) overlap
    for (long long i = i0 + sub; i < i1; i += 256) {
      const long long ib = i + 128;
      const bool hb = ib < i1;
      const float4 nrA = qn[i];
      const float4 nrB = hb ? qn[ib] : make_float4(0.f, 0.f, 0.f, -1.f);
      const double dA = dd[i], dB = hb ? dd[ib] : 0.0;
      const bool kA = pl_keep(nrA.w, a.min_planarity, a.pl_signed) && (fabs(dA - median) <= lim);
      const bool kB = hb && pl_keep(nrB.w, a.min_planarity, a.pl_signed) && (fabs(dB - median) <= lim);
      const long long jA = kA ? nn[i] : 0, jB = kB ? nn[ib] : 0;
      const long long ia = kA ? i : i0, ibb = kB ? ib : i0;
      const double pA0 = mv[3 * jA + 0], pA1 = mv[3 * jA + 1], pA2 = mv[3 * jA + 2];
      const double pB0 = mv[3 * jB + 0], pB1 = mv[3 * jB + 1], pB2 = mv[3 * jB + 2];
      const double fA0 = qx[3 * ia + 0], fA1 = qx[3 * ia + 1], fA2 = qx[3 * ia + 2];
      const double fB0 = qx[3 * ibb + 0], fB1 = qx[3 * ibb + 1], fB2 = qx[3 * ibb + 2];
      if (kA) accumulate(nrA, dA, pA0, pA1, pA2, fA0, fA1, fA2);
      if (kB) accumulate(nrB, dB, pB0, pB1, pB2, fB0, fB1, fB2);
      if (role == 0) {
        a.keep[i] = kA ? 1 : 0;
        if (hb) a.keep[ib] = kB ? 1 : 0;
      }
    }
#pragma unroll
    for (int j = 0; j < RS_NACC; ++j) {
      const double v = warp_sum(acc[j]);
      if (lane == 0) s.red[warp][j] = v;
    }
    __syncthreads();
    if (tid < RS_NPART) {
      const int r = tid / RS_NACC, j = tid % RS_NACC;
      double v = 0.0;
      for (int ww = r; ww < RS_WARPS; ww += 3) v += s.red[ww][j];
      if (MULTI)
        wk.partials[(size_t)tid * G + blockIdx.x] = v;
      else
        s.tot[tid] = v;
    }
  }
  RS_STAMP(3);
  gsync<MULTI>(wk.barrier);
  RS_STAMP(4);

  // ---- D: block 0 reduces the partials and solves
  if (blockIdx.x == 0) {
    if (MULTI) {
      // fixed-order sum of the per-block partials, stored value-major ([value][block]): each warp
      // owns a few values, reads their G block entries with coalesced, fully overlapped loads and
      // finishes with a shuffle tree (deterministic: the order depends on G only)
      // (all loads of a warp are issued before the first use: one L2 round trip, not 35)
      constexpr int NO = (RS_NPART + RS_WARPS - 1) / RS_WARPS;  // values per warp
      constexpr int NB = 8;                                      // 32 * 8 = 256 blocks max
      double r[NO][NB];
#pragma unroll
      for (int q = 0; q < NO; ++q) {
        const int o = warp + q * RS_WARPS;
#pragma unroll
        for (int u = 0; u < NB; ++u) {
          const int b = lane + 32 * u;
          r[q][u] = (o < RS_NPART && b < G) ? wk.partials[(size_t)o * G + b] : 0.0;
        }
      }
#pragma unroll
      for (int q = 0; q < NO; ++q) {
        const int o = warp + q * RS_WARPS;
        double v = 0.0;
#pragma unroll
        for (int u = 0; u < NB; ++u) v += r[q][u];
        v = warp_sum(v);
        if (lane == 0 && o < RS_NPART) s.tot[o] = v;
        if (q == 0) RS_STAMP(20);
      }
    }
    __syncthreads();
    RS_STAMP(17);
    // assemble M (13 x 13) from T (6 x 10), V (3 x 4), S
    for (int e = tid; e < 169; e += RS_THREADS) {
      const int r = e / 13, c = e % 13;
      double v;
      if (r == 12 && c == 12) {
        v = s.tot[0 * RS_NACC + 24];
      } else if (r == 12 || c == 12) {
        const int o = (r == 12) ? c : r;
        v = s.tot[(o / 4) * RS_NACC + 20 + (o % 4)];
      } else {
        int aa = r / 4, bb = r % 4, cc = c / 4, dd = c % 4;
        if (aa > cc) { int t = aa; aa = cc; cc = t; }
        if (bb > dd) { int t = bb; bb = dd; dd = t; }
        const int i6 = (aa == 0) ? cc : (aa == 1 ? 2 + cc : 5);          // (0,0)0 (0,1)1 (0,2)2 (1,1)3 (1,2)4 (2,2)5
        const int i10 = (bb == 0) ? dd : (bb == 1 ? 3 + dd : (bb == 2 ? 5 + dd : 9));  // (1,1)4 (1,2)5 (1,3)6 (2,2)7 (2,3)8 (3,3)9
        v = s.tot[(i6 / 2) * RS_NACC + (i6 % 2) * 10 + i10];
      }
      s.M[r][c] = v;
    }
    if (tid < 13) s.th_in[tid] = (tid == 12) ? 0.0 : theta_entry(Tin, cm, cf, tid);
    __syncthreads();
    RS_STAMP(18);
    if (warp == 0) {
      const long long n_kept = (long long)(s.tot[0 * RS_NACC + 25] + 0.5);
      const double sum_d = s.tot[1 * RS_NACC + 24], sum_d2 = s.tot[1 * RS_NACC + 25];
      const double mean_d = (n_kept > 0) ? sum_d / (double)n_kept : nan("");
      const double var_d = (n_kept > 0) ? fmax(sum_d2 / (double)n_kept - mean_d * mean_d, 0.0) : nan("");
      // the C++ driver prints the SAMPLE std of the kept distances as its "orig:0" row (simpleicp.cpp:95-100)
      const double var_d1 = (n_kept > 1) ? fmax(sum_d2 - (double)n_kept * mean_d * mean_d, 0.0) / (double)(n_kept - 1) : nan("");
      double w = st->w;
      if (a.variant) {
        w = 1.0;
      } else if (a.it == 0 || !(w > 0.0)) {
        w = a.w_param;
        if (!(w > 0.0)) w = 1.0 / var_d;  // distance_weights=None: 1/std(d)^2 (simpleicp.py:233-234)
      }
      int skip = (n_kept < 6) || !a.do_solve;
      LmOut lo;
      lo.iters = 0;
      lo.ok = 1;
      if (!skip && a.variant) {
        lin_solve(s, st->T, cf, lane);
        lo.iters = 1;
        lo.ok = s.spd;
#pragma unroll
        for (int j = 0; j < 6; ++j) lo.x[j] = s.delta[j];
      } else if (!skip) {
        lm_solve(s, a, w, st->x, cm, cf, lo, lane);
        if (lane == 0) {
          wk.phase_t[19] = global_timer_ns();
          wk.phase_t[21] = s.stamp[0];
          wk.phase_t[22] = s.stamp[1];
        }
      }
      if (lane == 0) {
        rec->n_kept = n_kept;
        rec->median = median;
        rec->mad = mad;
        st->pred_med = median;
        st->pred_mad = mad;
        st->pred_minpl = a.stat_minpl;
        st->pred_valid = (mad > 0.0 && isfinite(mad) && isfinite(median)) ? 1 : 0;
        rec->mean_dist = mean_d;
        rec->std_dist = sqrt(a.variant ? var_d1 : var_d);
        rec->distance_weight = w;
        rec->lm_iterations = lo.iters;
        rec->n_bruteforce = a.unresolved ? (int)a.unresolved[K] : 0;
        if (a.unresolved) a.unresolved[K] = 0u;  // the next match starts from a clean counter
        st->n_kept = n_kept;
        st->skip = skip;
        st->w = w;
        if (n_kept < 6 && a.do_solve && a.arm_stop) st->stop = 2;  // too few correspondences
        if (!skip) {
          for (int j = 0; j < 6; ++j) st->x_new[j] = lo.x[j];
          for (int e = 0; e < 36; ++e) st->An[e] = s.Ak[e];
          if (a.variant) {
            // cloud <- dH cloud (pointcloud.cpp:149-152), residuals of the linear model
            const Rigid dH = rigid_from_x(lo.x);
            st->T_new = rigid_compose(dH, Tin);
            Rigid L;  // I + [alpha]x, t
            L.r[0] = 1.0; L.r[1] = -lo.x[2]; L.r[2] = lo.x[1];
            L.r[3] = lo.x[2]; L.r[4] = 1.0; L.r[5] = -lo.x[0];
            L.r[6] = -lo.x[1]; L.r[7] = lo.x[0]; L.r[8] = 1.0;
            L.t[0] = lo.x[3]; L.t[1] = lo.x[4]; L.t[2] = lo.x[5];
            st->T_res = rigid_compose(L, Tin);
            const Rigid Hr = st->H_rep;
            st->H_rep = (a.variant == SICP_VARIANT_LINEARIZED_CPP) ? rigid_compose(Hr, dH) : rigid_compose(dH, Hr);
          } else {
            st->T_new = rigid_from_x(lo.x);
            st->T_res = st->T_new;
          }
          st->lm_ok = lo.ok;
        }
      }
    }
  }
  RS_STAMP(5);
  gsync<MULTI>(wk.barrier);
  RS_STAMP(6);
  if (st->skip) return;

  // ---- E: residuals at the solution, in the reference's operation order
  {
    const Rigid Tn = st->T_res;
    double sr = 0.0, sr2 = 0.0;
    for (long long i = blockIdx.x * (long long)RS_THREADS + tid; i < K; i += (long long)G * RS_THREADS) {
      if (!a.keep[i]) continue;
      const long long j = a.nn_idx[i];
      double tx, ty, tz;
      rigid_apply(Tn, a.mov_xyz[3 * j + 0], a.mov_xyz[3 * j + 1], a.mov_xyz[3 * j + 2], tx, ty, tz);
      const float4 nr = a.q_nrm[i];
      const double dx = tx - a.q_xyz[3 * i + 0], dy = ty - a.q_xyz[3 * i + 1], dz = tz - a.q_xyz[3 * i + 2];
      const double r = __dadd_rn(__dadd_rn(__dmul_rn(dx, (double)nr.x), __dmul_rn(dy, (double)nr.y)),
                                 __dmul_rn(dz, (double)nr.z));
      a.resid[i] = r;
      sr += r;
      sr2 = fma(r, r, sr2);
    }
    sr = warp_sum(sr);
    sr2 = warp_sum(sr2);
    if (lane == 0) {
      s.red[warp][0] = sr;
      s.red[warp][1] = sr2;
    }
    __syncthreads();
    if (tid == 0) {
      double t0 = 0, t1 = 0;
      for (int ww = 0; ww < RS_WARPS; ++ww) {
        t0 += s.red[ww][0];
        t1 += s.red[ww][1];
      }
      if (MULTI) {
        wk.partials[(size_t)G * RS_NPART + 2 * blockIdx.x + 0] = t0;
        wk.partials[(size_t)G * RS_NPART + 2 * blockIdx.x + 1] = t1;
      } else {
        s.bc[2] = t0;
        s.bc[3] = t1;
      }
    }
  }
  RS_STAMP(7);
  gsync<MULTI>(wk.barrier);
  RS_STAMP(8);
  if (blockIdx.x == 0 && warp == 0) {
    double t0 = 0, t1 = 0;
    if (MULTI) {
      double r0[8], r1[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int b = lane + 32 * u;
        r0[u] = (b < G) ? wk.partials[(size_t)G * RS_NPART + 2 * b + 0] : 0.0;
        r1[u] = (b < G) ? wk.partials[(size_t)G * RS_NPART + 2 * b + 1] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        t0 += r0[u];
        t1 += r1[u];
      }
      t0 = warp_sum(t0);
      t1 = warp_sum(t1);
    } else {
      t0 = s.bc[2];
      t1 = s.bc[3];
    }
    const long long n = st->n_kept;
    const double mean = t0 / (double)n;
    // population std (numpy default, simpleicp.py:263) / sample std (c++/src/simpleicp.cpp:184-188)
    const double sd = a.variant ? sqrt(fmax(t1 - (double)n * mean * mean, 0.0) / (double)(n - 1))
                                : sqrt(fmax(t1 / (double)n - mean * mean, 0.0));
    // one lane per parameter: sigma_j, and the new cumulative parameters
    if (a.variant) {
      if (lane < 6) {
        st->sigma[lane] = nan("");
        rec->x[lane] = st->x_new[lane];  // the increments of this iteration
      }
    } else {
      uncertainties(s, a, st->An, st->w, st->x_new, t1, n, lane, st->sigma);
      if (lane < 6) {
        rec->x[lane] = st->x_new[lane];
        st->x[lane] = st->x_new[lane];
      }
    }
    if (lane == 0) {
      rec->mean_res = mean;
      rec->std_res = sd;
      // Predictor of the NEXT iteration's order statistics: the residuals at the new transform, not
      // the distances this iteration started from — the first solves of a registration shrink the
      // distribution several-fold, and the next match finds (mostly) these very correspondences.
      // median ~ mean, MAD ~ 0.8 std of the kept residuals (truncated at 3 MAD ~ 2 sigma).
      if (sd > 0.0 && isfinite(sd) && isfinite(mean)) {
        st->pred_med = mean;
        st->pred_mad = 0.8 * sd;
        st->pred_valid = 1;
      }
      st->T = st->T_new;
      st->Tinv = rigid_inverse(st->T_new);
      if (!a.variant) st->H_rep = st->T_new;
      // stop rule (simpleicp.py:355-379): relative change in percent of mean and population std
      int stop = 0;
      if (a.it > 0) {
        const double m0 = st->prev_mean, s0 = st->prev_std;
        const double cmn = (m0 == 0.0) ? ((mean == 0.0) ? 0.0 : kInf) : fabs((mean - m0) / m0 * 100.0);
        const double csd = (s0 == 0.0) ? ((sd == 0.0) ? 0.0 : kInf) : fabs((sd - s0) / s0 * 100.0);
        stop = (cmn < a.min_change && csd < a.min_change) ? 1 : 0;
      }
      st->prev_mean = mean;
      st->prev_std = sd;
      st->iterations_done = a.it + 1;
      if (stop && a.arm_stop) st->stop = 1;
      st->converged = stop;
      wk.phase_t[9] = global_timer_ns();
    }
  }
}

// =============================================================================================
// k_rs_fused — the same five steps WITHOUT grid barriers and without a cooperative launch.
//
// The cooperative kernel above spends half its time in four grid barriers and in serial sections
// that 147 SMs wait for (profiles/r1_phase_timeline.md).  Here every dependency is resolved by
// construction instead of by waiting:
//   select     every block derives median and MAD ITSELF from the predictor histogram the match
//              kernel filled and the per-bin index store it filled with the same atomic (slot =
//              returned count): the few hundred members of the bins that hold the order
//              statistics are read directly — redundant, identical work on every SM, no exchange,
//              no pass over the K correspondences.  (A first version scanned a 2-byte bin code per
//              correspondence in every block: 38 us of 2 M thread-instructions per SM.)  Same exact
//              order statistics as predicted_median_mad().
//   accumulate each block streams its share of (normal, distance, matched point, fixed point) —
//              the match kernel stored the matched point, so there is no index chase — and
//              writes keep flags and per-block partial sums.
//   solve      the block that takes the LAST ticket reduces the partials in a fixed order and runs
//              the Gauss-Newton loop; everybody else has already left the SM.
//   statistics mean and standard deviation of the residuals at the solution come from the moment
//              sums themselves (sum r = theta . sum phi, sum r^2 = theta^T M theta): no residual pass
//              and no barrier in the loop.  The residual VECTOR of the final iteration is evaluated
//              once, after the loop (k_final_residuals), in the reference's operation order, and
//              its statistics are recomputed two-pass from it.
// If the prediction does not bracket the order statistics (large change between iterations) the
// kernel changes nothing, raises state->stop = 3 and the host re-runs that iteration with the
// general kernel (capi.cu: run_loop).
// =============================================================================================
constexpr int RSF_NACC = 30;             // accumulators per role
constexpr int RSF_NPART = 3 * RSF_NACC;  // partial sums per block

constexpr int RSF_TILE = 768;  // correspondences per TMA-staged tile of the moment pass

struct SharedF {
  Shared s;
  // the block's share of (normal, distance, matched point), staged by 1-D TMA bulk copies that are
  // issued at kernel entry: the moment pass does not depend on the select, only the keep test
  // does, so the data crosses L2/HBM while the block works out median and MAD
  alignas(16) float4 t_nrm[RSF_TILE];
  alignas(16) double t_dist[RSF_TILE];
  alignas(16) double t_xyz[3 * RSF_TILE];
  alignas(8) uint64_t t_bar;
  double redf[RS_WARPS][RSF_NACC];
  double totf[RSF_NPART];
  double m1[13];  // sum phi
  int is_last;
};

// Plan + gather + selection; true on success (median, mad, n1 set; n1 == 0 is a success).
// k-th smallest (0-based) and its successor among n <= RS_THREADS keys in shared memory by direct
// ranking — three block barriers instead of the eight radix passes block_select() needs when the
// keys share their leading bytes (they always do here: the candidates come from a handful of
// adjacent histogram bins).
__device__ __forceinline__ void rank_select(Shared& s, const unsigned long long* keys, int n, unsigned int k,
                                            unsigned long long& klo, unsigned long long& khi) {
  // work item = (candidate, quarter of the list): n * 4 items over the block's threads, the four
  // partial ranks of a candidate meet in a shared-memory counter
  constexpr int PARTS = 4;
  const int tid = threadIdx.x;
  for (int c = tid; c < n; c += RS_THREADS) s.rank_acc[c] = 0;
  __syncthreads();
  for (int w = tid; w < n * PARTS; w += RS_THREADS) {
    const int c = w / PARTS, part = w - c * PARTS;
    const unsigned long long key = keys[c];
    unsigned int r = 0;
    for (int j = part; j < n; j += PARTS) {
      const unsigned long long kj = keys[j];
      r += (kj < key || (kj == key && j < c)) ? 1u : 0u;
    }
    atomicAdd(&s.rank_acc[c], r);
  }
  __syncthreads();
  for (int c = tid; c < n; c += RS_THREADS) {
    const unsigned int rank = s.rank_acc[c];
    if (rank == k) s.small[0] = keys[c];
    if (rank == k + 1u) s.small[1] = keys[c];
  }
  __syncthreads();
  klo = s.small[0];
  khi = (k + 1u < (unsigned int)n) ? s.small[1] : ~0ull;
  __syncthreads();
}

#define RSF_STAMP(i) do { if (bid == 0 && tid == 0) wk.phase_t[i] = global_timer_ns(); } while (0)
__device__ bool fused_select(SharedF& sf, const RSArgs& a, RSWork wk, const DevState* st,
                             unsigned int& n1_out, double& median, double& mad, const int G, const int bid) {
  Shared& s = sf.s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int PER = (LH_BINS + RS_THREADS - 1) / RS_THREADS;
  const int b0 = tid * PER;
  unsigned int v[PER], sum = 0;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int b = b0 + j;
    v[j] = (b < LH_BINS) ? __ldcg(&wk.lin_hist[b]) : 0u;
    sum += v[j];
  }
  // (requested together with the bins: one round trip, not two)
  const unsigned int under = __ldcg(&wk.lin_hist[LH_BINS]), over = __ldcg(&wk.lin_hist[LH_BINS + 1]);
  unsigned int incl = sum;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s.scan_tmp[warp] = incl;
  __syncthreads();
  unsigned int woff = 0, total_in = 0;
  for (int i = 0; i < RS_WARPS; ++i) {
    if (i < warp) woff += s.scan_tmp[i];
    total_in += s.scan_tmp[i];
  }
  {
    unsigned int run = woff + incl - sum;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
      run += v[j];
      if (b0 + j < LH_BINS) s.hist[b0 + j] = run;  // inclusive prefix sums
    }
  }
  if (tid == 0) {
    s.lh_i[0] = -1;
    s.lh_i[1] = -1;
    s.lh_i[2] = LH_BINS + 1;
    s.lh_i[3] = -1;
  }
  __syncthreads();
  const unsigned int* P = s.hist;
  const unsigned int n1 = under + total_in + over;
  n1_out = n1;
  if (n1 == 0) return true;
  const unsigned int k = (n1 - 1) >> 1;
  const bool even = ((n1 & 1u) == 0u);
  const unsigned int k2 = k + (even ? 1u : 0u);
  if (k < under || k2 >= under + total_in) return false;
  const unsigned int r = k - under, r2 = k2 - under;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const int b = b0 + j;
    if (b < LH_BINS) {
      const unsigned int pb = P[b], pa = (b > 0) ? P[b - 1] : 0u;
      if (pa <= r && r < pb) s.lh_i[0] = b;
      if (pa <= r2 && r2 < pb) s.lh_i[1] = b;
    }
  }
  __syncthreads();
  const int bm = s.lh_i[0], bm2 = s.lh_i[1];
  if (bm < 0 || bm2 < bm) return false;
  const int g = bm2 - bm;
  if (g > 4) return false;
  const unsigned int below_m = (bm > 0) ? P[bm - 1] : 0u;
  const unsigned int cnt_med = P[bm2] - below_m;
  if (cnt_med > (unsigned int)(RS_CAP - 2)) return false;
  const unsigned int kA = r - below_m;
  auto Nin = [&](int t) -> unsigned int {
    const int hi = min(bm2 + t, LH_BINS - 1), lo = bm - t - 1;
    return P[hi] - ((lo >= 0) ? P[lo] : 0u);
  };
  int tmin = LH_BINS + 1, tmax = -1;
  for (int t = tid; t <= LH_BINS; t += RS_THREADS) {
    const unsigned int nin = Nin(t);
    if (nin >= k2 + 1u) tmin = min(tmin, t);
    if (nin <= k) tmax = max(tmax, t);
  }
  for (int o = 16; o > 0; o >>= 1) {
    tmin = min(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
    tmax = max(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
  }
  if (lane == 0) {
    atomicMin(&s.lh_i[2], tmin);
    atomicMax(&s.lh_i[3], tmax);
  }
  __syncthreads();
  const int t_hi = s.lh_i[2], t_lo = s.lh_i[3];
  if (t_hi > LH_BINS) return false;
  const int e_lo = max(t_lo - g, 0), e_hi = t_hi + g + 1;
  if (bm - e_hi < 0 || bm2 + e_hi > LH_BINS - 1) return false;
  const unsigned int n_inner = (t_lo - g - 1 >= 0) ? Nin(t_lo - g - 1) : 0u;
  const unsigned int cnt_edge = Nin(e_hi) - n_inner;
  if (cnt_edge > (unsigned int)(RS_CAP - 2) || k < n_inner || k2 - n_inner >= cnt_edge) return false;
  const unsigned int kM = k - n_inner;
  RSF_STAMP(10);

  // ---- read the members of the candidate bins from the per-bin index store the match kernel
  // filled (slot = the value its histogram atomic returned): no scan, no gather pass.  A bin with
  // more members than slots means the distribution narrowed a lot since the last iteration: that
  // iteration goes through the general path.
  {
    const int cap = a.bin_cap;
    int over = 0;
    const int lo_b = bm - e_hi, hi_b = bm2 + e_hi;
    for (int bb = lo_b + tid; bb <= hi_b; bb += RS_THREADS) {
      const int delta = (bb < bm) ? (bm - bb) : ((bb > bm2) ? (bb - bm2) : 0);
      if ((delta == 0 || (delta >= e_lo && delta <= e_hi)) && P[bb] - ((bb > 0) ? P[bb - 1] : 0u) > (unsigned int)cap)
        over = 1;
    }
    if (__syncthreads_or(over)) return false;
  }
  // position (in histogram order) -> (bin, slot) -> correspondence number
  auto member = [&](unsigned int pos) -> unsigned int {
    int lo = 0, hi = LH_BINS - 1;  // first bin with P[bin] > pos
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (P[mid] > pos) hi = mid; else lo = mid + 1;
    }
    const unsigned int slot = pos - ((lo > 0) ? P[lo - 1] : 0u);
    return __ldcg(a.binstore + (size_t)lo * a.bin_cap + slot);
  };
  const unsigned int edge_lo_start = (bm - e_hi > 0) ? P[bm - e_hi - 1] : 0u;
  const int el = max(e_lo, 1);
  // members of the low edge window [bm - e_hi, bm - el]; with e_lo == 0 the window runs through
  // the median bins to bm2 + e_hi in one piece
  const unsigned int c_low = (e_lo == 0) ? cnt_edge : (P[bm - el] - edge_lo_start);
  const unsigned int edge_hi_start = P[bm2 + el - 1];
  RSF_STAMP(11);
  unsigned long long klo, khi;
  for (int t = tid; t < (int)cnt_med; t += RS_THREADS) s.sortbuf[t] = f64_to_key(__ldcg(a.dist + member(below_m + t)));
  __syncthreads();
  if (cnt_med <= (unsigned int)RS_THREADS) rank_select(s, s.sortbuf, (int)cnt_med, kA, klo, khi);
  else block_select(s, s.sortbuf, (int)cnt_med, kA, 64, ~0ull, klo, khi);
  median = even ? (a.variant ? key_to_f64(khi) : 0.5 * (key_to_f64(klo) + key_to_f64(khi))) : key_to_f64(klo);
  __syncthreads();
  RSF_STAMP(12);
  for (int t = tid; t < (int)cnt_edge; t += RS_THREADS) {
    const unsigned int pos = ((unsigned int)t < c_low) ? edge_lo_start + t : edge_hi_start + (t - c_low);
    s.sortbuf[t] = f64_to_key(fabs(__ldcg(a.dist + member(pos)) - median));
  }
  __syncthreads();
  if (cnt_edge <= (unsigned int)RS_THREADS) rank_select(s, s.sortbuf, (int)cnt_edge, kM, klo, khi);
  else block_select(s, s.sortbuf, (int)cnt_edge, kM, 64, ~0ull, klo, khi);
  mad = even ? (a.variant ? key_to_f64(khi) : 0.5 * (key_to_f64(klo) + key_to_f64(khi))) : key_to_f64(klo);
  __syncthreads();
  if (bid == 0 && tid == 0) {
    wk.phase_t[26] = cnt_med;
    wk.phase_t[27] = cnt_edge;
  }
  return true;
}

__device__ void rs_fused_body(const RSArgs& a, RSWork wk, const int G, const int bid, SharedF& sf) {
  Shared& s = sf.s;
  DevState* st = a.state;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long K = a.K;
  pdl_launch_dependents();  // the next match may take the SMs this kernel's blocks leave early
  pdl_wait();               // everything below reads what the match kernel wrote
  if (st->stop) return;  // a previous iteration met the stop rule (or asked for a re-run)
  RSF_STAMP(0);

  // ---- this block's share; its first tile starts moving now (even tile starts keep every source
  // address 16-byte aligned; a last odd tile reads 8 bytes of slack the buffers are allocated with)
  const long long chunk = (((K + G - 1) / G) + 1) & ~1ll;
  const long long i0 = min((long long)bid * chunk, K), i1 = min(i0 + chunk, K);
  auto issue_tile = [&](long long t0) {
    const uint32_t nt = (uint32_t)min((long long)RSF_TILE, i1 - t0);
    const uint32_t b_n = nt * 16u, b_d = (nt * 8u + 15u) & ~15u, b_p = (nt * 24u + 15u) & ~15u;
    mbar_expect_tx(&sf.t_bar, b_n + b_d + b_p);
    tma_load_1d(sf.t_nrm, a.q_nrm + t0, b_n, &sf.t_bar);
    tma_load_1d(sf.t_dist, a.dist + t0, b_d, &sf.t_bar);
    tma_load_1d(sf.t_xyz, a.m_xyz + 3 * t0, b_p, &sf.t_bar);
  };
  if (tid == 0) {
    mbar_init(&sf.t_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const bool have_tile = i0 < i1;
  if (tid == 0 && have_tile) issue_tile(i0);
  uint32_t tile_phase = 0;

  // ---- select (every block, identical result)
  unsigned int n1 = 0;
  double median = 0.0, mad = 0.0;
  bool ok = a.hist_expected && st->pred_valid && st->pred_minpl == a.stat_minpl && st->pred_mad > 0.0;
  if (ok) ok = fused_select(sf, a, wk, st, n1, median, mad, G, bid);
  if (!ok && G == 1) {
    // a single block owns the whole problem (K <= 4096, or one pair of a batch): no prediction —
    // first iteration, large change — simply means the radix selection, here and now
    __syncthreads();
    radix_median<false, 0>(s, a, wk, 0.0, n1, 0, 1);
    if (n1 != 0) {
      median = a.variant ? s.bc[1] : 0.5 * (s.bc[0] + s.bc[1]);
      __syncthreads();
      unsigned int n1b = 0;
      radix_median<false, 1>(s, a, wk, median, n1b, 0, 1);
      mad = a.variant ? s.bc[1] : 0.5 * (s.bc[0] + s.bc[1]);
    }
    __syncthreads();
    ok = true;
  }
  const double lim = a.variant ? 3.0 * (1.4826 * mad) : 3.0 * mad;
  RSF_STAMP(2);

  // ---- accumulate this block's share
  const Rigid Tin = st->T;
  double cm[3] = {a.cm[0], a.cm[1], a.cm[2]}, cf[3];
  rigid_apply(Tin, cm[0], cm[1], cm[2], cf[0], cf[1], cf[2]);
  if (ok && n1 != 0) {
    const int role = warp % 3, sub = (warp / 3) * 32 + lane;  // 128 threads per role
    double acc[RSF_NACC];
#pragma unroll
    for (int j = 0; j < RSF_NACC; ++j) acc[j] = 0.0;
    auto accumulate = [&](const float4 nr, const double d, const double p0, const double p1,
                          const double p2, const double f0, const double f1, const double f2) {
      const double u0 = p0 - cm[0], u1 = p1 - cm[1], u2 = p2 - cm[2];
      (void)f0;
      (void)f1;
      (void)f2;
      const double n0 = (double)nr.x, n1d = (double)nr.y, n2 = (double)nr.z;
      const double sc = d;  // re-centred model: the scalar entry of phi is the distance itself
      double na, nb, nv;
      if (role == 0) {
        na = n0 * n0; nb = n0 * n1d; nv = n0;
      } else if (role == 1) {
        na = n0 * n2; nb = n1d * n1d; nv = n1d;
      } else {
        na = n1d * n2; nb = n2 * n2; nv = n2;
      }
      const double U[10] = {u0 * u0, u0 * u1, u0 * u2, u0, u1 * u1, u1 * u2, u1, u2 * u2, u2, 1.0};
#pragma unroll
      for (int t = 0; t < 10; ++t) {
        acc[t] = fma(na, U[t], acc[t]);
        acc[10 + t] = fma(nb, U[t], acc[10 + t]);
      }
      const double sn = sc * nv;
      acc[20] = fma(sn, u0, acc[20]);
      acc[21] = fma(sn, u1, acc[21]);
      acc[22] = fma(sn, u2, acc[22]);
      acc[23] += sn;
      // sum phi (for the mean of the residuals): n_role (x) (u, 1)
      acc[26] = fma(nv, u0, acc[26]);
      acc[27] = fma(nv, u1, acc[27]);
      acc[28] = fma(nv, u2, acc[28]);
      acc[29] += nv;
      if (role == 0) {
        acc[24] = fma(sc, sc, acc[24]);
        acc[25] += 1.0;
      } else if (role == 1) {
        acc[24] += d;
        acc[25] = fma(d, d, acc[25]);
      } else {
        acc[24] += sc;
      }
    };
    // tiles of RSF_TILE correspondences from shared memory (the first one has been in flight since
    // kernel entry; K <= 113 000 has a single tile per block)
    for (long long t0 = i0; t0 < i1; t0 += RSF_TILE) {
      const int nt = (int)min((long long)RSF_TILE, i1 - t0);
      mbar_wait(&sf.t_bar, tile_phase);
      tile_phase ^= 1u;
      for (int e = sub; e < nt; e += 128) {
        const float4 nr = sf.t_nrm[e];
        const double d = sf.t_dist[e];
        const bool kp = pl_keep(nr.w, a.min_planarity, a.pl_signed) && (fabs(d - median) <= lim);
        if (kp) accumulate(nr, d, sf.t_xyz[3 * e + 0], sf.t_xyz[3 * e + 1], sf.t_xyz[3 * e + 2], 0.0, 0.0, 0.0);
        if (role == 0) a.keep[t0 + e] = kp ? 1 : 0;
      }
      if (t0 + RSF_TILE < i1) {
        __syncthreads();  // everybody is done with the tile before it is overwritten
        if (tid == 0) issue_tile(t0 + RSF_TILE);
      }
    }
#pragma unroll
    for (int j = 0; j < RSF_NACC; ++j) {
      const double vv = warp_sum(acc[j]);
      if (lane == 0) sf.redf[warp][j] = vv;
    }
    __syncthreads();
    if (tid < RSF_NPART) {
      const int r = tid / RSF_NACC, j = tid % RSF_NACC;
      double vv = 0.0;
      for (int ww = r; ww < RS_WARPS; ww += 3) vv += sf.redf[ww][j];
      wk.partials[(size_t)tid * G + bid] = vv;
    }
  } else if (have_tile) {
    mbar_wait(&sf.t_bar, tile_phase);  // never leave with a bulk copy into this block's shared memory in flight
  }
  RSF_STAMP(3);

  // ---- ticket: the last block to arrive owns the serial part
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned int t = atomicAdd(wk.ticket, 1u);
    sf.is_last = (t == (unsigned int)G - 1u) ? 1 : 0;
  }
  __syncthreads();
  if (!sf.is_last) return;
  __threadfence();
  // state the serial tail needs: requested now, so that the round trips overlap the partial sums
  const double prev_mean = __ldcg(&st->prev_mean), prev_std = __ldcg(&st->prev_std), w_state = __ldcg(&st->w);
  const unsigned int n_bf = a.unresolved ? __ldcg(&a.unresolved[K]) : 0u;
  if (tid == 0) {
    *wk.ticket = 0u;
    if (a.unresolved) a.unresolved[K] = 0u;  // read above (n_bf): the next match starts from a clean counter
    wk.phase_t[4] = global_timer_ns();
    wk.phase_t[28] = 2;  // fused path
  }
  // the predictor histogram has been consumed by every block: leave it zeroed for the next match
  for (int i = tid; i < LH_BINS + 2; i += RS_THREADS) wk.lin_hist[i] = 0;
  sicp_iter_record* rec = a.rec;
  if (!ok) {
    if (tid == 0) st->stop = 3;  // re-run this iteration with the general kernel (host)
    return;
  }
  if (n1 == 0) {
    if (tid == 0) {
      rec->n_kept = 0;
      rec->median = rec->mad = nan("");
      st->n_kept = 0;
    }
    return;
  }
  {
    // fixed-order sum of the per-block partials ([value][block] layout, all loads in flight)
    constexpr int NO = (RSF_NPART + RS_WARPS - 1) / RS_WARPS;
    constexpr int NB = 8;  // 32 * 8 = 256 blocks max
    double r[NO][NB];
#pragma unroll
    for (int q = 0; q < NO; ++q) {
      const int o = warp + q * RS_WARPS;
#pragma unroll
      for (int u = 0; u < NB; ++u) {
        const int b = lane + 32 * u;
        r[q][u] = (o < RSF_NPART && b < G) ? __ldcg(&wk.partials[(size_t)o * G + b]) : 0.0;
      }
    }
#pragma unroll
    for (int q = 0; q < NO; ++q) {
      const int o = warp + q * RS_WARPS;
      double vv = 0.0;
#pragma unroll
      for (int u = 0; u < NB; ++u) vv += r[q][u];
      vv = warp_sum(vv);
      if (lane == 0 && o < RSF_NPART) sf.totf[o] = vv;
    }
  }
  __syncthreads();
  if (tid == 0) wk.phase_t[17] = global_timer_ns();
  for (int e = tid; e < 169 + 13; e += RS_THREADS) {
    if (e >= 169) {
      const int o = e - 169;
      sf.m1[o] = (o == 12) ? sf.totf[2 * RSF_NACC + 24] : sf.totf[(o / 4) * RSF_NACC + 26 + (o % 4)];
      continue;
    }
    const int r = e / 13, c = e % 13;
    double vv;
    if (r == 12 && c == 12) {
      vv = sf.totf[0 * RSF_NACC + 24];
    } else if (r == 12 || c == 12) {
      const int o = (r == 12) ? c : r;
      vv = sf.totf[(o / 4) * RSF_NACC + 20 + (o % 4)];
    } else {
      int aa = r / 4, bb = r % 4, cc = c / 4, dd2 = c % 4;
      if (aa > cc) { int t = aa; aa = cc; cc = t; }
      if (bb > dd2) { int t = bb; bb = dd2; dd2 = t; }
      const int i6 = (aa == 0) ? cc : (aa == 1 ? 2 + cc : 5);
      const int i10 = (bb == 0) ? dd2 : (bb == 1 ? 3 + dd2 : (bb == 2 ? 5 + dd2 : 9));
      vv = sf.totf[(i6 / 2) * RSF_NACC + (i6 % 2) * 10 + i10];
    }
    s.M[r][c] = vv;
  }
  __syncthreads();
  if (tid == 0) wk.phase_t[18] = global_timer_ns();
  if (warp != 0) return;
  if (lane < 13) s.th_in[lane] = (lane == 12) ? 0.0 : theta_entry(Tin, cm, cf, lane);
  __syncwarp();

  const long long n_kept = (long long)(sf.totf[0 * RSF_NACC + 25] + 0.5);
  const double sum_d = sf.totf[1 * RSF_NACC + 24], sum_d2 = sf.totf[1 * RSF_NACC + 25];
  const double mean_d = (n_kept > 0) ? sum_d / (double)n_kept : nan("");
  const double var_d = (n_kept > 0) ? fmax(sum_d2 / (double)n_kept - mean_d * mean_d, 0.0) : nan("");
  const double var_d1 = (n_kept > 1) ? fmax(sum_d2 - (double)n_kept * mean_d * mean_d, 0.0) / (double)(n_kept - 1) : nan("");
  double w = w_state;
  if (a.variant) {
    w = 1.0;
  } else if (a.it == 0 || !(w > 0.0)) {
    w = a.w_param;
    if (!(w > 0.0)) w = 1.0 / var_d;
  }
  const int skip = (n_kept < 6) || !a.do_solve;
  LmOut lo;
  lo.iters = 0;
  lo.ok = 1;
  if (!skip && a.variant) {
    lin_solve(s, st->T, cf, lane);
    lo.iters = 1;
    lo.ok = s.spd;
#pragma unroll
    for (int j = 0; j < 6; ++j) lo.x[j] = s.delta[j];
  } else if (!skip) {
    lm_solve(s, a, w, st->x, cm, cf, lo, lane);
  }
  if (lane == 0) {
    wk.phase_t[19] = global_timer_ns();
    wk.phase_t[21] = s.stamp[0];
    wk.phase_t[22] = s.stamp[1];
    rec->n_kept = n_kept;
    rec->median = median;
    rec->mad = mad;
    st->pred_med = median;
    st->pred_mad = mad;
    st->pred_minpl = a.stat_minpl;
    st->pred_valid = (mad > 0.0 && isfinite(mad) && isfinite(median)) ? 1 : 0;
    rec->mean_dist = mean_d;
    rec->std_dist = sqrt(a.variant ? var_d1 : var_d);
    rec->distance_weight = w;
    rec->lm_iterations = lo.iters;
    rec->n_bruteforce = (int)n_bf;
    st->n_kept = n_kept;
    st->skip = skip;
    st->w = w;
    if (n_kept < 6 && a.do_solve && a.arm_stop) st->stop = 2;
  }
  if (skip) return;
  // new transform(s)
  Rigid T_new, T_res;
  if (a.variant) {
    const Rigid dH = rigid_from_x(lo.x);
    T_new = rigid_compose(dH, Tin);
    Rigid L;
    L.r[0] = 1.0; L.r[1] = -lo.x[2]; L.r[2] = lo.x[1];
    L.r[3] = lo.x[2]; L.r[4] = 1.0; L.r[5] = -lo.x[0];
    L.r[6] = -lo.x[1]; L.r[7] = lo.x[0]; L.r[8] = 1.0;
    L.t[0] = lo.x[3]; L.t[1] = lo.x[4]; L.t[2] = lo.x[5];
    T_res = rigid_compose(L, Tin);
  } else {
    T_new = rigid_from_x(lo.x);
    T_res = T_new;
  }
  // residual statistics at the solution from the moments: r_i = phi_i . theta
  const double th = theta_entry(T_res, cm, cf, min(lane, 12)) - s.th_in[min(lane, 12)];
  double rowdot = 0.0, s1 = 0.0;
  if (lane < 13) {
#pragma unroll
    for (int m = 0; m < 13; ++m) rowdot = fma(s.M[lane][m], __shfl_sync(0x1fffu, th, m), rowdot);
    rowdot *= th;
    s1 = sf.m1[lane] * th;
  }
  const double sum_r2 = fmax(warp_sum(rowdot), 0.0);
  const double sum_r = warp_sum(s1);
  const double n = (double)n_kept;
  const double mean = sum_r / n;
  const double sd = a.variant ? sqrt(fmax(sum_r2 - n * mean * mean, 0.0) / (n - 1.0))
                              : sqrt(fmax(sum_r2 / n - mean * mean, 0.0));
  int stop = 0;
  if (a.it > 0) {
    const double m0 = prev_mean, s0 = prev_std;
    const double cmn = (m0 == 0.0) ? ((mean == 0.0) ? 0.0 : kInf) : fabs((mean - m0) / m0 * 100.0);
    const double csd = (s0 == 0.0) ? ((sd == 0.0) ? 0.0 : kInf) : fabs((sd - s0) / s0 * 100.0);
    stop = (cmn < a.min_change && csd < a.min_change) ? 1 : 0;
  }
  if (a.variant) {
    if (lane < 6) {
      st->sigma[lane] = nan("");
      rec->x[lane] = lo.x[lane];
    }
  } else {
    if ((stop && a.arm_stop) || a.want_sigma) {
      if (lane < 36) st->An[lane] = s.Ak[lane];
      if (lane + 32 < 36) st->An[lane + 32] = s.Ak[lane + 32];
      __syncwarp();
      uncertainties(s, a, s.Ak, w, lo.x, sum_r2, n_kept, lane, st->sigma);
    }
    if (lane < 6) {
      rec->x[lane] = lo.x[lane];
      st->x[lane] = lo.x[lane];
      st->x_new[lane] = lo.x[lane];
    }
  }
  if (lane == 0) {
    if (a.variant) {
      for (int j = 0; j < 6; ++j) st->x_new[j] = lo.x[j];
      const Rigid dH = rigid_from_x(lo.x);
      const Rigid Hr = st->H_rep;
      st->H_rep = (a.variant == SICP_VARIANT_LINEARIZED_CPP) ? rigid_compose(Hr, dH) : rigid_compose(dH, Hr);
    } else {
      st->H_rep = T_new;
    }
    st->lm_ok = lo.ok;
    st->T_new = T_new;
    st->T_res = T_res;
    st->T = T_new;
    st->Tinv = rigid_inverse(T_new);
    rec->mean_res = mean;
    rec->std_res = sd;
    // predictor of the next iteration from the residuals at the new transform (see k_reject_solve)
    if (sd > 0.0 && isfinite(sd) && isfinite(mean)) {
      st->pred_med = mean;
      st->pred_mad = 0.8 * sd;
      st->pred_valid = 1;
    }
    st->prev_mean = mean;
    st->prev_std = sd;
    st->iterations_done = a.it + 1;
    if (stop && a.arm_stop) st->stop = 1;
    st->converged = stop;
    wk.phase_t[9] = global_timer_ns();
  }
}

__global__ void __launch_bounds__(RS_THREADS, 1) k_rs_fused(RSArgs a, RSWork wk) {
  extern __shared__ __align__(16) unsigned char rsf_smem[];
  rs_fused_body(a, wk, gridDim.x, blockIdx.x, *reinterpret_cast<SharedF*>(rsf_smem));
}

// Batched form: one block per pair, every per-query pointer offset by the pair's q_off.
struct BatchRsArgs {
  RSArgs proto;  // shared parameters; per-query pointers are the batch arrays' bases
  const PairDev* pairs;
  DevState* state;
  sicp_iter_record* rec;  // n_pairs x rec_stride
  int rec_stride;
  unsigned int* lin_hist;
  double* partials;
  unsigned int* ticket;
  unsigned long long* phase_t;
};
__global__ void __launch_bounds__(RS_THREADS, 1) k_rs_batch(BatchRsArgs b) {
  extern __shared__ __align__(16) unsigned char rsf_smem[];
  const int pair = blockIdx.x;
  const PairDev& pd = b.pairs[pair];
  RSArgs a = b.proto;
  const long long q = pd.q_off;
  a.K = pd.K;
  a.dist += q;
  a.q_nrm += q;
  a.q_xyz += 3 * q;
  a.keep += q;
  a.binstore += (size_t)pair * LH_BINS * a.bin_cap;
  a.m_xyz += 3 * q;
  a.state = b.state + pair;
  a.rec = b.rec + (size_t)pair * b.rec_stride + a.it;
  a.cm[0] = pd.cm[0];
  a.cm[1] = pd.cm[1];
  a.cm[2] = pd.cm[2];
  RSWork wk{};
  wk.lin_hist = b.lin_hist + (size_t)pair * (LH_BINS + 2);
  wk.partials = b.partials + (size_t)pair * RSF_NPART;
  wk.ticket = b.ticket + pair;
  wk.phase_t = b.phase_t + (size_t)pair * 32;
  rs_fused_body(a, wk, 1, 0, *reinterpret_cast<SharedF*>(rsf_smem));
}

// End of a batched run, one block per pair: residuals of the kept correspondences at the final
// transform (reference operation order), their exact two-pass mean / std, and the result record.
__global__ void __launch_bounds__(256)
    k_finish_batch(const PairDev* __restrict__ pairs, const DevState* __restrict__ state,
                   const uint8_t* __restrict__ keep, const double* __restrict__ m_xyz,
                   const double* __restrict__ q_xyz, const float4* __restrict__ q_nrm, int variant,
                   int max_iterations, sicp_pair_result* __restrict__ out) {
  const int pair = blockIdx.x;
  const PairDev& pd = pairs[pair];
  const DevState& st = state[pair];
  const long long q = pd.q_off, K = pd.K;
  __shared__ double sh[8];
  __shared__ double mean_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const Rigid Tn = st.T_res;
  const bool have = st.iterations_done > 0;
  auto resid_of = [&](long long i) {
    double tx, ty, tz;
    rigid_apply(Tn, m_xyz[3 * (q + i) + 0], m_xyz[3 * (q + i) + 1], m_xyz[3 * (q + i) + 2], tx, ty, tz);
    const float4 nr = q_nrm[q + i];
    const double dx = tx - q_xyz[3 * (q + i) + 0], dy = ty - q_xyz[3 * (q + i) + 1], dz = tz - q_xyz[3 * (q + i) + 2];
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, (double)nr.x), __dmul_rn(dy, (double)nr.y)), __dmul_rn(dz, (double)nr.z));
  };
  double acc = 0.0, cnt = 0.0;
  if (have)
    for (long long i = threadIdx.x; i < K; i += 256)
      if (keep[q + i]) {
        acc += resid_of(i);
        cnt += 1.0;
      }
  acc = warp_sum(acc);
  cnt = warp_sum(cnt);
  if (lane == 0) sh[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += sh[i];
    mean_s = t;
  }
  __syncthreads();
  // (count reduced the same way)
  if (lane == 0) sh[warp] = cnt;
  __syncthreads();
  double n = 0.0;
  for (int i = 0; i < 8; ++i) n += sh[i];
  const double mean = (n > 0.0) ? mean_s / n : nan("");
  __syncthreads();
  acc = 0.0;
  if (have)
    for (long long i = threadIdx.x; i < K; i += 256)
      if (keep[q + i]) {
        const double d = resid_of(i) - mean;
        acc = fma(d, d, acc);
      }
  acc = warp_sum(acc);
  if (lane == 0) sh[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += sh[i];
    sicp_pair_result r;
    r.iterations = st.iterations_done;
    r.converged = (st.stop == 1) ? 1 : 0;
    r.n_selected = (int32_t)K;
    r.n_kept = st.n_kept;
    // fewer than 6 correspondences at some iteration (stop 2, or an iteration that never finished)
    const bool too_few = (st.stop == 2) || (!st.stop && st.iterations_done < max_iterations) || !have;
    r.status = too_few ? SICP_ERR_TOO_FEW_CORR : (st.lm_ok ? SICP_OK : SICP_ERR_SINGULAR);
    if (K == 0) r.status = SICP_ERR_NO_OVERLAP;  // the overlap filter kept no fixed point: the pair never ran
    const Rigid& H = variant ? st.H_rep : st.T;
    for (int a = 0; a < 3; ++a) {
      for (int c2 = 0; c2 < 3; ++c2) r.H[a * 4 + c2] = H.r[a * 3 + c2];
      r.H[a * 4 + 3] = H.t[a];
    }
    r.H[12] = r.H[13] = r.H[14] = 0.0;
    r.H[15] = 1.0;
    for (int j = 0; j < 6; ++j) {
      r.x[j] = variant ? st.x_new[j] : st.x[j];
      r.sigma[j] = st.sigma[j];
    }
    r.mean_res = mean;
    r.std_res = (n > 0.0) ? (variant ? sqrt(t / (n - 1.0)) : sqrt(t / n)) : nan("");
    out[pair] = r;
  }
}

// Residual vector of the LAST iteration (reference operation order, optimization.py:117-124) for
// the kept correspondences, from the matched points the match kernel stored.  One launch after
// the loop; the compaction and the exact two-pass statistics follow (k_resid_stats).
__global__ void __launch_bounds__(256)
    k_final_residuals(const DevState* __restrict__ st, const uint8_t* __restrict__ keep,
                      const double* __restrict__ m_xyz, const double* __restrict__ q_xyz,
                      const float4* __restrict__ q_nrm, long long K, double* __restrict__ resid) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K || !keep[i]) return;
  const Rigid Tn = st->T_res;
  double tx, ty, tz;
  rigid_apply(Tn, m_xyz[3 * i + 0], m_xyz[3 * i + 1], m_xyz[3 * i + 2], tx, ty, tz);
  const float4 nr = q_nrm[i];
  const double dx = tx - q_xyz[3 * i + 0], dy = ty - q_xyz[3 * i + 1], dz = tz - q_xyz[3 * i + 2];
  resid[i] = __dadd_rn(__dadd_rn(__dmul_rn(dx, (double)nr.x), __dmul_rn(dy, (double)nr.y)),
                       __dmul_rn(dz, (double)nr.z));
}

// Exact statistics of the compacted residuals: mean first, then the squared deviations from it
// (two passes, one block, fixed order) — written over the moment-based values of the last record.
__global__ void __launch_bounds__(1024)
    k_resid_stats(const double* __restrict__ r, const DevState* __restrict__ st, int sample_std,
                  sicp_iter_record* __restrict__ rec_base) {
  __shared__ double sh[32];
  __shared__ double mean_s;
  const long long n = st->n_kept;
  const int it = st->iterations_done - 1;
  if (n <= 0 || it < 0) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += 1024) acc += r[i];
  acc = warp_sum(acc);
  if (lane == 0) sh[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 32; ++i) t += sh[i];
    mean_s = t / (double)n;
  }
  __syncthreads();
  const double mean = mean_s;
  acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += 1024) {
    const double d = r[i] - mean;
    acc = fma(d, d, acc);
  }
  acc = warp_sum(acc);
  __syncthreads();
  if (lane == 0) sh[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 32; ++i) t += sh[i];
    rec_base[it].mean_res = mean;
    rec_base[it].std_res = sample_std ? sqrt(t / (double)(n - 1)) : sqrt(t / (double)n);
  }
}

// Ordered compaction of the kept residuals (final iteration only): block-level scan, one block
// per 4096 elements, two kernels.
__global__ void __launch_bounds__(256)
    k_compact_count(const uint8_t* __restrict__ keep, long long K, unsigned int* __restrict__ bsum) {
  const long long base = (long long)blockIdx.x * 4096;
  unsigned int c = 0;
  for (int j = threadIdx.x; j < 4096; j += 256)
    if (base + j < K) c += keep[base + j] ? 1u : 0u;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  __shared__ unsigned int sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = 0;
    for (int i = 0; i < 8; ++i) t += sh[i];
    bsum[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256)
    k_compact_write(const uint8_t* __restrict__ keep, const double* __restrict__ resid, long long K,
                    const unsigned int* __restrict__ bsum, double* __restrict__ out) {
  // offset of this block = sum of previous block counts (few hundred blocks at most)
  __shared__ unsigned int boff;
  __shared__ unsigned int wsum[8];
  if (threadIdx.x == 0) {
    unsigned int t = 0;
    for (unsigned int b = 0; b < blockIdx.x; ++b) t += bsum[b];
    boff = t;
  }
  __syncthreads();
  const long long base = (long long)blockIdx.x * 4096 + threadIdx.x * 16;
  unsigned int flags = 0, c = 0;
#pragma unroll
  for (int j = 0; j < 16; ++j)
    if (base + j < K && keep[base + j]) {
      flags |= 1u << j;
      ++c;
    }
  unsigned int incl = c;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  unsigned int woff = 0;
  for (int i = 0; i < w; ++i) woff += wsum[i];
  unsigned int pos = boff + woff + incl - c;
#pragma unroll
  for (int j = 0; j < 16; ++j)
    if (flags & (1u << j)) out[pos++] = resid[base + j];
}

}  // namespace

void reject_solve_launch(Ctx& c, const sicp_run_params& p, int it, bool do_solve, bool arm_stop,
                         int rec_slot) {
  const long long K = c.K;
  const bool multi = K > 4096;
  int G = 1;
  if (multi) {
    const int cap = (c.rs_blocks > 0) ? std::min(c.rs_blocks, c.num_sms) : std::min(c.num_sms, 256);
    G = (int)std::min<long long>(cap, (K + RS_THREADS - 1) / RS_THREADS);
  }
  // workspace: two parities
  const size_t hist_n = 2ull * RS_LEVELS * RS_BINS;
  if (c.ws.hist.cap < 2 * hist_n) {
    c.ws.hist.reserve(2 * hist_n);
    SICP_CUDA(cudaMemsetAsync(c.ws.hist.p, 0, 2 * hist_n * sizeof(unsigned int), c.stream));
    c.ws.cand.reserve(2ull * 2 * RS_CAP);
    c.ws.counters.reserve(64);
    SICP_CUDA(cudaMemsetAsync(c.ws.counters.p, 0, 64 * sizeof(unsigned int), c.stream));
    c.ws.minkey.reserve(16);
    SICP_CUDA(cudaMemsetAsync(c.ws.minkey.p, 0xff, 16 * sizeof(unsigned long long), c.stream));
    c.rs_parity = 0;
  }
  c.ws.partials.reserve((size_t)c.num_sms * (RS_NPART + 2) + 16);
  c.keep.reserve(K);
  c.resid.reserve(K);
  const int par = c.rs_parity;
  c.rs_parity ^= 1;

  RSArgs a;
  a.K = K;
  a.dist = c.dist.p;
  a.q_nrm = c.mov_attr ? c.q_nrm_eff.p : c.q_nrm.p;
  a.pl_signed = c.mov_attr ? 1 : 0;
  a.q_xyz = c.q_xyz.p;
  a.nn_idx = c.nn_idx.p;
  a.mov_xyz = c.mov_xyz.p;
  a.keep = c.keep.p;
  a.resid = c.resid.p;
  a.unresolved = (c.nn_engine == SICP_NN_AUTO) ? c.unresolved.p : nullptr;
  a.state = c.dev_state.p;
  a.rec = c.ws.rec.p + rec_slot;
  a.min_planarity = p.min_planarity;
  a.variant = c.variant;
  a.stat_minpl = c.variant ? -kInf : p.min_planarity;
  a.min_change = p.min_change;
  a.w_param = p.lsq.distance_weight;
  for (int j = 0; j < 6; ++j) {
    a.obs[j] = p.lsq.observed[j];
    a.wobs[j] = p.lsq.obs_weight[j];
  }
  for (int j = 0; j < 3; ++j) a.cm[j] = c.mov_center[j];
  a.it = it;
  a.do_solve = do_solve ? 1 : 0;
  a.arm_stop = arm_stop ? 1 : 0;
  c.lin_hist.reserve(LH_BINS + 2);
  if (!c.lin_hist_init) {
    SICP_CUDA(cudaMemsetAsync(c.lin_hist.p, 0, (LH_BINS + 2) * sizeof(unsigned int), c.stream));
    c.lin_hist_init = true;
  }
  a.hist_expected = c.lin_hist_pending ? 1 : 0;
  c.lin_hist_pending = false;  // the kernel leaves the histogram zeroed

  RSWork wk;
  wk.hist = c.ws.hist.p + par * hist_n;
  wk.hist_other = c.ws.hist.p + (par ^ 1) * hist_n;
  wk.cand = c.ws.cand.p + par * 2 * RS_CAP;
  wk.counters = c.ws.counters.p + par * 2;
  wk.counters_other = c.ws.counters.p + (par ^ 1) * 2;
  wk.minkey = c.ws.minkey.p + par * 2;
  wk.minkey_other = c.ws.minkey.p + (par ^ 1) * 2;
  wk.partials = c.ws.partials.p;
  c.phase_t.reserve(32);
  wk.phase_t = c.phase_t.p;
  if (c.grid_bar.p == nullptr) {
    c.grid_bar.reserve(2);
    SICP_CUDA(cudaMemsetAsync(c.grid_bar.p, 0, 2 * sizeof(unsigned int), c.stream));
  }
  wk.barrier = c.grid_bar.p;
  wk.lin_hist = c.lin_hist.p;

  if (multi) {
    void* args[] = {&a, &wk};
    SICP_CUDA(cudaLaunchCooperativeKernel((void*)k_reject_solve<true>, dim3(G), dim3(RS_THREADS),
                                          args, 0, c.stream));
  } else {
    k_reject_solve<false><<<1, RS_THREADS, 0, c.stream>>>(a, wk);
    SICP_CUDA(cudaGetLastError());
  }
  c.tm.kernel_launches += 1;
}

// Launch of the barrier-free kernel (iterations whose predecessor left a valid predictor).
void rs_fused_launch(Ctx& c, const sicp_run_params& p, int it, bool arm_stop, int rec_slot,
                     bool want_sigma) {
  const long long K = c.K;
  // K <= 4096: a single block (it never needs the host's re-run protocol, see rs_fused_body)
  const int G = (K <= 4096) ? 1 : (int)std::min<long long>(c.num_sms, std::max<long long>(1, (K + 767) / 768));
  if (!c.rsf_attr_set) {
    SICP_CUDA(cudaFuncSetAttribute(k_rs_fused, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)sizeof(SharedF)));
    c.rsf_attr_set = true;
  }
  c.ws.partials.reserve((size_t)c.num_sms * (RSF_NPART + 2) + 16);
  c.keep.reserve(K);
  c.resid.reserve(K);
  c.phase_t.reserve(32);
  if (c.rsf_ticket.p == nullptr) {
    c.rsf_ticket.reserve(4);
    SICP_CUDA(cudaMemsetAsync(c.rsf_ticket.p, 0, 4 * sizeof(unsigned int), c.stream));
  }
  RSArgs a;
  a.K = K;
  a.dist = c.dist.p;
  a.q_nrm = c.mov_attr ? c.q_nrm_eff.p : c.q_nrm.p;
  a.pl_signed = c.mov_attr ? 1 : 0;
  a.q_xyz = c.q_xyz.p;
  a.nn_idx = c.nn_idx.p;
  a.mov_xyz = c.mov_xyz.p;
  a.keep = c.keep.p;
  a.resid = c.resid.p;
  a.unresolved = (c.nn_engine == SICP_NN_AUTO) ? c.unresolved.p : nullptr;
  a.state = c.dev_state.p;
  a.rec = c.ws.rec.p + rec_slot;
  a.min_planarity = p.min_planarity;
  a.variant = c.variant;
  a.stat_minpl = c.variant ? -kInf : p.min_planarity;
  a.min_change = p.min_change;
  a.w_param = p.lsq.distance_weight;
  for (int j = 0; j < 6; ++j) {
    a.obs[j] = p.lsq.observed[j];
    a.wobs[j] = p.lsq.obs_weight[j];
  }
  for (int j = 0; j < 3; ++j) a.cm[j] = c.mov_center[j];
  a.it = it;
  a.do_solve = 1;
  a.arm_stop = arm_stop ? 1 : 0;
  a.hist_expected = c.lin_hist_pending ? 1 : 0;
  c.lin_hist_pending = false;  // the kernel leaves the histogram zeroed
  a.binstore = c.binstore.p;
  a.bin_cap = c.bin_cap;
  a.m_xyz = c.m_xyz.p;
  a.want_sigma = want_sigma ? 1 : 0;
  RSWork wk{};
  wk.partials = c.ws.partials.p;
  wk.phase_t = c.phase_t.p;
  wk.lin_hist = c.lin_hist.p;
  wk.ticket = c.rsf_ticket.p;
  launch_kernel(k_rs_fused, dim3(G), dim3(RS_THREADS), sizeof(SharedF), c.stream, c.pdl != 0, a, wk);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

void batch_rs_launch(Ctx& c, Batch& b, const sicp_run_params& p, int it, bool want_sigma) {
  if (!c.rsb_attr_set) {
    SICP_CUDA(cudaFuncSetAttribute(k_rs_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SharedF)));
    c.rsb_attr_set = true;
  }
  BatchRsArgs ba;
  RSArgs& a = ba.proto;
  a = RSArgs{};
  a.dist = b.dist.p;
  a.q_nrm = b.q_nrm.p;
  a.pl_signed = 0;
  a.q_xyz = b.q_xyz.p;
  a.keep = b.keep.p;
  a.binstore = b.binstore.p;
  a.bin_cap = b.bin_cap;
  a.m_xyz = b.m_xyz.p;
  a.min_planarity = p.min_planarity;
  a.variant = c.variant;
  a.stat_minpl = c.variant ? -kInf : p.min_planarity;
  a.min_change = p.min_change;
  a.w_param = p.lsq.distance_weight;
  for (int j = 0; j < 6; ++j) {
    a.obs[j] = p.lsq.observed[j];
    a.wobs[j] = p.lsq.obs_weight[j];
  }
  a.it = it;
  a.do_solve = 1;
  a.arm_stop = 1;
  a.hist_expected = 1;  // every batched match feeds the per-pair histogram (when its predictor is valid)
  a.want_sigma = want_sigma ? 1 : 0;
  ba.pairs = b.pairs.p;
  ba.state = b.state.p;
  ba.rec = b.rec.p;
  ba.rec_stride = p.max_iterations;
  ba.lin_hist = b.lin_hist.p;
  ba.partials = b.partials.p;
  ba.ticket = b.ticket.p;
  ba.phase_t = b.phase_t.p;
  launch_kernel(k_rs_batch, dim3(b.n_pairs), dim3(RS_THREADS), sizeof(SharedF), c.stream, c.pdl != 0, ba);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

void batch_finish_launch(Ctx& c, Batch& b, int max_iterations) {
  k_finish_batch<<<b.n_pairs, 256, 0, c.stream>>>(b.pairs.p, b.state.p, b.keep.p, b.m_xyz.p, b.q_xyz.p, b.q_nrm.p,
                                                  c.variant, max_iterations, b.results.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

// Residual vector, ordered compaction and exact statistics of the final iteration.
void final_residuals_launch(Ctx& c) {
  const long long K = c.K;
  c.resid.reserve(K);
  k_final_residuals<<<(unsigned)((K + 255) / 256), 256, 0, c.stream>>>(
      c.dev_state.p, c.keep.p, c.m_xyz.p, c.q_xyz.p, c.q_nrm.p, K, c.resid.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
  compact_residuals_launch(c);
  k_resid_stats<<<1, 1024, 0, c.stream>>>(c.resid_compact.p, c.dev_state.p, c.variant != SICP_VARIANT_PYTHON,
                                         c.ws.rec.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 1;
}

void compact_residuals_launch(Ctx& c) {
  const long long K = c.K;
  const unsigned int nb = (unsigned int)((K + 4095) / 4096);
  c.ws.counters.reserve(64);
  c.compact_sums.reserve(nb + 1);
  c.resid_compact.reserve(std::max<long long>(K, 1));
  k_compact_count<<<nb, 256, 0, c.stream>>>(c.keep.p, K, c.compact_sums.p);
  k_compact_write<<<nb, 256, 0, c.stream>>>(c.keep.p, c.resid.p, K, c.compact_sums.p,
                                           c.resid_compact.p);
  SICP_CUDA(cudaGetLastError());
  c.tm.kernel_launches += 2;
}

}  // namespace sicp
