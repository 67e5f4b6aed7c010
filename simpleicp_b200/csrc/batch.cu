// batch.cu — sicp_register_batch: SimpleICP.run (python/simpleicp/simpleicp.py:75-324) for many
// independent pairs with ONE set of launches per stage and per iteration (BASELINE.json
// configs[4]: 512 pairs of 100 000 points, 64 per GPU; SURVEY.md section 8e).
//
// A registration of a 100 000-point pair with 1000 correspondences is far too small to fill a
// B200: one match launch has 16 000 threads, one reject/solve launch one block, and the host
// drives ~30 launches per iteration-loop through a Python thread.  Here every kernel carries a
// pair dimension instead:
//   upload        one cudaMemcpyAsync per cloud straight from the caller's (pinned) arrays; the
//                 movable clouds cross PCIe while the fixed-side work runs
//   grids         segmented counting sort over all clouds of a side (grid.cu: grid_build_batch)
//   overlap       (max_overlap_distance only) keep flags of all fixed points in one launch, one
//                 scan over the batch, ordered kept lists; per-pair K set on the device (nn.cu)
//   select+gather rint(linspace) picks and their coordinates, all pairs in one launch
//   normals       k-NN + PCA, blockIdx.y = pair
//   loop          per iteration ONE match launch over (pair, query) and ONE reject/solve launch
//                 with a block per pair (the barrier-free kernel with G = 1: predictor histogram
//                 select, or the in-block radix select when there is no usable prediction), every
//                 pair with its own device-resident state and stop flag
//   finish        exact residual statistics + result record per pair, one small download
// No host work per pair except the two copies.
#include <algorithm>
#include <cstring>
#include <vector>

#include "ctx.cuh"

namespace sicp {

namespace {

__global__ void k_gather_flags(const DevState* __restrict__ st, int n, int* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  flags[2 * i + 0] = st[i].stop;
  flags[2 * i + 1] = st[i].iterations_done;
}

template <typename T>
void pinned_reserve(T*& p, size_t& cap, size_t n) {
  if (n <= cap) return;
  if (p) cudaFreeHost(p);
  p = nullptr;
  SICP_CUDA(cudaMallocHost(&p, n * sizeof(T)));
  cap = n;
}

}  // namespace

static void register_batch(Ctx& c, int n_pairs, const double* const* fix_xyz, const int64_t* n_fix,
                           const double* const* mov_xyz, const int64_t* n_mov,
                           const sicp_register_params* rp, sicp_pair_result* out) {
  SICP_REQUIRE(n_pairs >= 1 && n_pairs <= 65535, SICP_ERR_BAD_ARG, "n_pairs must be in [1, 65535]");
  SICP_REQUIRE(fix_xyz && n_fix && mov_xyz && n_mov && rp && out, SICP_ERR_BAD_ARG, "NULL argument");
  SICP_REQUIRE(rp->correspondences >= 1 && rp->correspondences <= 4096, SICP_ERR_BAD_ARG,
               "the batched engine runs one block per pair: correspondences must be in [1, 4096]");
  // the same rule as sicp_register: anything else means the clouds fully overlap
  const bool overlap = rp->max_overlap_distance > 0 && std::isfinite(rp->max_overlap_distance);
  const sicp_run_params& p = rp->run;
  SICP_REQUIRE(p.max_iterations >= 1 && p.max_iterations <= 4096, SICP_ERR_BAD_ARG,
               "max_iterations must be in [1, 4096]");
  bool any_finite = false;
  for (int j = 0; j < 6; ++j) {
    SICP_REQUIRE(p.lsq.obs_weight[j] >= 0, SICP_ERR_BAD_ARG,
                 "All elements of rbp_observation_weights must be >= 0.");
    any_finite = any_finite || std::isfinite(p.lsq.obs_weight[j]);
    SICP_REQUIRE(c.variant == SICP_VARIANT_PYTHON || p.lsq.obs_weight[j] == 0.0, SICP_ERR_BAD_ARG,
                 "the linearised variants have no observed or fixed parameters");
  }
  SICP_REQUIRE(any_finite, SICP_ERR_BAD_ARG, "At least one element in rbp_observation_weights must be finite.");
  if (!c.batch) c.batch = new Batch();
  Batch& b = *c.batch;
  b.n_pairs = n_pairs;
  std::vector<long long> fo((size_t)n_pairs + 1, 0), mo((size_t)n_pairs + 1, 0);
  long long Kmax = 0;
  for (int i = 0; i < n_pairs; ++i) {
    SICP_REQUIRE(fix_xyz[i] && mov_xyz[i], SICP_ERR_BAD_ARG, "cloud pointer is NULL");
    SICP_REQUIRE(n_fix[i] >= rp->neighbors && n_mov[i] >= 1, SICP_ERR_BAD_ARG,
                 "every fixed cloud needs at least `neighbors` points, every movable cloud one");
    fo[(size_t)i + 1] = fo[(size_t)i] + n_fix[i];
    mo[(size_t)i + 1] = mo[(size_t)i] + n_mov[i];
    Kmax = std::max<long long>(Kmax, std::min<long long>(rp->correspondences, n_fix[i]));
  }
  Kmax = (Kmax + 1) & ~1ll;  // even: every pair's slice of the per-query arrays starts 16-byte aligned
  b.total_fix = fo[(size_t)n_pairs];
  b.total_mov = mo[(size_t)n_pairs];
  b.Kmax = Kmax;
  cudaStream_t st = c.stream;

  // ---- uploads: fixed clouds on the context's stream, movable ones behind them on the copy stream
  b.fix_xyz.reserve(3 * (size_t)b.total_fix);
  b.mov_xyz.reserve(3 * (size_t)b.total_mov);
  SICP_CUDA(cudaEventRecord(c.ev_user, st));
  SICP_CUDA(cudaStreamWaitEvent(c.copy_stream, c.ev_user, 0));  // buffers of an earlier call are free
  for (int i = 0; i < n_pairs; ++i)
    SICP_CUDA(cudaMemcpyAsync(b.fix_xyz.p + 3 * fo[(size_t)i], fix_xyz[i], sizeof(double) * 3 * (size_t)n_fix[i],
                              cudaMemcpyDefault, st));
  for (int i = 0; i < n_pairs; ++i)
    SICP_CUDA(cudaMemcpyAsync(b.mov_xyz.p + 3 * mo[(size_t)i], mov_xyz[i], sizeof(double) * 3 * (size_t)n_mov[i],
                              cudaMemcpyDefault, c.copy_stream));
  SICP_CUDA(cudaEventRecord(c.ev_copy, c.copy_stream));

  // ---- per-pair buffers
  const size_t nq = (size_t)n_pairs * (size_t)Kmax;
  b.pairs.reserve(n_pairs);
  b.sel_idx.reserve(nq);
  b.nn_idx.reserve(nq);
  b.q_xyz.reserve(3 * nq);
  b.dist.reserve(nq);
  b.m_xyz.reserve(3 * nq);
  b.q_nrm.reserve(nq);
  b.bin_cap = bin_cap_for(Kmax);
  b.binstore.reserve((size_t)n_pairs * LH_BINS * (size_t)b.bin_cap);
  b.nn_pos.reserve(nq);
  b.keep.reserve(nq);
  b.state.reserve(n_pairs);
  b.lin_hist.reserve((size_t)n_pairs * (LH_BINS + 2));
  b.rec.reserve((size_t)n_pairs * (size_t)p.max_iterations);
  b.partials.reserve((size_t)n_pairs * 96 + 16);
  b.ticket.reserve(n_pairs);
  b.phase_t.reserve((size_t)n_pairs * 32);
  b.flags.reserve(2 * (size_t)n_pairs);
  b.results.reserve(n_pairs);
  pinned_reserve(b.flags_host, b.flags_cap, 2 * (size_t)n_pairs);
  pinned_reserve(b.results_host, b.results_cap, (size_t)n_pairs);
  SICP_CUDA(cudaMemsetAsync(b.lin_hist.p, 0, sizeof(unsigned int) * (size_t)n_pairs * (LH_BINS + 2), st));
  SICP_CUDA(cudaMemsetAsync(b.ticket.p, 0, sizeof(unsigned int) * (size_t)n_pairs, st));
  SICP_CUDA(cudaMemsetAsync(b.rec.p, 0, sizeof(sicp_iter_record) * (size_t)n_pairs * (size_t)p.max_iterations, st));
  SICP_CUDA(cudaMemsetAsync(b.nn_pos.p, 0xff, sizeof(uint32_t) * nq, st));
  SICP_CUDA(cudaMemsetAsync(b.keep.p, 0, nq, st));
  {
    DevState h;
    std::memset(&h, 0, sizeof(h));
    for (int j = 0; j < 6; ++j) h.x[j] = p.lsq.x0[j];
    h.T = rigid_from_x(h.x);
    h.Tinv = rigid_inverse(h.T);
    h.T_res = h.T;
    h.H_rep = h.T;
    std::vector<DevState> hs((size_t)n_pairs, h);
    SICP_CUDA(cudaMemcpyAsync(b.state.p, hs.data(), sizeof(DevState) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
    if (overlap) {
      b.fix_off.reserve((size_t)n_pairs + 1);
      SICP_CUDA(cudaMemcpyAsync(b.fix_off.p, fo.data(), sizeof(long long) * ((size_t)n_pairs + 1), cudaMemcpyHostToDevice, st));
    }
    SICP_CUDA(cudaStreamSynchronize(st));  // hs is a local (also: the fixed clouds have arrived)
  }

  // ---- fixed side: grids, subsample + gather, normals (the movable clouds are still in flight).
  // With the overlap filter the selection needs the movable grids: fixed grids, movable grids,
  // filter, select + gather, normals.
  std::vector<PairDev> pd((size_t)n_pairs);
  std::vector<BatchHostCloud> clouds((size_t)n_pairs);
  std::vector<GridView> views;
  std::vector<double> centres;
  for (int i = 0; i < n_pairs; ++i) clouds[(size_t)i] = BatchHostCloud{b.fix_xyz.p + 3 * fo[(size_t)i], n_fix[i], fo[(size_t)i]};
  {
    StageTimer t(c, &c.tm.grid_fix_ms);
    grid_build_batch(c, b, b.gfix, clouds, views, centres);
    t.stop();
  }
  for (int i = 0; i < n_pairs; ++i) {
    PairDev& d = pd[(size_t)i];
    std::memset(&d, 0, sizeof(d));
    d.gfix = views[(size_t)i];
    d.n_fix = n_fix[i];
    d.n_mov = n_mov[i];
    d.fix_off = fo[(size_t)i];
    d.mov_off = mo[(size_t)i];
    d.K = std::min<long long>(rp->correspondences, n_fix[i]);
    d.q_off = (long long)i * Kmax;
    d.n_cand = n_fix[i];
  }
  auto fixed_side = [&]() {
    batch_select_gather_launch(c, b, rp->correspondences, c.variant != SICP_VARIANT_PYTHON, overlap);
    StageTimer t(c, &c.tm.normals_ms);
    batch_normals_launch(c, b, rp->neighbors);
    t.stop();
  };
  if (!overlap) {
    SICP_CUDA(cudaMemcpyAsync(b.pairs.p, pd.data(), sizeof(PairDev) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
    fixed_side();
  }

  // ---- movable side
  SICP_CUDA(cudaStreamWaitEvent(st, c.ev_copy, 0));
  for (int i = 0; i < n_pairs; ++i) clouds[(size_t)i] = BatchHostCloud{b.mov_xyz.p + 3 * mo[(size_t)i], n_mov[i], mo[(size_t)i]};
  {
    StageTimer t(c, &c.tm.grid_mov_ms);
    grid_build_batch(c, b, b.gmov, clouds, views, centres);
    t.stop();
  }
  for (int i = 0; i < n_pairs; ++i) {
    pd[(size_t)i].gmov = views[(size_t)i];
    for (int a = 0; a < 3; ++a) pd[(size_t)i].cm[a] = centres[(size_t)i * 3 + a];
  }
  SICP_CUDA(cudaMemcpyAsync(b.pairs.p, pd.data(), sizeof(PairDev) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
  c.tm.overlap_ms = 0;
  if (overlap) {
    // the filter sets K, n_cand and kept_off of every descriptor on the device: nothing re-uploads
    // them after this point
    StageTimer t(c, &c.tm.overlap_ms);
    batch_overlap_launch(c, b, rp->correspondences, rp->max_overlap_distance);
    t.stop();
    fixed_side();
  }

  // ---- the loop: two launches per iteration for the whole batch
  cudaEvent_t e0, e1;
  SICP_CUDA(cudaEventCreate(&e0));
  SICP_CUDA(cudaEventCreate(&e1));
  SICP_CUDA(cudaEventRecord(e0, st));
  const int every = std::max(1, c.host_sync_every);
  int next_sync = 1;
  for (int it = 0; it < p.max_iterations; ++it) {
    batch_match_launch(c, b, c.warm_start && it > 0);
    batch_rs_launch(c, b, p, it, it + 1 == p.max_iterations);
    if (it >= next_sync || it + 1 == p.max_iterations) {
      next_sync = it + every;
      k_gather_flags<<<(n_pairs + 127) / 128, 128, 0, st>>>(b.state.p, n_pairs, b.flags.p);
      SICP_CUDA(cudaMemcpyAsync(b.flags_host, b.flags.p, sizeof(int) * 2 * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
      SICP_CUDA(cudaStreamSynchronize(st));
      bool running = false;
      for (int i = 0; i < n_pairs; ++i) {
        const int stop = b.flags_host[2 * i], done = b.flags_host[2 * i + 1];
        // a pair without a stop flag that is not keeping up ran out of correspondences (< 6): it
        // stays where it is; everybody else decides
        if (stop == 0 && done == it + 1) running = true;
      }
      if (!running) break;
    }
  }
  SICP_CUDA(cudaEventRecord(e1, st));
  batch_finish_launch(c, b, p.max_iterations);
  SICP_CUDA(cudaMemcpyAsync(b.results_host, b.results.p, sizeof(sicp_pair_result) * (size_t)n_pairs,
                            cudaMemcpyDeviceToHost, st));
  SICP_CUDA(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  c.tm.reject_solve_ms = ms;
  std::memcpy(out, b.results_host, sizeof(sicp_pair_result) * (size_t)n_pairs);
}

}  // namespace sicp

using namespace sicp;

extern "C" int32_t sicp_register_batch(sicp_ctx* ctx, int32_t n_pairs, const double* const* fix_xyz,
                                       const int64_t* n_fix, const double* const* mov_xyz,
                                       const int64_t* n_mov, const sicp_register_params* p,
                                       sicp_pair_result* out) {
  if (!ctx) {
    sicp::set_thread_error("sicp_ctx is NULL");
    return SICP_ERR_BAD_ARG;
  }
  Ctx& c = ctx->c;
  try {
    SICP_CUDA(cudaSetDevice(c.device));
    register_batch(c, n_pairs, fix_xyz, n_fix, mov_xyz, n_mov, p, out);
  } catch (const sicp::Error& e) {
    c.err = e.msg;
    sicp::set_thread_error(e.msg);
    if (e.code == SICP_ERR_CUDA) cudaGetLastError();
    return e.code;
  } catch (const std::exception& e) {
    c.err = e.what();
    sicp::set_thread_error(c.err);
    return SICP_ERR_CUDA;
  }
  return SICP_OK;
}
