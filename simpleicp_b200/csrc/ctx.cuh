// ctx.cuh — the context behind sicp_ctx and the stage entry points each .cu implements.
#pragma once
#include "common.cuh"
#include "reject_solve.cuh"
#include "upload.cuh"

namespace sicp {

// Cell-sorted copy of one cloud + its uniform grid (HBM resident, L2 resident for <= ~2M points).
struct Grid {
  DevBuf<Rec> recs;              // n points, sorted by cell
  DevBuf<uint32_t> cell_start;   // n_cells + 1
  DevBuf<uint32_t> cid;          // scratch: cell id per point
  DevBuf<uint32_t> fill;         // scratch: per-cell counter
  DevBuf<uint32_t> block_sums;   // scratch for the scan
  double o[3] = {0, 0, 0};
  double h = 1.0;
  int dims[3] = {1, 1, 1};
  long long n = 0;
  long long n_cells = 0;
  long long n_occupied = 0;
  bool built = false;
  GridView view() const {
    GridView v;
    v.recs = recs.p;
    v.cell_start = cell_start.p;
    v.ox = o[0];
    v.oy = o[1];
    v.oz = o[2];
    v.h = h;
    v.inv_h = 1.0 / h;
    v.nx = dims[0];
    v.ny = dims[1];
    v.nz = dims[2];
    v.n_points = n;
    return v;
  }
};

// Workspace of the fused reject + solve kernel (all device memory).
struct SolveWs {
  DevBuf<unsigned int> hist;        // radix histograms: 2 selects x levels x bins
  DevBuf<unsigned long long> cand;  // candidate keys for the in-block sort, 2 selects
  DevBuf<unsigned int> counters;    // small atomic counters / flags
  DevBuf<unsigned long long> minkey;  // min key above the selected bin, per select
  DevBuf<double> partials;          // per-block partial sums
  DevBuf<double> scal;              // broadcast scalars: median, mad, x, ...
  DevBuf<sicp_iter_record> rec;     // device copy of the per-iteration record ring
};

struct Batch;

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int num_sms = 148;
  std::string err;

  // options
  int nn_engine = SICP_NN_AUTO;
  int sign_mode = SICP_SIGN_DGEEV;
  int variant = SICP_VARIANT_PYTHON;
  double grid_target_occ = 3.0;
  int grid_max_rings = 8;
  int host_sync_every = 4;
  int grid_sort_cells = 0;  // 1: sort the records inside each cell by index (layout only)
  int rs_blocks = 0;     // blocks of the cooperative reject/solve kernel (0 = one per SM)
  int match_group = 0;   // lanes cooperating on one grid query: 0 = by K, else 1, 4, 8 or 16

  // clouds
  DevBuf<double> fix_xyz, mov_xyz;
  long long n_fix = 0, n_mov = 0;
  DevBuf<float4> mov_f4;  // centred float copy in caller order, for the TMA brute-force engine
  double mov_center[3] = {0, 0, 0};
  double mov_radius = 0;  // max |centred coordinate|
  Grid gmov, gfix;

  // selection (ascending fixed-cloud indices) and per-query data
  long long K = 0;
  DevBuf<long long> sel_idx;
  DevBuf<long long> sel_tmp;
  DevBuf<double> q_xyz;   // K x 3 gathered fixed points
  DevBuf<float4> q_nrm;   // (nx, ny, nz, planarity) float32 as the reference stores them
  bool have_normals = false;
  // movable-side attributes (sicp_set_mov_normals): per movable point, in its own frame
  DevBuf<float4> mov_nrm;
  DevBuf<float4> q_nrm_eff;  // K: fixed normal + effective planarity of the current match (nn.cu: effective_planarity)
  bool mov_attr = false;
  double mov_cos_max = -1.0; // cos(max angle between normals); < 0 = no angle test
  int knn_k = 0;
  DevBuf<long long> knn_idx;
  DevBuf<double> knn_d2;
  DevBuf<uint32_t> knn_pos;  // K x k record positions (cooperative k-NN kernel -> PCA kernel)
  int keep_knn = 0;          // option "keep_knn": store neighbour indices / distances for sicp_get_knn
  int knn_coop = -1;         // option "knn_coop": 1 cooperative lanes (k <= 16), 0 one thread per query, -1 by K

  // per-iteration arrays
  DevBuf<long long> nn_idx;
  DevBuf<double> dist;
  DevBuf<uint8_t> keep;
  DevBuf<unsigned int> binstore;     // LH_BINS x bin_cap: members of every predictor-histogram bin (match -> fused reject/solve)
  int bin_cap = 0;
  DevBuf<double> m_xyz;              // K x 3: matched movable point, caller coordinates
  DevBuf<uint32_t> nn_pos;           // K: record position of the last match (warm start of the next one)
  bool nn_pos_valid = false;         // nn_pos belongs to the current movable grid and selection
  long long nn_pos_K = 0;
  int warm_start = 1;                // option "warm_start"
  int sphere_scan = 1;               // option "sphere_scan"
  int pdl = 1;                       // option "pdl": programmatic dependent launch between the two kernels of an iteration
  bool unresolved_clean = false;     // unresolved[K] is zero: the reject/solve kernel that read it last reset it
  DevBuf<double> resid;          // K, valid where keep
  DevBuf<double> resid_compact;  // kept order
  DevBuf<unsigned int> unresolved;  // query ids the grid could not bound + counter at [K]
  DevBuf<unsigned char> bf_scratch;
  long long n_kept = 0;
  bool matched = false, rejected = false, solved = false;
  // record slot 0, dev_state and nn_idx / dist / keep are those of the last sicp_iterate or
  // sicp_time_stages iteration (what sicp_get_iteration reads back)
  bool stepped = false;
  bool expect_unresolved = true;  // last known: did some query exceed the ring limit?
  double min_planarity_last = 0.0;

  // last solve state (for uncertainties)
  double last_x[6] = {0, 0, 0, 0, 0, 0};
  double last_T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};  // transform applied to the movable cloud
  double last_sigma[6] = {0, 0, 0, 0, 0, 0};
  sicp_lsq_params last_lsq{};

  SolveWs ws;
  DevBuf<DevState> dev_state;
  int rs_parity = 0;
  DevBuf<unsigned int> compact_sums;
  DevBuf<unsigned long long> bbox_keys;   // grid build scratch (kept apart from the select workspace)
  DevBuf<unsigned int> misc_counters;     // grid build / API scratch counters
  DevBuf<unsigned char> flush_buf;        // 256 MiB scratch for cold-L2 measurements
  DevBuf<unsigned long long> phase_t;     // %globaltimer stamps of the reject/solve kernel
  DevBuf<unsigned int> grid_bar;          // grid barrier of the cooperative reject/solve kernel
  DevBuf<unsigned int> lin_hist;          // predictor histogram (match kernels -> reject kernel)
  bool lin_hist_pending = false;          // filled by a match, not yet consumed by a reject
  bool lin_hist_init = false;
  bool rsb_attr_set = false;
  bool rsf_attr_set = false;              // k_rs_fused's dynamic shared memory limit raised on this device
  DevBuf<unsigned int> rsf_ticket;        // blocks-finished counter of the barrier-free reject/solve kernel
  int n_fused_last = 0, n_rerun_last = 0; // last run: iterations through k_rs_fused / repeated after a missed prediction
  int fused = 1;                          // option "fused": 0 = always the cooperative kernel
  bool bf_attr_set = false;               // k_bf_nn's dynamic shared memory limit raised on this device
  sicp_iter_record* rec_host = nullptr;  // pinned
  double* scal_host = nullptr;           // pinned staging for small reads
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t copy_stream = nullptr;   // second stream: fixed-cloud upload overlaps the movable grid build
  PageableUploader up;                  // clouds in pageable host memory (NumPy arrays): threaded staging, upload.cuh
  int upload_threads = 2;               // option "upload_threads": 0 = plain cudaMemcpyAsync for every source (measured: 2, 3, 4 threads alike, tools/upload_probe.py)
  cudaEvent_t ev_copy = nullptr, ev_user = nullptr;
  sicp_timings tm{};

  // staging for host inputs
  DevBuf<unsigned char> stage;

  Batch* batch = nullptr;  // created by the first sicp_register_batch
};
// what the match kernels / reject kernels see of the movable-side attributes
inline const float4* mov_attr_nrm(Ctx& c) { return c.mov_attr ? c.mov_nrm.p : nullptr; }
inline float4* mov_attr_eff(Ctx& c) {
  if (!c.mov_attr) return nullptr;
  c.q_nrm_eff.reserve(c.K > 0 ? c.K : 1);
  return c.q_nrm_eff.p;
}

// ---- batched engine: many small pairs per launch (BASELINE configs[4], SURVEY.md section 8e) ----
// One descriptor per pair, resident in device memory; every batched kernel takes the pair from
// blockIdx.y (or blockIdx.x for the one-block-per-pair kernels) and reads its descriptor.
struct PairDev {
  GridView gmov, gfix;
  long long n_fix, n_mov;
  long long fix_off, mov_off;  // first point of this pair in the concatenated clouds
  long long K;                 // selected fixed points (<= Kmax)
  long long q_off;             // first entry of this pair in the per-query arrays
  double cm[3];                // centre of the movable grid's box (moment centring)
};

// One cloud of a batched grid build (filled by the host from the bounding boxes).
struct CloudPlan {
  const double* xyz;
  long long n;
  long long rec_base;   // position of its first record in the shared record array (= point offset)
  long long cell_base;  // first entry of its cell table in the shared table
  double ox, oy, oz, h, inv_h;
  int nx, ny, nz, pad;
};

// The grids of one side (all fixed or all movable clouds of a batch): one record array, one cell table.
struct BatchGrid {
  DevBuf<Rec> recs;
  DevBuf<uint32_t> cell_table, fill, cid, block_sums;
};

struct Batch {
  int n_pairs = 0;
  long long Kmax = 0, total_fix = 0, total_mov = 0;
  DevBuf<double> fix_xyz, mov_xyz;  // concatenated clouds
  BatchGrid gfix, gmov;
  DevBuf<unsigned int> occ;
  DevBuf<unsigned long long> bbox_keys;
  DevBuf<CloudPlan> plans;
  DevBuf<PairDev> pairs;
  // per-query arrays, n_pairs x Kmax
  DevBuf<long long> sel_idx, nn_idx;
  DevBuf<double> q_xyz, dist, m_xyz;
  DevBuf<float4> q_nrm;
  DevBuf<uint32_t> knn_pos;        // n_pairs x Kmax x k
  DevBuf<unsigned int> binstore;  // n_pairs x LH_BINS x bin_cap
  int bin_cap = 0;
  DevBuf<uint32_t> nn_pos;
  DevBuf<uint8_t> keep;
  // per-pair state
  DevBuf<DevState> state;
  DevBuf<unsigned int> lin_hist;       // n_pairs x (LH_BINS + 2)
  DevBuf<sicp_iter_record> rec;        // n_pairs x max_iterations
  DevBuf<double> partials;             // n_pairs x RSF_NPART (+ slack)
  DevBuf<unsigned int> ticket;         // n_pairs
  DevBuf<unsigned long long> phase_t;  // 32 (diagnostics of pair 0)
  DevBuf<int> flags;                   // n_pairs x 2: {stop, iterations_done}
  DevBuf<sicp_pair_result> results;
  int* flags_host = nullptr;                 // pinned
  sicp_pair_result* results_host = nullptr;  // pinned
  size_t flags_cap = 0, results_cap = 0;
  unsigned long long* keys_host = nullptr;   // pinned: bounding boxes / occupancies
  size_t keys_cap = 0;
  ~Batch() {
    if (flags_host) cudaFreeHost(flags_host);
    if (results_host) cudaFreeHost(results_host);
    if (keys_host) cudaFreeHost(keys_host);
  }
};

// ---- stage entry points (each implemented in its own translation unit) ---------------------
void grid_build(Ctx& c, Grid& g, const double* xyz_dev, long long n);
void make_float4_copy(Ctx& c);

// 1-NN of K transformed queries into the movable cloud; fused point-to-plane distance.
// If out_d2 != nullptr the squared NN distance is written instead of the plane distance epilogue
// being required (overlap filter).
// The transform is read from c.dev_state (T, Tinv) on the device.
// allow_bf: bound the ring expansion by grid_max_rings and answer the rest with the brute-force
// pass; otherwise the grid search runs to completion on its own (no extra launches).
// in_loop: called from launch_iteration — the counter of unresolved queries was reset by the
// previous iteration's reject/solve kernel (no memset between the kernels), and the kernel may be
// launched programmatically dependent on it (option "pdl").
void match_launch(Ctx& c, bool with_distance, double* out_d2, cudaEvent_t mid = nullptr,
                  bool allow_bf = true, double cap2 = -1.0, bool in_loop = false);

// kernel launch, optionally with the programmatic-stream-serialization attribute (common.cuh: pdl_wait)
template <typename... KArgs, typename... Args>
inline void launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                          bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  SICP_CUDA(cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...));
}
void set_state_transform(Ctx& c, const double x[6], const Rigid* T_or_null, bool reset_loop);
void estimate_normals_launch(Ctx& c, int k);
void reject_solve_launch(Ctx& c, const sicp_run_params& p, int it, bool do_solve, bool arm_stop,
                         int rec_slot);
void compact_residuals_launch(Ctx& c);
void rs_fused_launch(Ctx& c, const sicp_run_params& p, int it, bool arm_stop, int rec_slot, bool want_sigma);
void final_residuals_launch(Ctx& c);
void transform_launch(Ctx& c, const Rigid& T, const double* in_dev, double* out_dev, long long n);
void gather_queries_launch(Ctx& c);

// batched launches
struct BatchHostCloud {
  const double* xyz_dev;
  long long n;
  long long point_off;  // first record of this cloud in the shared record array
};
void grid_build_batch(Ctx& c, Batch& b, BatchGrid& bg, const std::vector<BatchHostCloud>& clouds,
                      std::vector<GridView>& views, std::vector<double>& centres /* 3 per cloud */);
void batch_select_gather_launch(Ctx& c, Batch& b, long long correspondences, int round_away);
void batch_normals_launch(Ctx& c, Batch& b, int k);
void batch_match_launch(Ctx& c, Batch& b, bool warm);
void batch_rs_launch(Ctx& c, Batch& b, const sicp_run_params& p, int it, bool want_sigma);
void batch_finish_launch(Ctx& c, Batch& b, int max_iterations);

int bin_cap_for(long long K);

// helpers in capi.cu
bool is_device_ptr(const void* p);

struct StageTimer {
  Ctx& c;
  double* slot;
  StageTimer(Ctx& c_, double* s) : c(c_), slot(s) { cudaEventRecord(c.ev0, c.stream); }
  void stop() {
    cudaEventRecord(c.ev1, c.stream);
    cudaEventSynchronize(c.ev1);
    float ms = 0;
    cudaEventElapsedTime(&ms, c.ev0, c.ev1);
    *slot = ms;
  }
};

}  // namespace sicp

struct sicp_ctx {
  sicp::Ctx c;
  int it_counter = 0;
};
