// capi.cu — the extern "C" boundary declared in include/sicp_b200.h.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "ctx.cuh"

namespace sicp {

static thread_local std::string g_thread_error;
void set_thread_error(const std::string& m) { g_thread_error = m; }

bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

namespace {

constexpr int kMaxRecords = 4096;

__global__ void k_iota(long long* p, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

// PointCloud.select_n_points (pointcloud.py:121-147): sel[i] = src[rint(linspace(0, m-1, n)[i])],
// numpy's linspace arithmetic (i * step, last element forced to m-1), rint = round-half-even.
// away = 1 gives the native drivers' C round() (c++/src/pointcloud.cpp:92-96).  src == NULL: iota.
__global__ void k_select_n(const long long* __restrict__ src, long long m, long long n, int away,
                           long long* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double step = (n > 1) ? (double)(m - 1) / (double)(n - 1) : 0.0;
  const double y = (i == n - 1 && n > 1) ? (double)(m - 1) : (double)i * step;
  const long long j = (long long)(away ? round(y) : rint(y));
  out[i] = src ? src[j] : j;
}

__global__ void k_check_sel(const long long* __restrict__ sel, long long K, long long n,
                            unsigned int* __restrict__ bad) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K) return;
  const long long v = sel[i];
  if (v < 0 || v >= n || (i > 0 && sel[i - 1] >= v)) atomicAdd(bad, 1u);
}

__global__ void k_range_keep(const double* __restrict__ d2, long long K, double r2,
                             uint8_t* __restrict__ keep, unsigned int* __restrict__ count) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  unsigned int k = 0;
  if (i < K) {
    k = (d2[i] < r2) ? 1u : 0u;  // strict: cKDTree distance_upper_bound semantics
    keep[i] = (uint8_t)k;
  }
  const unsigned int m = __ballot_sync(0xffffffffu, k);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, (unsigned int)__popc(m));
}

__global__ void k_split_f4(const float4* __restrict__ in, long long K, float* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K) return;
  const float4 v = in[i];
  out[i] = v.x;
  out[K + i] = v.y;
  out[2 * K + i] = v.z;
  out[3 * K + i] = v.w;
}

__global__ void k_join_f4(const float* __restrict__ in, long long K, float4* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= K) return;
  out[i] = make_float4(in[i], in[K + i], in[2 * K + i], in[3 * K + i]);
}

void copy_any(Ctx& c, void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return;
  SICP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, c.stream));
}

void sync(Ctx& c) { SICP_CUDA(cudaStreamSynchronize(c.stream)); }

// A whole cloud, host -> device.  Pageable sources (NumPy arrays) take the threaded staging path
// of upload.cuh; pinned / device sources are one cudaMemcpyAsync.
constexpr size_t kThreadedUploadMin = 4u << 20;
bool threaded_upload(Ctx& c, const void* src, size_t bytes) {
  return c.upload_threads > 0 && bytes >= kThreadedUploadMin && PageableUploader::is_pageable(src);
}
// ... on the context's stream, complete (stream-ordered) when the call returns
void upload_cloud(Ctx& c, void* dst, const void* src, size_t bytes) {
  if (!threaded_upload(c, src, bytes)) {
    copy_any(c, dst, src, bytes);
    return;
  }
  SICP_CUDA(cudaEventRecord(c.ev_user, c.stream));
  c.up.start(c.device, c.upload_threads, dst, src, bytes, c.ev_user);
  c.up.finish(c.stream);
}
// ... in the background (copy stream or worker threads) after everything queued on the context's
// stream so far; wait_background_upload() makes the context's stream wait for it
void start_background_upload(Ctx& c, void* dst, const void* src, size_t bytes) {
  SICP_CUDA(cudaEventRecord(c.ev_user, c.stream));
  if (threaded_upload(c, src, bytes)) {
    c.up.start(c.device, c.upload_threads, dst, src, bytes, c.ev_user);
    return;
  }
  SICP_CUDA(cudaStreamWaitEvent(c.copy_stream, c.ev_user, 0));
  SICP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, c.copy_stream));
  SICP_CUDA(cudaEventRecord(c.ev_copy, c.copy_stream));
}
void wait_background_upload(Ctx& c) {
  if (c.up.active()) c.up.finish(c.stream);
  else SICP_CUDA(cudaStreamWaitEvent(c.stream, c.ev_copy, 0));
}

void init_state(Ctx& c, const double x[6], const Rigid* T_or_null, bool reset_loop) {
  c.unresolved_clean = false;
  c.stepped = false;
  // small pageable H2D copies are staged by the runtime before the call returns
  DevState h;
  if (reset_loop) {
    std::memset(&h, 0, sizeof(h));
  } else {
    SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
    sync(c);
  }
  if (x)
    for (int j = 0; j < 6; ++j) h.x[j] = x[j];
  h.T = T_or_null ? *T_or_null : rigid_from_x(h.x);
  h.Tinv = rigid_inverse(h.T);
  h.T_res = h.T;
  h.H_rep = h.T;
  if (reset_loop) h.stop = 0;
  SICP_CUDA(cudaMemcpyAsync(c.dev_state.p, &h, sizeof(h), cudaMemcpyHostToDevice, c.stream));
  sync(c);
}

void require_clouds(Ctx& c) {
  SICP_REQUIRE(c.n_fix > 0 && c.n_mov > 0, SICP_ERR_STATE, "sicp_set_clouds has not been called");
}
void require_selected(Ctx& c) {
  require_clouds(c);
  SICP_REQUIRE(c.K > 0, SICP_ERR_STATE, "no fixed points are selected");
}
void require_normals(Ctx& c) {
  require_selected(c);
  SICP_REQUIRE(c.have_normals, SICP_ERR_STATE,
               "normals are missing: call sicp_estimate_normals or sicp_set_normals first");
}

// One iteration's launches: match, then the barrier-free reject/solve kernel when the previous
// iteration of this run left a predictor (it > 0), else the general cooperative kernel.
void launch_iteration(Ctx& c, const sicp_run_params& p, int it, bool arm_stop, int rec_slot,
                      bool allow_fused, bool want_sigma, cudaEvent_t mid = nullptr, cudaEvent_t after_match = nullptr) {
  match_launch(c, true, nullptr, mid, c.expect_unresolved, -1.0, true);
  if (after_match) SICP_CUDA(cudaEventRecord(after_match, c.stream));
  // K <= 4096: one block owns the whole problem and falls back to the radix selection by itself
  // when there is no prediction (first iteration) — the barrier-free kernel serves every iteration
  if (allow_fused && c.fused && (it > 0 || c.K <= 4096))
    rs_fused_launch(c, p, it, arm_stop, rec_slot, want_sigma);
  else
    reject_solve_launch(c, p, it, true, arm_stop, rec_slot);
  c.unresolved_clean = true;  // both kernels reset the counter after reading it
}

// The fused kernel found its prediction unusable and parked the pipeline (state.stop == 3):
// clear the flag so that the iteration can be repeated with the general kernel.
void clear_stop_flag(Ctx& c) {
  c.unresolved_clean = false;
  static const int zero = 0;
  SICP_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(c.dev_state.p) + offsetof(DevState, stop), &zero,
                            sizeof(int), cudaMemcpyHostToDevice, c.stream));
}

void fetch_records(Ctx& c, int first, int count) {
  SICP_CUDA(cudaMemcpyAsync(c.rec_host + first, c.ws.rec.p + first, sizeof(sicp_iter_record) * count,
                            cudaMemcpyDeviceToHost, c.stream));
}

}  // namespace

void set_state_transform(Ctx& c, const double x[6], const Rigid* T_or_null, bool reset_loop) {
  init_state(c, x, T_or_null, reset_loop);
}

}  // namespace sicp

using namespace sicp;

#define API_BEGIN(ctxptr)                                    \
  if (!(ctxptr)) {                                           \
    sicp::set_thread_error("sicp_ctx is NULL");              \
    return SICP_ERR_BAD_ARG;                                 \
  }                                                          \
  Ctx& c = (ctxptr)->c;                                      \
  try {                                                      \
    SICP_CUDA(cudaSetDevice(c.device));

#define API_END                                              \
  }                                                          \
  catch (const sicp::Error& e) {                             \
    c.up.abandon();                                          \
    c.err = e.msg;                                           \
    sicp::set_thread_error(e.msg);                           \
    if (e.code == SICP_ERR_CUDA) cudaGetLastError();         \
    return e.code;                                           \
  }                                                          \
  catch (const std::exception& e) {                          \
    c.up.abandon();                                          \
    c.err = e.what();                                        \
    sicp::set_thread_error(c.err);                           \
    return SICP_ERR_CUDA;                                    \
  }                                                          \
  return SICP_OK;

extern "C" {

int32_t sicp_abi_version(void) { return SICP_ABI_VERSION; }

const char* sicp_last_error(sicp_ctx* ctx) {
  if (ctx) return ctx->c.err.c_str();
  return sicp::g_thread_error.c_str();
}

int32_t sicp_create(int32_t device, void* cuda_stream, sicp_ctx** out) {
  if (!out) {
    sicp::set_thread_error("out is NULL");
    return SICP_ERR_BAD_ARG;
  }
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    sicp::set_thread_error(std::string("no CUDA device available: ") + cudaGetErrorString(e));
    return SICP_ERR_CUDA;
  }
  if (device < 0 || device >= n_dev) {
    sicp::set_thread_error("device index out of range");
    return SICP_ERR_BAD_ARG;
  }
  sicp_ctx* h = new (std::nothrow) sicp_ctx();
  if (!h) return SICP_ERR_CUDA;
  Ctx& c = h->c;
  try {
    c.device = device;
    SICP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    SICP_CUDA(cudaGetDeviceProperties(&prop, device));
    SICP_REQUIRE(prop.major >= 10, SICP_ERR_CUDA,
                 std::string("libsicp_b200 is built for sm_100a only; device is sm_") +
                     std::to_string(prop.major) + std::to_string(prop.minor));
    c.num_sms = prop.multiProcessorCount;
    c.stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    SICP_CUDA(cudaEventCreate(&c.ev0));
    SICP_CUDA(cudaEventCreate(&c.ev1));
    SICP_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    SICP_CUDA(cudaEventCreateWithFlags(&c.ev_copy, cudaEventDisableTiming));
    SICP_CUDA(cudaEventCreateWithFlags(&c.ev_user, cudaEventDisableTiming));
    SICP_CUDA(cudaMallocHost(&c.rec_host, sizeof(sicp_iter_record) * kMaxRecords));
    SICP_CUDA(cudaMallocHost(&c.scal_host, sizeof(double) * 256));
    c.ws.rec.reserve(kMaxRecords);
    c.ws.scal.reserve(256);
    c.ws.counters.reserve(64);
    c.ws.minkey.reserve(16);
    c.dev_state.reserve(1);
    SICP_CUDA(cudaMemsetAsync(c.dev_state.p, 0, sizeof(DevState), c.stream));
    SICP_CUDA(cudaStreamSynchronize(c.stream));
  } catch (const sicp::Error& er) {
    sicp::set_thread_error(er.msg);
    delete h;
    return er.code;
  }
  *out = h;
  return SICP_OK;
}

int32_t sicp_destroy(sicp_ctx* ctx) {
  if (!ctx) return SICP_OK;
  Ctx& c = ctx->c;
  cudaSetDevice(c.device);
  cudaStreamSynchronize(c.stream);
  if (c.ev0) cudaEventDestroy(c.ev0);
  if (c.ev1) cudaEventDestroy(c.ev1);
  if (c.ev_copy) cudaEventDestroy(c.ev_copy);
  if (c.ev_user) cudaEventDestroy(c.ev_user);
  if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
  delete c.batch;
  c.batch = nullptr;
  if (c.rec_host) cudaFreeHost(c.rec_host);
  if (c.scal_host) cudaFreeHost(c.scal_host);
  delete ctx;
  return SICP_OK;
}

int32_t sicp_set_option(sicp_ctx* ctx, const char* key, double value) {
  API_BEGIN(ctx)
  SICP_REQUIRE(key != nullptr, SICP_ERR_BAD_ARG, "key is NULL");
  const std::string k(key);
  if (k == "defaults") {
    const Ctx d;  // the member initialisers are the defaults
    c.nn_engine = d.nn_engine;
    c.sign_mode = d.sign_mode;
    c.variant = d.variant;
    c.grid_target_occ = d.grid_target_occ;
    c.grid_max_rings = d.grid_max_rings;
    c.grid_sort_cells = d.grid_sort_cells;
    c.rs_blocks = d.rs_blocks;
    c.match_group = d.match_group;
    c.host_sync_every = d.host_sync_every;
    c.upload_threads = d.upload_threads;
    c.up.chunk = d.up.chunk;
    c.fused = d.fused;
    c.warm_start = d.warm_start;
    c.sphere_scan = d.sphere_scan;
    c.pdl = d.pdl;
    c.keep_knn = d.keep_knn;
    c.knn_coop = d.knn_coop;
  } else if (k == "nn_engine") {
    SICP_REQUIRE(value == 0 || value == 1 || value == 2, SICP_ERR_BAD_ARG, "nn_engine must be 0, 1 or 2");
    c.nn_engine = (int)value;
  } else if (k == "sign_mode") {
    SICP_REQUIRE(value == 0 || value == 1, SICP_ERR_BAD_ARG, "sign_mode must be 0 or 1");
    c.sign_mode = (int)value;
  } else if (k == "variant") {
    SICP_REQUIRE(value == 0 || value == 1 || value == 2, SICP_ERR_BAD_ARG, "variant must be 0, 1 or 2");
    c.variant = (int)value;
  } else if (k == "grid_target_occupancy") {
    SICP_REQUIRE(value >= 0.25 && value <= 64, SICP_ERR_BAD_ARG, "grid_target_occupancy out of range");
    c.grid_target_occ = value;
  } else if (k == "grid_max_rings") {
    SICP_REQUIRE(value >= 1 && value <= 1e6, SICP_ERR_BAD_ARG, "grid_max_rings out of range");
    c.grid_max_rings = (int)value;
  } else if (k == "grid_sort_cells") {
    c.grid_sort_cells = (value != 0) ? 1 : 0;
  } else if (k == "keep_knn") {
    c.keep_knn = (value != 0) ? 1 : 0;
  } else if (k == "knn_coop") {
    c.knn_coop = (value < 0) ? -1 : ((value >= 2) ? 2 : ((value != 0) ? 1 : 0));
  } else if (k == "pdl") {
    c.pdl = (value != 0) ? 1 : 0;
  } else if (k == "sphere_scan") {
    c.sphere_scan = (value != 0) ? 1 : 0;
  } else if (k == "warm_start") {
    c.warm_start = (value != 0) ? 1 : 0;
  } else if (k == "fused") {
    c.fused = (value != 0) ? 1 : 0;
  } else if (k == "rs_blocks") {
    SICP_REQUIRE(value >= 0 && value <= 256, SICP_ERR_BAD_ARG, "rs_blocks out of range");
    c.rs_blocks = (int)value;
  } else if (k == "match_group") {
    SICP_REQUIRE(value == 0 || value == 1 || value == 2 || value == 4 || value == 8 || value == 16, SICP_ERR_BAD_ARG,
                 "match_group must be 0 (auto), 1, 2, 4, 8 or 16");
    c.match_group = (int)value;
  } else if (k == "upload_threads") {
    SICP_REQUIRE(value >= 0 && value <= PageableUploader::kMaxThreads, SICP_ERR_BAD_ARG,
                 "upload_threads must be within [0, 8]");
    c.upload_threads = (int)value;
  } else if (k == "upload_chunk_kb") {
    SICP_REQUIRE(value >= 64 && value <= 4096, SICP_ERR_BAD_ARG, "upload_chunk_kb must be within [64, 4096]");
    c.up.chunk = (size_t)value << 10;
  } else if (k == "host_sync_every") {
    SICP_REQUIRE(value >= 1 && value <= 1024, SICP_ERR_BAD_ARG, "host_sync_every out of range");
    c.host_sync_every = (int)value;
  } else {
    SICP_REQUIRE(false, SICP_ERR_BAD_ARG, "unknown option: " + k);
  }
  API_END
}

int32_t sicp_set_selected(sicp_ctx* ctx, const int64_t* idx, int64_t K) {
  API_BEGIN(ctx)
  require_clouds(c);
  SICP_REQUIRE(K > 0 && K <= c.n_fix, SICP_ERR_BAD_ARG, "K must be in [1, n_fix]");
  c.sel_idx.reserve(K);
  if (idx == nullptr) {
    SICP_REQUIRE(K == c.n_fix, SICP_ERR_BAD_ARG, "idx == NULL selects all points: K must equal n_fix");
    k_iota<<<(unsigned)((K + 255) / 256), 256, 0, c.stream>>>(c.sel_idx.p, K);
  } else {
    copy_any(c, c.sel_idx.p, idx, sizeof(long long) * K);
    SICP_CUDA(cudaMemsetAsync(c.misc_counters.p + 8, 0, sizeof(unsigned int), c.stream));
    k_check_sel<<<(unsigned)((K + 255) / 256), 256, 0, c.stream>>>(c.sel_idx.p, K, c.n_fix,
                                                                  c.misc_counters.p + 8);
    unsigned int bad = 0;
    SICP_CUDA(cudaMemcpyAsync(&bad, c.misc_counters.p + 8, sizeof(bad), cudaMemcpyDeviceToHost, c.stream));
    sync(c);
    SICP_REQUIRE(bad == 0, SICP_ERR_BAD_ARG,
                 "selected indices must be strictly ascending and inside [0, n_fix)");
  }
  c.K = K;
  gather_queries_launch(c);
  c.have_normals = false;
  c.nn_pos_valid = false;
  c.matched = c.rejected = c.solved = c.stepped = false;
  sync(c);
  API_END
}

int32_t sicp_set_clouds(sicp_ctx* ctx, const double* fix_xyz, int64_t n_fix, const double* mov_xyz,
                        int64_t n_mov) {
  API_BEGIN(ctx)
  SICP_REQUIRE(fix_xyz && mov_xyz, SICP_ERR_BAD_ARG, "cloud pointer is NULL");
  SICP_REQUIRE(n_fix > 0 && n_mov > 0, SICP_ERR_BAD_ARG, "clouds must not be empty");
  SICP_REQUIRE(n_fix < (1ll << 31) && n_mov < (1ll << 31), SICP_ERR_BAD_ARG,
               "clouds are limited to 2^31 - 1 points");
  {
    // movable cloud on the context's stream; the fixed cloud follows on a second stream (after
    // everything already queued on the caller's stream) so that its transfer overlaps the grid
    // build of the movable cloud
    StageTimer t(c, &c.tm.upload_ms);
    c.fix_xyz.reserve(3 * n_fix);
    c.mov_xyz.reserve(3 * n_mov);
    upload_cloud(c, c.mov_xyz.p, mov_xyz, sizeof(double) * 3 * n_mov);
    t.stop();
  }
  start_background_upload(c, c.fix_xyz.p, fix_xyz, sizeof(double) * 3 * n_fix);
  c.n_fix = n_fix;
  c.n_mov = n_mov;
  c.gfix.built = false;
  {
    StageTimer t(c, &c.tm.grid_mov_ms);
    grid_build(c, c.gmov, c.mov_xyz.p, n_mov);
    make_float4_copy(c);
    t.stop();
  }
  wait_background_upload(c);
  SICP_CUDA(cudaStreamSynchronize(c.copy_stream));  // the caller may reuse fix_xyz after return
  c.K = 0;
  c.have_normals = false;
  c.mov_attr = false;
  c.nn_pos_valid = false;
  c.matched = c.rejected = c.solved = c.stepped = false;
  API_END
}

int32_t sicp_select_in_range(sicp_ctx* ctx, const double H0[16], double max_range, uint8_t* keep,
                             int64_t* n_kept) {
  API_BEGIN(ctx)
  require_selected(c);
  SICP_REQUIRE(H0 && n_kept, SICP_ERR_BAD_ARG, "NULL argument");
  SICP_REQUIRE(max_range > 0, SICP_ERR_BAD_ARG, "max_range must be > 0");
  const Rigid T = rigid_from_H(H0);
  init_state(c, nullptr, &T, true);
  StageTimer t(c, &c.tm.overlap_ms);
  c.dist.reserve(c.K);
  c.keep.reserve(c.K);
  // the overlap filter needs no normals: the epilogue is skipped (with_distance = false)
  // only the side of max_range matters: bounded search (nn.cu: grid_nn, cap2)
  match_launch(c, false, c.dist.p, nullptr, true, max_range * max_range);
  SICP_CUDA(cudaMemsetAsync(c.misc_counters.p + 8, 0, sizeof(unsigned int), c.stream));
  k_range_keep<<<(unsigned)((c.K + 255) / 256), 256, 0, c.stream>>>(
      c.dist.p, c.K, max_range * max_range, c.keep.p, c.misc_counters.p + 8);
  unsigned int cnt = 0;
  SICP_CUDA(cudaMemcpyAsync(&cnt, c.misc_counters.p + 8, sizeof(cnt), cudaMemcpyDeviceToHost, c.stream));
  if (keep) copy_any(c, keep, c.keep.p, (size_t)c.K);
  t.stop();
  *n_kept = cnt;
  SICP_REQUIRE(cnt > 0, SICP_ERR_NO_OVERLAP,
               "Point clouds do not overlap within max_overlap_distance");
  API_END
}

int32_t sicp_estimate_normals(sicp_ctx* ctx, int32_t neighbors, float* nx, float* ny, float* nz,
                              float* planarity) {
  API_BEGIN(ctx)
  require_selected(c);
  if (!c.gfix.built) {
    StageTimer t(c, &c.tm.grid_fix_ms);
    grid_build(c, c.gfix, c.fix_xyz.p, c.n_fix);
    t.stop();
  }
  StageTimer t(c, &c.tm.normals_ms);
  estimate_normals_launch(c, neighbors);
  c.have_normals = true;
  if (nx || ny || nz || planarity) {
    c.stage.reserve(sizeof(float) * 4 * c.K);
    float* s = reinterpret_cast<float*>(c.stage.p);
    k_split_f4<<<(unsigned)((c.K + 255) / 256), 256, 0, c.stream>>>(c.q_nrm.p, c.K, s);
    if (nx) copy_any(c, nx, s, sizeof(float) * c.K);
    if (ny) copy_any(c, ny, s + c.K, sizeof(float) * c.K);
    if (nz) copy_any(c, nz, s + 2 * c.K, sizeof(float) * c.K);
    if (planarity) copy_any(c, planarity, s + 3 * c.K, sizeof(float) * c.K);
  }
  t.stop();
  API_END
}

int32_t sicp_set_normals(sicp_ctx* ctx, const float* nx, const float* ny, const float* nz,
                         const float* planarity) {
  API_BEGIN(ctx)
  require_selected(c);
  SICP_REQUIRE(nx && ny && nz && planarity, SICP_ERR_BAD_ARG, "NULL normal array");
  c.stage.reserve(sizeof(float) * 4 * c.K);
  float* s = reinterpret_cast<float*>(c.stage.p);
  copy_any(c, s, nx, sizeof(float) * c.K);
  copy_any(c, s + c.K, ny, sizeof(float) * c.K);
  copy_any(c, s + 2 * c.K, nz, sizeof(float) * c.K);
  copy_any(c, s + 3 * c.K, planarity, sizeof(float) * c.K);
  c.q_nrm.reserve(c.K);
  k_join_f4<<<(unsigned)((c.K + 255) / 256), 256, 0, c.stream>>>(s, c.K, c.q_nrm.p);
  c.have_normals = true;
  sync(c);
  API_END
}

int32_t sicp_set_mov_normals(sicp_ctx* ctx, const float* nx, const float* ny, const float* nz,
                             const float* planarity, double max_angle_rad) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.n_mov > 0, SICP_ERR_STATE, "no clouds: call sicp_set_clouds first");
  if (!nx && !ny && !nz && !planarity) {  // back to the default run
    c.mov_attr = false;
    c.mov_cos_max = -1.0;
    c.matched = c.rejected = c.solved = c.stepped = false;
    return SICP_OK;
  }
  SICP_REQUIRE(nx && ny && nz && planarity, SICP_ERR_BAD_ARG, "NULL normal array");
  SICP_REQUIRE(!(max_angle_rad > 1.5707963267948966), SICP_ERR_BAD_ARG,
               "max_angle_rad must be <= pi/2 (normals are axes), or negative for no angle test");
  c.stage.reserve(sizeof(float) * 4 * c.n_mov);
  float* s = reinterpret_cast<float*>(c.stage.p);
  copy_any(c, s, nx, sizeof(float) * c.n_mov);
  copy_any(c, s + c.n_mov, ny, sizeof(float) * c.n_mov);
  copy_any(c, s + 2 * c.n_mov, nz, sizeof(float) * c.n_mov);
  copy_any(c, s + 3 * c.n_mov, planarity, sizeof(float) * c.n_mov);
  c.mov_nrm.reserve(c.n_mov);
  k_join_f4<<<(unsigned)((c.n_mov + 255) / 256), 256, 0, c.stream>>>(s, c.n_mov, c.mov_nrm.p);
  SICP_CUDA(cudaGetLastError());
  c.mov_attr = true;
  c.mov_cos_max = (max_angle_rad >= 0.0) ? (max_angle_rad >= 1.5707963267948966 ? 0.0 : cos(max_angle_rad)) : -1.0;
  c.matched = c.rejected = c.solved = c.stepped = false;
  sync(c);
  API_END
}

int32_t sicp_get_knn(sicp_ctx* ctx, int64_t* idx, double* dist2) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.knn_k > 0 && c.have_normals, SICP_ERR_STATE,
               "no neighbour lists: set option keep_knn = 1 before sicp_estimate_normals");
  if (idx) copy_any(c, idx, c.knn_idx.p, sizeof(long long) * c.K * c.knn_k);
  if (dist2) copy_any(c, dist2, c.knn_d2.p, sizeof(double) * c.K * c.knn_k);
  sync(c);
  API_END
}

int32_t sicp_match(sicp_ctx* ctx, const double H[16], int64_t* pc2_idx, double* dist) {
  API_BEGIN(ctx)
  require_normals(c);
  SICP_REQUIRE(H != nullptr, SICP_ERR_BAD_ARG, "H is NULL");
  const Rigid T = rigid_from_H(H);
  init_state(c, nullptr, &T, true);
  StageTimer t(c, &c.tm.match_ms);
  match_launch(c, true, nullptr);
  if (pc2_idx) copy_any(c, pc2_idx, c.nn_idx.p, sizeof(long long) * c.K);
  if (dist) copy_any(c, dist, c.dist.p, sizeof(double) * c.K);
  t.stop();
  c.matched = true;
  c.rejected = c.solved = false;
  API_END
}

int32_t sicp_reject(sicp_ctx* ctx, double min_planarity, uint8_t* keep, int64_t* n_kept,
                    double stats[4]) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.matched, SICP_ERR_STATE, "sicp_match has not been called");
  SICP_REQUIRE(n_kept != nullptr, SICP_ERR_BAD_ARG, "n_kept is NULL");
  sicp_run_params p;
  std::memset(&p, 0, sizeof(p));
  p.min_planarity = min_planarity;
  p.lsq.distance_weight = 1.0;
  reject_solve_launch(c, p, 0, false, false, 0);
  fetch_records(c, 0, 1);
  if (keep) copy_any(c, keep, c.keep.p, (size_t)c.K);
  sync(c);
  const sicp_iter_record& r = c.rec_host[0];
  *n_kept = r.n_kept;
  c.n_kept = r.n_kept;
  if (stats) {
    stats[0] = r.median;
    stats[1] = r.mad;
    stats[2] = r.mean_dist;
    stats[3] = r.std_dist;
  }
  c.min_planarity_last = min_planarity;
  c.rejected = true;
  c.stepped = false;
  API_END
}

int32_t sicp_solve(sicp_ctx* ctx, const sicp_lsq_params* lp, double x[6], double H[16],
                   double* residuals, double stats[2], double* distance_weight_used) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.rejected, SICP_ERR_STATE, "sicp_reject has not been called");
  SICP_REQUIRE(lp && x && H, SICP_ERR_BAD_ARG, "NULL argument");
  sicp_run_params p;
  std::memset(&p, 0, sizeof(p));
  p.min_planarity = c.min_planarity_last;
  p.min_change = 0.0;
  p.lsq = *lp;
  // keep the matching transform (it only fixes the centring), start the solve from x0
  DevState h;
  SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
  sync(c);
  for (int j = 0; j < 6; ++j) h.x[j] = lp->x0[j];
  h.stop = 0;
  h.w = 0.0;
  SICP_CUDA(cudaMemcpyAsync(c.dev_state.p, &h, sizeof(h), cudaMemcpyHostToDevice, c.stream));
  StageTimer t(c, &c.tm.reject_solve_ms);
  reject_solve_launch(c, p, 0, true, false, 0);
  t.stop();
  fetch_records(c, 0, 1);
  SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
  sync(c);
  const sicp_iter_record& r = c.rec_host[0];
  c.n_kept = r.n_kept;
  SICP_REQUIRE(r.n_kept >= 6, SICP_ERR_TOO_FEW_CORR,
               "Too few correspondences! At least 6 correspondences are needed to estimate the 6 "
               "rigid body transformation parameters. The current number of correspondences is " +
                   std::to_string(r.n_kept) + ".");
  SICP_REQUIRE(h.lm_ok, SICP_ERR_SINGULAR, "normal equations are singular");
  for (int j = 0; j < 6; ++j) {
    x[j] = r.x[j];
    c.last_x[j] = r.x[j];
    c.last_sigma[j] = h.sigma[j];
  }
  H_from_rigid(h.T, H);
  H_from_rigid(h.T, c.last_T);
  if (stats) {
    stats[0] = r.mean_res;
    stats[1] = r.std_res;
  }
  if (distance_weight_used) *distance_weight_used = r.distance_weight;
  if (residuals) {
    compact_residuals_launch(c);
    copy_any(c, residuals, c.resid_compact.p, sizeof(double) * r.n_kept);
    sync(c);
  }
  c.solved = true;
  c.stepped = false;
  API_END
}

int32_t sicp_uncertainties(sicp_ctx* ctx, double sigma[6]) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.solved, SICP_ERR_STATE, "no solve has been run");
  SICP_REQUIRE(sigma != nullptr, SICP_ERR_BAD_ARG, "sigma is NULL");
  for (int j = 0; j < 6; ++j) sigma[j] = c.last_sigma[j];
  API_END
}

int32_t sicp_iterate(sicp_ctx* ctx, const sicp_run_params* p, const double x_in[6],
                     sicp_iter_record* rec) {
  API_BEGIN(ctx)
  require_normals(c);
  SICP_REQUIRE(p != nullptr, SICP_ERR_BAD_ARG, "params is NULL");
  if (x_in) {
    init_state(c, x_in, nullptr, true);
    ctx->it_counter = 0;
  }
  if (x_in) c.expect_unresolved = true;
  launch_iteration(c, *p, ctx->it_counter, false, 0, true, false);
  c.matched = c.rejected = c.stepped = true;
  if (rec) {
    DevState h;
    fetch_records(c, 0, 1);
    SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
    sync(c);
    if (h.stop == 3) {  // prediction unusable: the same iteration through the general kernel
      clear_stop_flag(c);
      launch_iteration(c, *p, ctx->it_counter, false, 0, false, false);
      fetch_records(c, 0, 1);
      sync(c);
    }
    *rec = c.rec_host[0];
    c.expect_unresolved = rec->n_bruteforce > 0;
  }
  ctx->it_counter++;
  API_END
}

// The iteration loop of SimpleICP.run (simpleicp.py:184-281); shared by sicp_run and sicp_register.
static void run_loop(sicp_ctx* ctx, Ctx& c, const sicp_run_params* p, sicp_run_result* out,
                     sicp_iter_record* log) {
  (void)ctx;
  require_normals(c);
  SICP_REQUIRE(p && out, SICP_ERR_BAD_ARG, "NULL argument");
  SICP_REQUIRE(p->max_iterations >= 1 && p->max_iterations <= kMaxRecords, SICP_ERR_BAD_ARG,
               "max_iterations must be in [1, 4096]");
  bool any_finite = false;
  for (int j = 0; j < 6; ++j) {
    SICP_REQUIRE(p->lsq.obs_weight[j] >= 0, SICP_ERR_BAD_ARG,
                 "All elements of rbp_observation_weights must be >= 0.");
    any_finite = any_finite || std::isfinite(p->lsq.obs_weight[j]);
  }
  SICP_REQUIRE(any_finite, SICP_ERR_BAD_ARG,
               "At least one element in rbp_observation_weights must be finite.");
  if (c.variant != SICP_VARIANT_PYTHON)
    for (int j = 0; j < 6; ++j)
      SICP_REQUIRE(p->lsq.obs_weight[j] == 0.0, SICP_ERR_BAD_ARG,
                   "the linearised variants have no observed or fixed parameters: "
                   "rbp_observation_weights must be all zero");
  static const bool trace = std::getenv("SICP_TRACE_RUN") != nullptr;
  const auto tr0 = std::chrono::steady_clock::now();
  auto tr = [&](const char* what, int it) {
    if (trace)
      fprintf(stderr, "[sicp_run] %-12s it=%d t=%.1f us\n", what, it,
              std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tr0).count());
  };
  init_state(c, p->lsq.x0, nullptr, true);
  std::memset(out, 0, sizeof(*out));
  // iterations queued past the stop flag return without writing their record: keep the slots defined
  SICP_CUDA(cudaMemsetAsync(c.ws.rec.p, 0, sizeof(sicp_iter_record) * (size_t)p->max_iterations, c.stream));
  tr("init", -1);

  cudaEvent_t e0, e1;
  SICP_CUDA(cudaEventCreate(&e0));
  SICP_CUDA(cudaEventCreate(&e1));
  SICP_CUDA(cudaEventRecord(e0, c.stream));
  int done = 0, fetched = 0, converged = 0, n_rerun = 0;
  std::vector<char> path((size_t)p->max_iterations, 0);  // 1: iteration served by the barrier-free kernel
  DevState h;
  // host reads: after the second iteration (it tells whether the brute-force pass is still
  // needed, and whether the first barrier-free iteration could use its prediction), then every
  // host_sync_every iterations; the device-side stop flag turns iterations queued past
  // convergence into immediate returns.  A read drains the pipeline (~25 us of idle GPU), an
  // iteration queued in vain costs ~8 us.
  const int every = std::max(1, c.host_sync_every);
  int next_sync = std::min(1, every - 1);
  int general_at = -1;  // iteration to repeat with the general kernel (fused prediction missed)
  c.expect_unresolved = true;
  for (int it = 0; it < p->max_iterations; ++it) {
    const bool fused = c.fused && (it > 0 || c.K <= 4096) && it != general_at;
    launch_iteration(c, *p, it, true, it, fused, it + 1 == p->max_iterations);
    path[(size_t)it] = fused ? 1 : 0;
    tr(fused ? "it (fused)" : "it (general)", it);
    if (it >= next_sync || it + 1 == p->max_iterations) {
      next_sync = it + every;
      fetch_records(c, fetched, it + 1 - fetched);
      SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
      sync(c);
      tr("synced", it);
      done = h.iterations_done;
      if (h.stop == 3) {
        // the barrier-free kernel of iteration `done` could not use its prediction; everything
        // queued behind it returned immediately.  Repeat from there with the general kernel.
        clear_stop_flag(c);
        SICP_CUDA(cudaMemsetAsync(c.ws.rec.p + done, 0, sizeof(sicp_iter_record) * (size_t)(it + 1 - done), c.stream));
        general_at = done;
        fetched = std::min(fetched, done);
        it = done - 1;
        next_sync = done;
        ++n_rerun;
        continue;
      }
      fetched = it + 1;
      c.expect_unresolved = c.rec_host[it].n_bruteforce > 0;
      if (h.stop == 2 || (done < it + 1 && !h.stop)) {
        // an iteration ended with fewer than 6 correspondences
        const long long nk = c.rec_host[std::min(done, it)].n_kept;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        SICP_REQUIRE(false, SICP_ERR_TOO_FEW_CORR,
                     "Too few correspondences! At least 6 correspondences are needed to estimate "
                     "the 6 rigid body transformation parameters. The current number of "
                     "correspondences is " + std::to_string(nk) + ".");
      }
      if (h.stop == 1) {
        converged = 1;
        break;
      }
    }
  }
  SICP_CUDA(cudaEventRecord(e1, c.stream));
  // residual vector of the final iteration (reference operation order), its ordered compaction
  // and exact two-pass statistics (they replace the moment-based values of the last record)
  final_residuals_launch(c);
  SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
  if (h.iterations_done > 0 || done > 0) fetch_records(c, std::max(done - 1, 0), 1);
  sync(c);
  c.n_fused_last = 0;
  for (int i = 0; i < h.iterations_done && i < p->max_iterations; ++i) c.n_fused_last += path[(size_t)i];
  c.n_rerun_last = n_rerun;
  tr("final", -1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  done = h.iterations_done;
  SICP_REQUIRE(h.lm_ok, SICP_ERR_SINGULAR, "normal equations are singular");
  out->iterations = done;
  out->converged = converged;
  for (int j = 0; j < 6; ++j) {
    // linearised variants: x holds the increments of the last iteration, H the reported matrix
    out->x[j] = c.variant ? h.x_new[j] : h.x[j];
    out->sigma[j] = h.sigma[j];
    c.last_x[j] = out->x[j];
    c.last_sigma[j] = h.sigma[j];
  }
  H_from_rigid(c.variant ? h.H_rep : h.T, out->H);
  H_from_rigid(h.T, c.last_T);
  out->n_residuals = h.n_kept;
  out->loop_ms = ms;
  c.n_kept = h.n_kept;
  c.tm.match_ms = 0;
  c.tm.reject_solve_ms = ms;
  if (log) std::memcpy(log, c.rec_host, sizeof(sicp_iter_record) * done);
  c.matched = c.rejected = c.solved = true;
  c.stepped = false;
}

int32_t sicp_run(sicp_ctx* ctx, const sicp_run_params* p, sicp_run_result* out,
                 sicp_iter_record* log) {
  API_BEGIN(ctx)
  run_loop(ctx, c, p, out, log);
  API_END
}

int32_t sicp_get_transform(sicp_ctx* ctx, double T[16]) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.solved, SICP_ERR_STATE, "no solve has been run");
  SICP_REQUIRE(T != nullptr, SICP_ERR_BAD_ARG, "T is NULL");
  for (int j = 0; j < 16; ++j) T[j] = c.last_T[j];
  API_END
}

int32_t sicp_get_residuals(sicp_ctx* ctx, double* residuals, int64_t cap, int64_t* n) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.solved, SICP_ERR_STATE, "no solve has been run");
  SICP_REQUIRE(n != nullptr, SICP_ERR_BAD_ARG, "n is NULL");
  *n = c.n_kept;
  if (residuals) {
    SICP_REQUIRE(cap >= c.n_kept, SICP_ERR_BAD_ARG, "residual buffer too small");
    copy_any(c, residuals, c.resid_compact.p, sizeof(double) * c.n_kept);
    sync(c);
  }
  API_END
}

static void transform_to(Ctx& c, const Rigid& T, double* mov_xyz_out) {
  StageTimer t(c, &c.tm.transform_ms);
  if (is_device_ptr(mov_xyz_out)) {
    transform_launch(c, T, c.mov_xyz.p, mov_xyz_out, c.n_mov);
  } else {
    c.stage.reserve(sizeof(double) * 3 * c.n_mov);
    double* s = reinterpret_cast<double*>(c.stage.p);
    transform_launch(c, T, c.mov_xyz.p, s, c.n_mov);
    copy_any(c, mov_xyz_out, s, sizeof(double) * 3 * c.n_mov);
  }
  t.stop();
}

int32_t sicp_transform(sicp_ctx* ctx, const double H[16], double* mov_xyz_out) {
  API_BEGIN(ctx)
  require_clouds(c);
  SICP_REQUIRE(H && mov_xyz_out, SICP_ERR_BAD_ARG, "NULL argument");
  transform_to(c, rigid_from_H(H), mov_xyz_out);
  API_END
}

int32_t sicp_select_n_points(sicp_ctx* ctx, int64_t n, int64_t* idx_out) {
  API_BEGIN(ctx)
  require_selected(c);
  SICP_REQUIRE(n >= 1, SICP_ERR_BAD_ARG, "n must be >= 1");
  if (n < c.K) {
    // pointcloud.py:137-147: only when fewer points are asked for than are selected
    c.sel_tmp.reserve(n);
    k_select_n<<<(unsigned)((n + 255) / 256), 256, 0, c.stream>>>(c.sel_idx.p, c.K, n, c.variant != SICP_VARIANT_PYTHON,
                                                                  c.sel_tmp.p);
    c.sel_idx.reserve(n);
    SICP_CUDA(cudaMemcpyAsync(c.sel_idx.p, c.sel_tmp.p, sizeof(long long) * n, cudaMemcpyDeviceToDevice, c.stream));
    c.K = n;
    gather_queries_launch(c);
    c.have_normals = false;
    c.nn_pos_valid = false;
    c.matched = c.rejected = c.solved = c.stepped = false;
  }
  if (idx_out) copy_any(c, idx_out, c.sel_idx.p, sizeof(long long) * c.K);
  sync(c);
  API_END
}

int32_t sicp_register(sicp_ctx* ctx, const double* fix_xyz, int64_t n_fix, const double* mov_xyz,
                      int64_t n_mov, const sicp_register_params* rp, sicp_run_result* out,
                      sicp_iter_record* log, double* mov_xyz_out, int64_t* n_selected) {
  API_BEGIN(ctx)
  SICP_REQUIRE(fix_xyz && mov_xyz && rp && out, SICP_ERR_BAD_ARG, "NULL argument");
  SICP_REQUIRE(n_fix > 0 && n_mov > 0, SICP_ERR_BAD_ARG, "clouds must not be empty");
  SICP_REQUIRE(n_fix < (1ll << 31) && n_mov < (1ll << 31), SICP_ERR_BAD_ARG,
               "clouds are limited to 2^31 - 1 points");
  SICP_REQUIRE(rp->correspondences >= 1, SICP_ERR_BAD_ARG, "correspondences must be >= 1");
  const bool overlap = rp->max_overlap_distance > 0 && std::isfinite(rp->max_overlap_distance);
  static const bool trace = std::getenv("SICP_TRACE_RUN") != nullptr;
  const auto tr0 = std::chrono::steady_clock::now();
  auto tr = [&](const char* what) {
    if (trace)
      fprintf(stderr, "[sicp_register] %-14s t=%.1f us\n", what,
              std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tr0).count());
  };
  c.fix_xyz.reserve(3 * n_fix);
  c.mov_xyz.reserve(3 * n_mov);
  c.n_fix = n_fix;
  c.n_mov = n_mov;
  c.gfix.built = false;
  c.K = 0;
  c.have_normals = false;
  c.mov_attr = false;
  c.nn_pos_valid = false;
  c.matched = c.rejected = c.solved = c.stepped = false;
  // Transfers in the order the pipeline consumes them.  The fixed cloud goes first on the
  // context's stream; the movable cloud follows on the copy stream, and while it crosses PCIe the
  // fixed-side work (subsample, k-NN + PCA normals) runs.  With the overlap filter the selection
  // itself needs the movable grid, so there the order is mov, fix as in sicp_set_clouds.
  // The second transfer is queued only AFTER the first cloud's grid build: that build reads a few
  // bytes back (bounding box, occupancy) and every device->host transaction issued while the
  // 24 MB host->device copy is in flight was measured to complete only when the copy ends
  // (bbox read-back 0.46 ms instead of 0.03 ms, whether by memcpy or by a store to mapped memory).
  {
    StageTimer t(c, &c.tm.upload_ms);
    upload_cloud(c, overlap ? c.mov_xyz.p : c.fix_xyz.p, overlap ? mov_xyz : fix_xyz,
                 sizeof(double) * 3 * (overlap ? n_mov : n_fix));
    t.stop();
  }
  auto queue_second_copy = [&]() {
    start_background_upload(c, overlap ? c.fix_xyz.p : c.mov_xyz.p, overlap ? fix_xyz : mov_xyz,
                            sizeof(double) * 3 * (overlap ? n_fix : n_mov));
    tr("2nd copy queued");
  };
  auto build_mov = [&]() {
    StageTimer t(c, &c.tm.grid_mov_ms);
    grid_build(c, c.gmov, c.mov_xyz.p, n_mov);
    make_float4_copy(c);
    t.stop();
  };
  auto build_fix = [&]() {
    StageTimer t(c, &c.tm.grid_fix_ms);
    grid_build(c, c.gfix, c.fix_xyz.p, n_fix);
    t.stop();
  };
  c.sel_idx.reserve(n_fix);
  c.tm.overlap_ms = 0;
  if (overlap) {
    build_mov();
    queue_second_copy();
    wait_background_upload(c);
    // PointCloud.select_in_range on all fixed points (simpleicp.py:160-170), compacted on the host
    k_iota<<<(unsigned)((n_fix + 255) / 256), 256, 0, c.stream>>>(c.sel_idx.p, n_fix);
    c.K = n_fix;
    gather_queries_launch(c);
    Rigid T0 = rigid_from_x(rp->run.lsq.x0);
    init_state(c, nullptr, &T0, true);
    StageTimer t(c, &c.tm.overlap_ms);
    c.dist.reserve(c.K);
    c.keep.reserve(c.K);
    match_launch(c, false, c.dist.p, nullptr, true, rp->max_overlap_distance * rp->max_overlap_distance);
    SICP_CUDA(cudaMemsetAsync(c.misc_counters.p + 8, 0, sizeof(unsigned int), c.stream));
    k_range_keep<<<(unsigned)((c.K + 255) / 256), 256, 0, c.stream>>>(
        c.dist.p, c.K, rp->max_overlap_distance * rp->max_overlap_distance, c.keep.p, c.misc_counters.p + 8);
    std::vector<uint8_t> keep((size_t)n_fix);
    copy_any(c, keep.data(), c.keep.p, (size_t)n_fix);
    t.stop();
    std::vector<long long> idx;
    idx.reserve((size_t)n_fix);
    for (long long i = 0; i < n_fix; ++i)
      if (keep[(size_t)i]) idx.push_back(i);
    SICP_REQUIRE(!idx.empty(), SICP_ERR_NO_OVERLAP, "Point clouds do not overlap within max_overlap_distance");
    copy_any(c, c.sel_idx.p, idx.data(), sizeof(long long) * idx.size());
    sync(c);  // idx is a local
    c.K = (long long)idx.size();
    build_fix();
  } else {
    build_fix();
    queue_second_copy();
    if (rp->correspondences < n_fix) {
      k_select_n<<<(unsigned)((rp->correspondences + 255) / 256), 256, 0, c.stream>>>(
          nullptr, n_fix, rp->correspondences, c.variant != SICP_VARIANT_PYTHON, c.sel_idx.p);
      c.K = rp->correspondences;
    } else {
      k_iota<<<(unsigned)((n_fix + 255) / 256), 256, 0, c.stream>>>(c.sel_idx.p, n_fix);
      c.K = n_fix;
    }
  }
  if (rp->correspondences < c.K) {
    c.sel_tmp.reserve(rp->correspondences);
    k_select_n<<<(unsigned)((rp->correspondences + 255) / 256), 256, 0, c.stream>>>(
        c.sel_idx.p, c.K, rp->correspondences, c.variant != SICP_VARIANT_PYTHON, c.sel_tmp.p);
    SICP_CUDA(cudaMemcpyAsync(c.sel_idx.p, c.sel_tmp.p, sizeof(long long) * rp->correspondences,
                              cudaMemcpyDeviceToDevice, c.stream));
    c.K = rp->correspondences;
  }
  tr("fix grid+select");
  gather_queries_launch(c);
  {
    StageTimer t(c, &c.tm.normals_ms);
    estimate_normals_launch(c, rp->neighbors);
    c.have_normals = true;
    t.stop();
  }
  tr("normals");
  if (!overlap) {
    wait_background_upload(c);
    build_mov();
  }
  tr("mov grid");
  if (n_selected) *n_selected = c.K;
  run_loop(ctx, c, &rp->run, out, log);
  tr("loop");
  if (mov_xyz_out) {
    transform_to(c, rigid_from_H(c.last_T), mov_xyz_out);
  }
  SICP_CUDA(cudaStreamSynchronize(c.copy_stream));
  sync(c);
  tr("transform+d2h");
  API_END
}

int32_t sicp_time_stages(sicp_ctx* ctx, const sicp_run_params* p, int32_t reps, int32_t flush_l2,
                         double ms[4]) {
  API_BEGIN(ctx)
  require_normals(c);
  SICP_REQUIRE(p && ms && reps >= 1, SICP_ERR_BAD_ARG, "bad argument");
  const size_t kFlushBytes = 256ull << 20;
  // flush_l2: bit 0 = overwrite the 256 MiB scratch before every iteration; bit 1 = record only the
  // two outer events (the three inner ones cost ~8 us of stream bubbles per iteration: the
  // whole-iteration time is taken without them, the per-kernel split in a second call with them)
  const bool outer_only = (flush_l2 & 2) != 0;
  flush_l2 &= 1;
  if (flush_l2) c.flush_buf.reserve(kFlushBytes);
  cudaEvent_t e[4];
  for (auto& ev : e) SICP_CUDA(cudaEventCreate(&ev));
  double acc[4] = {0, 0, 0, 0};
  bool allow_fused = true;
  for (int attempt = 0; attempt < 2; ++attempt) {
    for (int i = 0; i < 4; ++i) acc[i] = 0;
    for (int r = 0; r < reps; ++r) {
      if (flush_l2) SICP_CUDA(cudaMemsetAsync(c.flush_buf.p, r & 0xff, kFlushBytes, c.stream));
      SICP_CUDA(cudaEventRecord(e[0], c.stream));
      launch_iteration(c, *p, ctx->it_counter, false, 0, allow_fused, false, outer_only ? nullptr : e[1],
                       outer_only ? nullptr : e[2]);
      SICP_CUDA(cudaEventRecord(e[3], c.stream));
      SICP_CUDA(cudaEventSynchronize(e[3]));
      ctx->it_counter++;
      float t01 = 0, t12 = 0, t23 = 0, t03 = 0;
      if (!outer_only) {
        cudaEventElapsedTime(&t01, e[0], e[1]);
        cudaEventElapsedTime(&t12, e[1], e[2]);
        cudaEventElapsedTime(&t23, e[2], e[3]);
      }
      cudaEventElapsedTime(&t03, e[0], e[3]);
      acc[0] += t01;
      acc[1] += t12;
      acc[2] += t23;
      acc[3] += t03;
    }
    // a missed prediction parks the pipeline (every later launch returns at once): such a
    // measurement is void — repeat it through the general kernel
    DevState h;
    SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
    sync(c);
    if (h.stop != 3) break;
    clear_stop_flag(c);
    allow_fused = false;
  }
  for (auto& ev : e) cudaEventDestroy(ev);
  for (int i = 0; i < 4; ++i) ms[i] = acc[i] / reps;
  c.matched = c.rejected = c.stepped = true;
  API_END
}

int32_t sicp_get_iteration(sicp_ctx* ctx, sicp_iter_record* rec, double T[16], int64_t* nn_idx,
                           double* dist, uint8_t* keep) {
  API_BEGIN(ctx)
  SICP_REQUIRE(c.stepped, SICP_ERR_STATE, "no sicp_iterate / sicp_time_stages iteration to read back");
  DevState h;
  fetch_records(c, 0, 1);
  SICP_CUDA(cudaMemcpyAsync(&h, c.dev_state.p, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
  if (nn_idx) copy_any(c, nn_idx, c.nn_idx.p, sizeof(long long) * c.K);
  if (dist) copy_any(c, dist, c.dist.p, sizeof(double) * c.K);
  if (keep) copy_any(c, keep, c.keep.p, (size_t)c.K);
  sync(c);
  if (rec) *rec = c.rec_host[0];
  if (T) H_from_rigid(h.T, T);
  API_END
}

int32_t sicp_get_phase_times(sicp_ctx* ctx, double us[32]) {
  API_BEGIN(ctx)
  SICP_REQUIRE(us != nullptr, SICP_ERR_BAD_ARG, "us is NULL");
  SICP_REQUIRE(c.phase_t.p != nullptr, SICP_ERR_STATE, "no reject/solve kernel has run");
  unsigned long long t[32];
  SICP_CUDA(cudaMemcpyAsync(t, c.phase_t.p, sizeof(t), cudaMemcpyDeviceToHost, c.stream));
  sync(c);
  for (int i = 0; i < 32; ++i)
    us[i] = (i >= 24) ? (double)t[i] : ((t[i] >= t[0]) ? (double)(t[i] - t[0]) * 1e-3 : -1.0);
  API_END
}

int32_t sicp_get_timings(sicp_ctx* ctx, sicp_timings* t) {
  API_BEGIN(ctx)
  SICP_REQUIRE(t != nullptr, SICP_ERR_BAD_ARG, "t is NULL");
  c.tm.fused_iterations = c.n_fused_last;
  c.tm.rerun_iterations = c.n_rerun_last;
  *t = c.tm;
  API_END
}

}  // extern "C"
