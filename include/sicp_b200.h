/*
 * sicp_b200.h — C ABI of libsicp_b200.so: the B200 (sm_100a) ICP inner loop behind the
 * simpleICP Python API.
 *
 * The reference (pglira/simpleICP) has no FFI/plugin layer (SURVEY.md §0.9); its boundary is the
 * Python class surface exported at python/simpleicp/__init__.py:12-14.  This header is the
 * C boundary a binding of that surface needs: one entry point per reference method on the hot
 * path, each citing the reference code it replaces (paths relative to the reference repo).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch / C++ types.
 *  - Every function returns a sicp_status; sicp_last_error(ctx) gives the message.
 *  - Pointers marked [h|d] may be host or device memory (detected with
 *    cudaPointerGetAttributes); [h] must be host memory.  The caller owns every buffer it passes
 *    and allocates every output; the library never frees or keeps caller memory.
 *  - All point arrays are row-major n x 3 float64 (NumPy's layout for PointCloud.X,
 *    python/simpleicp/pointcloud.py:81-84).  Indices are int64 like NumPy's.
 *  - A context is bound to one device and one CUDA stream (e.g. torch's current stream); calls
 *    on one context are not thread-safe, different contexts are independent.
 *  - Angles are radians at this boundary (the Python facade converts degrees,
 *    python/simpleicp/simpleicp.py:146-148).
 */
#ifndef SICP_B200_H
#define SICP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SICP_ABI_VERSION 2

typedef enum {
  SICP_OK = 0,
  SICP_ERR_BAD_ARG = 1,       /* argument checks, simpleicp.py:326-353, pointcloud.py:158-159   */
  SICP_ERR_NO_OVERLAP = 2,    /* "Point clouds do not overlap ...", simpleicp.py:165-170         */
  SICP_ERR_TOO_FEW_CORR = 3,  /* "Too few correspondences!" (< 6), simpleicp.py:209-214          */
  SICP_ERR_CUDA = 4,
  SICP_ERR_SINGULAR = 5,      /* normal equations not positive definite                          */
  SICP_ERR_STATE = 6          /* call order violated (e.g. match before set_clouds)              */
} sicp_status;

typedef struct sicp_ctx sicp_ctx;

/* Nearest-neighbour engine selection (both engines are exact). */
typedef enum {
  SICP_NN_AUTO = 0,  /* uniform-grid search, TMA brute force for queries the grid cannot bound */
  SICP_NN_GRID = 1,  /* grid only, ring expansion until proven exact                           */
  SICP_NN_BRUTE = 2  /* TMA-staged tiled brute force for every query                           */
} sicp_nn_engine;

/* Normal sign convention.  The reference's sign is whatever LAPACK dgeev returns
 * (pointcloud.py:191-197, np.linalg.eig) — see DESIGN.md "normal sign". */
typedef enum {
  SICP_SIGN_DGEEV = 0,     /* reproduce np.linalg.eig's sign (Hessenberg-QR path of dgeev)       */
  SICP_SIGN_CANONICAL = 1  /* largest-magnitude component positive                              */
} sicp_sign_mode;

/* Algorithm variant of reject + solve (option key "variant").  The default is the Python package's
 * algorithm (the north-star path).  The linearised variants restate the C++ driver
 * (c++/src/corrpts.cpp:59-156, c++/src/simpleicp.cpp:54-80; pinned to those sources, see
 * tests/test_cpp_reference_pin.py): median/MAD over ALL distances with the upper middle element
 * (std::nth_element at n/2), sigma = 1.4826 MAD, one linear solve A x = l per iteration, cloud
 * moved by the RIGID dH = H(euler(x), t), residuals A x - l, sample standard deviation, no
 * parameter uncertainties and no observed/fixed parameters.  They differ in the matrix that is
 * REPORTED: H * dH (the C++ driver, c++/src/simpleicp.cpp:66) or dH * H, the transform really
 * applied to the cloud and the composition order of the Rust / Julia / MATLAB drivers
 * (rust/src/icp.rs:164, julia/simpleicp.jl:272, matlab/simpleicp.m:55).  Those three ports differ
 * from the C++ arithmetic in two more points that are NOT reproduced: they move the cloud by the
 * linearised matrix I + [x]_x itself (rust/src/icp.rs:339-344, matlab/simpleicp.m:146-152) -- not
 * a rotation, so distances are not preserved and the search could not stay in the static grid
 * of the untouched cloud -- and they average the two middle elements of an even-sized sample
 * (rust/src/icp.rs:392-404).  Both effects are second order in the per-iteration angles.
 * Normals stay in the float32 storage of the default variant (the C++ code keeps float64), see
 * DESIGN.md.                                                                                    */
typedef enum {
  SICP_VARIANT_PYTHON = 0,
  SICP_VARIANT_LINEARIZED = 1,        /* C++ arithmetic, reports dH * H                          */
  SICP_VARIANT_LINEARIZED_CPP = 2     /* C++ arithmetic, reports H * dH (the C++ driver itself)  */
} sicp_variant;

/* ---- life cycle --------------------------------------------------------------------------- */
int32_t sicp_abi_version(void);
int32_t sicp_create(int32_t device, void* cuda_stream, sicp_ctx** out);
int32_t sicp_destroy(sicp_ctx* ctx);
const char* sicp_last_error(sicp_ctx* ctx); /* ctx may be NULL: last error of the calling thread */
int32_t sicp_set_option(sicp_ctx* ctx, const char* key, double value);
/*  keys: "nn_engine" (sicp_nn_engine), "sign_mode" (sicp_sign_mode), "variant" (sicp_variant),
 *        "grid_target_occupancy"
 *        (points per occupied cell, default 3), "grid_max_rings" (ring limit before the
 *        brute-force pass takes over, default 8), "grid_sort_cells" (0/1), "host_sync_every"
 *        (iterations queued between host reads in sicp_run, default 4), "match_group" (lanes per
 *        query in the grid search: 0 = by K, 1, 4, 8, 16), "rs_blocks" (blocks of the cooperative
 *        reject/solve kernel, 0 = one per SM), "fused" (1: iterations after the first run their
 *        reject + solve in the barrier-free kernel, 0: always the cooperative kernel),
 *        "warm_start" (1: the grid search of an iteration starts from the previous iteration's
 *        neighbour as upper bound), "keep_knn" (see sicp_get_knn), "knn_coop" (k-NN search: 1 cooperative
 *        lanes per query (k <= 16), 0 one thread per query, -1 (default) by the number of queries),
 *        "upload_threads" (worker threads that stage a cloud given in PAGEABLE host memory --
 *        e.g. a NumPy array -- through pinned buffers, default 2; 0: plain cudaMemcpyAsync, which
 *        the driver stages on the calling thread; pinned and device sources never use them),
 *        "upload_chunk_kb" (slice size of that staging, default 2048), "defaults" (any value:
 *        every option back to its default)                              */

/* ---- clouds: SimpleICP.add_point_clouds (simpleicp.py:58-73) + PointCloud.X ---------------- */
int32_t sicp_set_clouds(sicp_ctx* ctx, const double* fix_xyz /*[h|d] n_fix x 3*/, int64_t n_fix,
                        const double* mov_xyz /*[h|d] n_mov x 3*/, int64_t n_mov);

/* ---- selection: PointCloud.idx_selected / select_n_points (pointcloud.py:91-147) ----------- */
/* idx ascending fixed-cloud indices; idx == NULL selects all n_fix points.                    */
int32_t sicp_set_selected(sicp_ctx* ctx, const int64_t* idx /*[h|d] K or NULL*/, int64_t K);

/* PointCloud.select_in_range (pointcloud.py:149-171) as used at simpleicp.py:158-170:
 * keep[i] = 1 iff the nearest point of H0 * X_mov to selected fixed point i is STRICTLY closer
 * than max_range.  n_kept == 0 returns SICP_ERR_NO_OVERLAP.                                    */
int32_t sicp_select_in_range(sicp_ctx* ctx, const double H0[16], double max_range,
                             uint8_t* keep /*[h|d] K*/, int64_t* n_kept /*[h]*/);

/* ---- normals: PointCloud.estimate_normals (pointcloud.py:173-203) ---------------------------
 * k-NN (self included) in the fixed cloud, covariance (ddof=1), symmetric 3x3 eigen-solve;
 * normal = eigenvector of the smallest eigenvalue, planarity = (l_mid - l_min) / l_max, float32.
 * Outputs may be NULL (kept on the device for sicp_match either way).                          */
int32_t sicp_estimate_normals(sicp_ctx* ctx, int32_t neighbors, float* nx, float* ny, float* nz,
                              float* planarity /*[h|d] K each*/);
/* The reference's "columns already present" hook (simpleicp.py:176-178).                       */
int32_t sicp_set_normals(sicp_ctx* ctx, const float* nx, const float* ny, const float* nz,
                         const float* planarity /*[h|d] K each*/);
/* Movable-side attributes (optional; the default run has none).  Arrays of n_mov floats in the
 * movable cloud's own frame, NaN where not estimated; all four NULL clears them; a new movable
 * cloud (sicp_set_clouds / sicp_register) clears them too.
 *  - planarity: second branch of CorrPts.reject_wrt_planarity (corrpts.py:157-162): when pc_mov
 *    carries a planarity column, a correspondence must pass min_planarity on BOTH sides; NaN
 *    fails.  The median / MAD of the distance rejection are taken over that set.
 *  - max_angle_rad in [0, pi/2]: CorrPts.reject_wrt_to_angle_between_normals — the hook the
 *    reference declares, calls after the distance rejection (simpleicp.py:207, commented out)
 *    and leaves `raise NotImplementedError` (corrpts.py:190-193).  Here: a correspondence that
 *    survived both rejections is dropped when acos|n_fix . (R n_mov)| > max_angle_rad, R the
 *    rotation of the iteration's transform.  Negative: no angle test.
 * Both act in sicp_match/sicp_reject/sicp_solve, sicp_iterate and sicp_run; sicp_register and
 * sicp_register_batch take their clouds themselves and always run without them.               */
int32_t sicp_set_mov_normals(sicp_ctx* ctx, const float* nx, const float* ny, const float* nz,
                             const float* planarity /*[h|d] n_mov each*/, double max_angle_rad);
/* neighbour indices of the last sicp_estimate_normals (test/inspection hook), K x neighbors; they
 * are only kept when option "keep_knn" was 1 during that call.                                  */
int32_t sicp_get_knn(sicp_ctx* ctx, int64_t* idx /*[h|d] K x k*/, double* dist2 /*[h|d] or NULL*/);

/* ---- one ICP iteration, stage by stage ------------------------------------------------------ */
/* CorrPts.match (corrpts.py:124-137, 195-211): pc2_idx[i] = argmin_j |H x_mov_j - x_fix_sel_i|,
 * dist[i] = (H x_mov_pc2idx - x_fix_sel_i) . n_i.                                              */
int32_t sicp_match(sicp_ctx* ctx, const double H[16], int64_t* pc2_idx /*[h|d] K or NULL*/,
                   double* dist /*[h|d] K or NULL*/);

/* CorrPts.reject_wrt_planarity + reject_wrt_point_to_plane_distances (corrpts.py:139-188):
 * (double)planarity_f32 >= min_planarity (NaN drops), then |d - median| <= 3 * MAD with the
 * RAW median absolute deviation (SciPy scale=1.0, corrpts.py:186).
 * stats[4] = {median, mad, mean(d kept), popstd(d kept)}.                                      */
int32_t sicp_reject(sicp_ctx* ctx, double min_planarity, uint8_t* keep /*[h|d] K or NULL*/,
                    int64_t* n_kept /*[h]*/, double stats[4] /*[h] or NULL*/);

typedef struct {
  double x0[6];           /* start values alpha1..3 [rad], tx,ty,tz (simpleicp.py:223-227)       */
  double observed[6];     /* rbp_observed_values, radians                                      */
  double obs_weight[6];   /* rbp_observation_weights: 0 free, +inf fixed, else observed          */
  double distance_weight; /* > 0; <= 0 or NaN means "None": 1/std(d kept)^2 (simpleicp.py:233)   */
} sicp_lsq_params;

/* SimpleICPOptimization.estimate_parameters (optimization.py:65-124): argmin over the free
 * parameters of sum (w n.(R(x) p2 + t - p1))^2 + sum (w_j (x_j - obs_j))^2, solved to
 * convergence (Levenberg-Marquardt on the exact Euler model).  residuals = unweighted signed
 * distances at the solution, in kept order.  stats[2] = {mean, population std} of them.        */
int32_t sicp_solve(sicp_ctx* ctx, const sicp_lsq_params* p, double x[6] /*[h]*/,
                   double H[16] /*[h]*/, double* residuals /*[h|d] n_kept or NULL*/,
                   double stats[2] /*[h] or NULL*/, double* distance_weight_used /*[h] or NULL*/);

/* SimpleICPOptimization.estimate_parameter_uncertainties (optimization.py:126-170) for the last
 * sicp_solve / sicp_run: sigma[j] = sqrt(Cxx_jj), NaN for fixed parameters.                     */
int32_t sicp_uncertainties(sicp_ctx* ctx, double sigma[6] /*[h]*/);

/* ---- the fused loop: SimpleICP.run iterations (simpleicp.py:184-281) ------------------------ */
typedef struct {
  double min_planarity;
  double min_change;       /* percent, simpleicp.py:355-379                                     */
  int32_t max_iterations;
  int32_t reserved;
  sicp_lsq_params lsq;     /* x0 = observed values on iteration 0, as the reference              */
} sicp_run_params;

typedef struct {
  int64_t n_kept;
  double median, mad;          /* of the planarity survivors                                    */
  double mean_dist, std_dist;  /* kept distances before the solve ("orig:0" row on iteration 0)  */
  double x[6];
  double mean_res, std_res;    /* residuals after the solve (log row, stop rule)                */
  double distance_weight;
  int32_t lm_iterations;
  int32_t n_bruteforce;        /* queries answered by the brute-force engine                    */
} sicp_iter_record;

typedef struct {
  int32_t iterations;          /* number of iterations run (the reference's it + 1)             */
  int32_t converged;           /* 1 if the stop rule fired, 0 if max_iterations was reached     */
  double x[6];
  double H[16];
  double sigma[6];
  int64_t n_residuals;
  double loop_ms;              /* device time of the iteration loop (CUDA events)               */
} sicp_run_result;

int32_t sicp_run(sicp_ctx* ctx, const sicp_run_params* p, sicp_run_result* out /*[h]*/,
                 sicp_iter_record* log /*[h] max_iterations entries or NULL*/);
/* The rigid transform the last sicp_run / sicp_solve actually applied to the movable cloud.  Equal
 * to the result's H except for SICP_VARIANT_LINEARIZED_CPP, whose reported H = H * dH is a
 * different product of the same increments (c++/src/simpleicp.cpp:62-66: the cloud is moved by
 * dH on the left, the report multiplies on the right).                                         */
int32_t sicp_get_transform(sicp_ctx* ctx, double T[16] /*[h]*/);
/* residuals of the final iteration in kept order (simpleicp.py:324, 4th return value).          */
int32_t sicp_get_residuals(sicp_ctx* ctx, double* residuals /*[h|d] cap*/, int64_t cap,
                           int64_t* n /*[h]*/);

/* One iteration (match + reject + solve) with no host round trip except the record; used by the
 * benchmark to time the hot path in isolation.  x_in/out: cumulative parameters.              */
int32_t sicp_iterate(sicp_ctx* ctx, const sicp_run_params* p, const double x_in[6],
                     sicp_iter_record* rec /*[h] or NULL: fully asynchronous*/);

/* PointCloud.select_n_points (pointcloud.py:121-147) applied to the CURRENT selection on the
 * device: keeps the points at rint(linspace(0, m-1, n)) (numpy arithmetic; the linearised
 * variants round half away from zero as c++/src/pointcloud.cpp:92-96 does); no-op when n >= m.
 * idx_out (may be NULL) receives the resulting selection, sicp_set_selected's K is updated.     */
int32_t sicp_select_n_points(sicp_ctx* ctx, int64_t n, int64_t* idx_out /*[h|d] min(n, m) or NULL*/);

/* ---- SimpleICP.run as ONE call (simpleicp.py:75-324) --------------------------------------------
 * add_point_clouds + [select_in_range] + select_n_points + estimate_normals + the iteration loop
 * + the final transform_by_H, scheduled so that the host->device transfer of the movable cloud
 * overlaps the fixed-side work (grid, subsample, normals).  Equivalent to sicp_set_clouds,
 * sicp_set_selected(NULL), [sicp_select_in_range], sicp_select_n_points, sicp_estimate_normals,
 * sicp_run, sicp_transform in sequence; every stage-by-stage call remains valid afterwards
 * (sicp_get_residuals, sicp_get_knn, sicp_match ...).                                            */
typedef struct {
  int64_t correspondences;       /* simpleicp.py:78 (default 1000)                                */
  int32_t neighbors;             /* simpleicp.py:79 (default 10)                                  */
  int32_t reserved;
  double max_overlap_distance;   /* <= 0 or +inf: clouds fully overlap (simpleicp.py:81)          */
  sicp_run_params run;
} sicp_register_params;
int32_t sicp_register(sicp_ctx* ctx, const double* fix_xyz /*[h|d] n_fix x 3*/, int64_t n_fix,
                      const double* mov_xyz /*[h|d] n_mov x 3*/, int64_t n_mov,
                      const sicp_register_params* p, sicp_run_result* out /*[h]*/,
                      sicp_iter_record* log /*[h] max_iterations entries or NULL*/,
                      double* mov_xyz_out /*[h|d] n_mov x 3 or NULL*/,
                      int64_t* n_selected /*[h] or NULL*/);

/* ---- many independent pairs in one call (BASELINE.json configs[4]; SURVEY.md section 8e) --------
 * SimpleICP.run (simpleicp.py:75-324) for n_pairs independent (fixed, movable) pairs on ONE GPU
 * with ONE set of kernel launches per stage and per iteration for the whole batch: the grids of
 * all 2 n_pairs clouds are built in one segmented counting sort, the searches of all pairs run in
 * one launch, reject + solve run one block per pair, every pair has its own stop flag.  Results
 * per pair equal those of sicp_register on that pair.
 * fix_xyz[i] / mov_xyz[i] point to the i-th pair's clouds (host, ideally pinned, or device);
 * correspondences must be <= 4096 (one block per pair).  A finite max_overlap_distance > 0 runs
 * the partial-overlap filter of sicp_register on every pair (simpleicp.py:150-170, from the
 * initial transform of p->run.lsq.x0, one distance and one initial transform for the whole call).
 * out[i].status is the sicp_status of pair i (a pair without enough correspondences, or whose
 * clouds do not overlap within max_overlap_distance, fails alone); the call itself fails only on
 * bad arguments or CUDA errors.                                                                   */
typedef struct {
  int32_t status;
  int32_t iterations;
  int32_t converged;
  int32_t n_selected;         /* fixed points the loop used (sicp_register's n_selected); 0 when
                                 status is SICP_ERR_NO_OVERLAP                                     */
  int64_t n_kept;
  double H[16];
  double x[6];
  double sigma[6];
  double mean_res, std_res;   /* of the final residuals (exact, two-pass)                       */
} sicp_pair_result;
int32_t sicp_register_batch(sicp_ctx* ctx, int32_t n_pairs, const double* const* fix_xyz /*[h|d]*/,
                            const int64_t* n_fix, const double* const* mov_xyz /*[h|d]*/,
                            const int64_t* n_mov, const sicp_register_params* p,
                            sicp_pair_result* out /*[h] n_pairs*/);

/* ---- PointCloud.transform_by_H (pointcloud.py:205-217), final application simpleicp.py:316 -- */
int32_t sicp_transform(sicp_ctx* ctx, const double H[16], double* mov_xyz_out /*[h|d] n_mov x 3*/);

/* ---- device timing of the last call of each stage, milliseconds ---------------------------- */
typedef struct {
  double upload_ms, grid_mov_ms, grid_fix_ms, overlap_ms, normals_ms, match_ms, reject_solve_ms,
      transform_ms;
  int64_t kernel_launches; /* kernels of this library launched on this context so far           */
  int64_t fused_iterations; /* last sicp_run / sicp_register: iterations whose reject + solve ran
                               in the barrier-free kernel (all but the first, normally)          */
  int64_t rerun_iterations; /* ... iterations repeated through the general kernel because the
                               order-statistic prediction of the barrier-free kernel missed       */
} sicp_timings;
int32_t sicp_get_timings(sicp_ctx* ctx, sicp_timings* t /*[h]*/);

/* Measurement hook: run `reps` iterations from the current device state and return the average
 * device time (CUDA events on the context's stream) of each kernel group, in milliseconds:
 * ms[0] grid match kernel, ms[1] brute-force pass (launched, usually empty), ms[2] reject+solve
 * kernel, ms[3] whole iteration.  flush_l2 bit 0: overwrite a 256 MiB scratch buffer before every
 * iteration (outside the timed intervals) so each one starts with a cold L2; bit 1: record only
 * the two outer events (ms[0..2] = 0) — the inner events cost several microseconds of stream
 * bubbles per iteration, so the whole-iteration time is taken without them.                     */
int32_t sicp_time_stages(sicp_ctx* ctx, const sicp_run_params* p, int32_t reps, int32_t flush_l2,
                         double ms[4] /*[h]*/);
/* What the last iteration of sicp_iterate or sicp_time_stages computed, read back without
 * launching anything: its record, the cumulative transform after it, and per selected point the
 * matched movable index, the point-to-plane distance and the keep flag of the rejection (K entries
 * each).  Any output may be NULL.  SICP_ERR_STATE once another call has changed the loop state.  */
int32_t sicp_get_iteration(sicp_ctx* ctx, sicp_iter_record* rec /*[h]*/, double T[16] /*[h]*/,
                           int64_t* nn_idx /*[h|d] K*/, double* dist /*[h|d] K*/,
                           uint8_t* keep /*[h|d] K*/);
/* Diagnostics: %globaltimer stamps block 0 took in the last reject+solve kernel, microseconds
 * relative to kernel entry.  [1] median done, [2] MAD done, [3] moments accumulated, [4] grid
 * barrier passed, [5] LM solve done, [6] barrier, [7] residual pass, [8] barrier, [9] exit;
 * [10..12] / [14..16] radix levels done / gather barrier / sort done for the median / MAD;
 * [24],[25] radix levels used, [26],[27] candidates sorted (raw counts, not times); [28] path:
 * 0 radix select, 1 predictor histogram (cooperative kernel), 2 barrier-free kernel (there
 * [2] = select done, [3] = accumulation done in block 0, [4] = last block starts, [17] partials
 * reduced, [18] M assembled, [19] solve done, [9] exit).                                        */
int32_t sicp_get_phase_times(sicp_ctx* ctx, double us[32] /*[h]*/);

/* ---- .xyz text I/O (host only; SURVEY.md section 8f: file parsing dominates end-to-end time on
 * the lidar sets).  Contract of the reference readers (c++/src/simpleicp-cli.cpp:72-128,
 * rust/src/io.rs:9-37, np.genfromtxt in python/simpleicp/tests/test_simpleicp.py:102-103):
 * whitespace-separated x y z per line; '/' or '#' comment lines and blank lines are skipped.
 * sicp_xyz_load allocates *xyz (n x 3 float64, row-major); release it with sicp_xyz_free.
 * sicp_xyz_save mirrors PointCloud.write_xyz (python/simpleicp/pointcloud.py:219-226):
 * header != 0 writes the "//X Y Z" line, decimals < 0 writes round-trip precision.            */
int32_t sicp_xyz_load(const char* path, double** xyz /*out*/, int64_t* n /*out*/);
void sicp_xyz_free(double* xyz);
int32_t sicp_xyz_save(const char* path, const double* xyz /*[h] n x 3*/, int64_t n,
                      int32_t decimals, int32_t header);
const char* sicp_io_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* SICP_B200_H */
