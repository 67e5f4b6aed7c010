"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden vectors
captured from the unmodified reference.  Tolerances are written next to each comparison:
bit-exact for indices and masks, 1e-12 for float64 quantities computed the same way, and the
reference solver's own slack (lmfit/TRF ftol = xtol = 1e-8 -> ~3e-6 per iteration, SURVEY.md
§0.2) where the comparison crosses the least-squares solve."""
import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial import cKDTree

from conftest import load_golden, load_pair
from oracle import simpleicp_oracle as O

import simpleicp_b200 as sb
from simpleicp_b200 import _capi

pytestmark = pytest.mark.gpu

CONFIGS = ["dragon", "bunny", "multisensor", "webots", "dragon_observed", "airborne", "terrestrial"]


def obs_rad(kwargs):
    obs = np.array(kwargs.get("rbp_observed_values", (0.0,) * 6), dtype=float)
    obs[:3] *= np.pi / 180
    return obs


def H_inputs(g):
    """H used for matching in every iteration of the golden run."""
    xs = [obs_rad(g["kwargs"])] + [g["it_x"][i] for i in range(g["it_x"].shape[0] - 1)]
    return [O.rbp_to_H(x) for x in xs]


def full_normals(g, n_fix):
    out = [np.full(n_fix, np.nan, dtype=np.float32) for _ in range(4)]
    for a in range(3):
        out[a][g["idx_sel"]] = g["normals"][:, a]
    out[3][g["idx_sel"]] = g["planarity"]
    return tuple(out)


@pytest.fixture(scope="module")
def engines(gpu):
    cache = {}

    def get(name, engine_mode=_capi.NN_AUTO):
        key = (name, engine_mode)
        if key not in cache:
            g = load_golden(name)
            X_fix, X_mov = load_pair(name)
            e = _capi.Engine()
            e.set_option("nn_engine", engine_mode)
            e.set_clouds(X_fix, X_mov)
            e.set_selected(g["idx_sel"])
            e.set_normals(g["normals"][:, 0], g["normals"][:, 1], g["normals"][:, 2], g["planarity"])
            cache[key] = (e, g, X_fix, X_mov)
        return cache[key]

    yield get
    for e, *_ in cache.values():
        e.close()


def assert_same_nn(idx_gpu, idx_ref, q, X_mov_t, what):
    """Indices equal; where they differ both candidates must be at the same distance (ties:
    cKDTree's tie order is unspecified, ours is lowest index)."""
    bad = np.flatnonzero(idx_gpu != idx_ref)
    for i in bad:
        da = np.linalg.norm(X_mov_t[idx_gpu[i]] - q[i])
        db = np.linalg.norm(X_mov_t[idx_ref[i]] - q[i])
        assert abs(da - db) <= 1e-12 * max(1.0, db), f"{what}: query {i}: {da} vs {db}"
    return len(bad)


@pytest.mark.parametrize("mode", [_capi.NN_AUTO, _capi.NN_GRID, _capi.NN_BRUTE])
@pytest.mark.parametrize("name", CONFIGS)
def test_match_lockstep(engines, name, mode):
    """CorrPts.match for every golden iteration: pc2_idx identical, distances to 1e-12."""
    e, g, X_fix, X_mov = engines(name, mode)
    q = X_fix[g["idx_sel"]]
    n_ties = 0
    for it, H in enumerate(H_inputs(g)):
        idx, d = e.match(H)
        X_t = O.transform_by_H(X_mov, H)
        n_ties += assert_same_nn(idx, g["it_pc2_idx"][it], q, X_t, f"{name} it {it}")
        same = idx == g["it_pc2_idx"][it]
        np.testing.assert_allclose(d[same], g["it_dist"][it][same], rtol=0, atol=1e-12)
    # webots is a synthetic scene on a regular 1 mm lattice: a sixth of its queries have exactly
    # equidistant candidates; terrestrial is a mm-resolution scan stored with 3 decimals (3.4 % of
    # its queries have exact ties); the other scanned data sets have a handful
    limit = {"webots": 0.25, "terrestrial": 0.05}.get(name, 0.01)
    assert n_ties <= limit * q.shape[0] * len(H_inputs(g))


@pytest.mark.parametrize("name", CONFIGS)
def test_reject_lockstep(engines, name):
    """Planarity + median/MAD rejection: keep mask bit-identical, median/MAD to 1e-15."""
    e, g, X_fix, X_mov = engines(name)
    for it, H in enumerate(H_inputs(g)):
        idx, d = e.match(H)
        keep, n_kept, st = e.reject(g["kwargs"].get("min_planarity", 0.3))
        keep_o, med_o, mad_o = O.reject(d, g["planarity"], g["kwargs"].get("min_planarity", 0.3))
        assert np.array_equal(keep, keep_o), f"{name} it {it}"
        assert n_kept == int(keep_o.sum())
        assert st[0] == med_o and st[1] == mad_o  # exact order statistics
        if np.array_equal(idx, g["it_pc2_idx"][it]):
            assert np.array_equal(keep, g["it_keep"][it])
        np.testing.assert_allclose(st[2], d[keep].mean(), rtol=0, atol=1e-14)
        np.testing.assert_allclose(st[3], d[keep].std(), rtol=1e-10)


def tight_solution(p1, n1, p2, w, x0, obs, w_obs):
    obs, w_obs = np.asarray(obs, float), np.asarray(w_obs, float)
    free = np.flatnonzero(np.isfinite(w_obs))
    xf = np.array(x0, dtype=float)

    def fun(v):
        xf[free] = v
        return O._residual_vector(xf, p1, n1.astype(np.float64), p2, w, obs, w_obs)

    # 3-point differences: a 2-point Jacobian (what lmfit uses) limits the solution to ~1e-8
    r = least_squares(fun, xf[free].copy(), jac="3-point", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    xf[free] = r.x
    return xf.copy()


@pytest.mark.parametrize("name", CONFIGS)
def test_solve_lockstep(engines, name):
    """estimate_parameters: x against a tightly converged SciPy solve of the same problem
    (<= 1e-9), against the reference's lmfit result (its own ftol slack, <= 1e-5), residuals
    at the solution against the oracle's residual function (<= 1e-12)."""
    e, g, X_fix, X_mov = engines(name)
    kw = g["kwargs"]
    obs = obs_rad(kw)
    w_obs = np.array(kw.get("rbp_observation_weights", (0.0,) * 6), dtype=float)
    w = kw.get("distance_weights", 1)
    x_prev = obs
    for it, H in enumerate(H_inputs(g)):
        idx, d = e.match(H)
        keep, n_kept, st = e.reject(kw.get("min_planarity", 0.3))
        w_it = g["it_w"][it] if w is None else w
        x, Hs, res, rs, w_used = e.solve(x_prev, obs, w_obs, w_it, n_kept)
        p1 = X_fix[g["idx_sel"][keep]]
        p2 = X_mov[idx[keep]]
        n1 = g["normals"][keep]
        x_t = tight_solution(p1, n1, p2, w_it, x_prev, obs, w_obs)
        np.testing.assert_allclose(x, x_t, rtol=0, atol=2e-8, err_msg=f"{name} it {it}")
        if np.array_equal(keep, g["it_keep"][it]) and np.array_equal(idx, g["it_pc2_idx"][it]):
            np.testing.assert_allclose(x, g["it_x"][it], rtol=0, atol=1e-5)
        np.testing.assert_allclose(Hs, O.rbp_to_H(x), rtol=0, atol=1e-15)
        r_o = O._residual_vector(x, p1, n1.astype(np.float64), p2, 1.0, obs, np.zeros(6))
        np.testing.assert_allclose(res, r_o, rtol=0, atol=1e-12)
        np.testing.assert_allclose(rs[0], res.mean(), rtol=0, atol=1e-14)
        np.testing.assert_allclose(rs[1], res.std(), rtol=1e-9)
        # fixed parameters stay put
        for j in range(6):
            if not np.isfinite(w_obs[j]):
                assert x[j] == x_prev[j]
        sig = e.uncertainties()
        # oracle sigmas from a finite-difference Jacobian at the GPU's solution
        xo, res_u, res_w, jac = O.estimate_parameters(p1, n1, p2, w_it, x, obs, w_obs)
        sig_o = O.estimate_parameter_uncertainties(res_w, jac, n_kept, w_it, w_obs)
        np.testing.assert_allclose(sig, sig_o, rtol=1e-5, equal_nan=True)
        x_prev = g["it_x"][it]


def test_auto_distance_weight(engines):
    """distance_weights=None: w = 1 / std(kept distances)^2 on iteration 0 (simpleicp.py:233)."""
    e, g, X_fix, X_mov = engines("dragon_observed")
    kw = g["kwargs"]
    H = H_inputs(g)[0]
    idx, d = e.match(H)
    keep, n_kept, st = e.reject(0.3)
    x, Hs, res, rs, w_used = e.solve(obs_rad(kw), obs_rad(kw), kw["rbp_observation_weights"], None, n_kept)
    np.testing.assert_allclose(w_used, 1 / np.std(d[keep]) ** 2, rtol=1e-10)
    np.testing.assert_allclose(w_used, g["it_w"][0], rtol=1e-10)


NORMAL_CASES = [("dragon", 10), ("bunny", 10), ("webots", 40), ("multisensor", 10), ("airborne", 10),
                ("terrestrial", 10)]


@pytest.mark.parametrize("name,k", NORMAL_CASES)
def test_normals(gpu, name, k):
    """k-NN + PCA: neighbour distances equal cKDTree's (1e-12), normals equal the reference's up
    to sign (float32 store: 2e-7), planarity to 1e-6."""
    g = load_golden(name)
    X_fix, X_mov = load_pair(name)
    with _capi.Engine() as e:
        e.set_option("sign_mode", _capi.SIGN_CANONICAL)
        e.set_option("keep_knn", 1)
        e.set_clouds(X_fix, X_mov)
        e.set_selected(g["idx_sel"])
        nx, ny, nz, pl = e.estimate_normals(k)
        idx_knn, d2 = e.get_knn(k)
    dd, ii = cKDTree(X_fix).query(X_fix[g["idx_sel"]], k=k)
    np.testing.assert_allclose(np.sqrt(d2), dd, rtol=0, atol=1e-12)
    same_rows = (np.sort(idx_knn, axis=1) == np.sort(ii, axis=1)).all(axis=1)
    # the rest are equal-distance ties at the k-th neighbour (common on webots' regular lattice
    # and on the mm-quantised terrestrial scan: distances above are equal to 1e-12 in every row)
    assert same_rows.mean() > {"webots": 0.5, "terrestrial": 0.75}.get(name, 0.98)
    n_gpu = np.column_stack((nx, ny, nz)).astype(np.float64)
    n_ref = g["normals"].astype(np.float64)
    ok = np.isfinite(g["planarity"]) & same_rows
    dots = np.sum(n_gpu * n_ref, axis=1)
    aligned = n_gpu * np.sign(dots)[:, None]
    # poorly conditioned normals (nearly isotropic neighbourhoods) are excluded by the eigen gap
    gap_ok = ok & (g["planarity"] > 0.05)
    assert np.abs(aligned - n_ref)[gap_ok].max() < 5e-6
    assert np.abs(aligned - n_ref)[gap_ok & (g["planarity"] > 0.3)].max() < 1e-6
    np.testing.assert_allclose(pl[ok], g["planarity"][ok], rtol=0, atol=1e-6)
    # canonical sign: largest-magnitude component positive
    lead = np.take_along_axis(n_gpu, np.abs(n_gpu).argmax(axis=1)[:, None], axis=1)[:, 0]
    assert (lead[np.isfinite(lead)] >= 0).all()


@pytest.mark.parametrize("name", ["bunny", "multisensor", "webots"])
def test_overlap_filter(gpu, name):
    """select_in_range: the strictly-closer-than rule gives the reference's index set exactly."""
    g = load_golden(name)
    X_fix, X_mov = load_pair(name)
    H0 = O.rbp_to_H(obs_rad(g["kwargs"]))
    with _capi.Engine() as e:
        e.set_clouds(X_fix, X_mov)
        e.set_selected(None)
        keep = e.select_in_range(H0, g["kwargs"]["max_overlap_distance"])
    assert np.array_equal(np.flatnonzero(keep), g["idx_overlap"])


@pytest.mark.parametrize("name", CONFIGS)
def test_full_run_with_reference_normals(gpu, name):
    """Whole pipeline with the reference's normals injected through the reference's own
    pre-computed-columns hook: same iteration count, same kept counts, H within 1e-6 Frobenius
    (expected ~1e-9: both sides sit on the same ICP fixed point)."""
    g = load_golden(name)
    X_fix, X_mov = load_pair(name)
    res = sb.register(X_fix, X_mov, normals=full_normals(g, X_fix.shape[0]), **g["kwargs"])
    assert np.array_equal(res.idx_selected, g["idx_sel"])
    dH = np.linalg.norm(res.H - g["H"])
    kept = [r["n_kept"] for r in res.records]
    ref_kept = [int(k.sum()) for k in g["it_keep"]]
    print(f"{name}: |dH|_F = {dH:.3e}, iterations {res.iterations} vs {len(ref_kept)}, kept {kept[-3:]} vs {ref_kept[-3:]}")
    assert dH < 1e-6
    # terrestrial: 3.4 % of the queries have exactly equidistant candidates (cKDTree's pick among
    # them is unspecified); the fixed point is the same to 1e-12, the fragile stop rule
    # (SURVEY.md section 0.7) may fire one iteration earlier or later
    assert abs(res.iterations - len(ref_kept)) <= (1 if name == "terrestrial" else 0)
    assert abs(kept[-1] - ref_kept[-1]) <= 2
    if kept[-1] == ref_kept[-1]:
        np.testing.assert_allclose(res.residuals, g["residuals"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(res.rbp.get_parameter_attributes_as_list("estimated_uncertainty"),
                               g["sigma"], rtol=2e-2, equal_nan=True)
    np.testing.assert_allclose(np.asarray(res.X_mov_transformed)[:64], g["X_mov_t_head"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("name,k", NORMAL_CASES)
def test_normal_signs_follow_numpy_eig(gpu, name, k):
    """Default sign mode: the kernel walks LAPACK dgeev's algorithm, so eigenvector signs (and
    with them the float32 normals) equal the reference's np.linalg.eig output; the few
    exceptions are rounding-borderline deflations (DESIGN.md "normal sign")."""
    g = load_golden(name)
    X_fix, X_mov = load_pair(name)
    with _capi.Engine() as e:
        e.set_clouds(X_fix, X_mov)
        e.set_selected(g["idx_sel"])
        nx, ny, nz, pl = e.estimate_normals(k)
    n_gpu = np.column_stack((nx, ny, nz))
    ok = np.isfinite(g["planarity"]) & (g["planarity"] > 0.05)
    same_sign = np.sum(n_gpu.astype(np.float64) * g["normals"].astype(np.float64), axis=1) > 0
    frac = same_sign[ok].mean()
    exact = (n_gpu[ok] == g["normals"][ok]).all(axis=1).mean()
    print(f"{name}: sign agreement {frac:.4f}, bit-identical float32 normals {exact:.4f}")
    # webots (k = 40 on a regular lattice) and terrestrial (mm-quantised coordinates) have
    # equal-distance ties at the k-th neighbour in ~28 % / ~20 % of their neighbourhoods; cKDTree's
    # tie order is unspecified, ours is lowest index: another neighbour set, another (equally
    # valid) covariance
    assert frac > (0.9 if name == "terrestrial" else 0.985)
    assert exact > {"webots": 0.8, "terrestrial": 0.75}.get(name, 0.98)


@pytest.mark.parametrize("name", CONFIGS)
def test_full_run_standalone(gpu, name):
    """Everything on the GPU, normals included (dgeev-sign mode): H against the reference's."""
    g = load_golden(name)
    X_fix, X_mov = load_pair(name)
    res = sb.register(X_fix, X_mov, **g["kwargs"])
    dH = np.linalg.norm(res.H - g["H"])
    print(f"{name} stand-alone: |dH|_F = {dH:.3e}, iterations {res.iterations} vs {g['it_x'].shape[0]}")
    # dragon (graded: 1e-5), dragon_observed and bunny reproduce the reference far below its own
    # solver tolerance.  webots / multisensor inherit inputs on which the reference itself is not
    # uniquely defined (k-th-neighbour ties on a lattice; a 316-point radar cloud whose stop rule
    # flips on single correspondences): a handful of differing normals moves H at the 1e-3..1e-2
    # level there — with the reference's normals injected both reproduce it to 3e-10
    # (test_full_run_with_reference_normals).
    tol = {"dragon": 1e-9, "dragon_observed": 1e-8, "bunny": 1e-5, "webots": 1e-2, "multisensor": 5e-2,
           "airborne": 1e-5, "terrestrial": 1e-5}[name]
    assert dH < tol


def test_dragon_end_to_end_graded(gpu):
    """BASELINE.json north star: H within 1e-5 Frobenius of the Python reference on data/dragon,
    everything (normals included) computed on the GPU."""
    g = load_golden("dragon")
    X_fix, X_mov = load_pair("dragon")
    H, X_t, rbp, res = sb.simpleicp(X_fix, X_mov)
    dH = np.linalg.norm(H - g["H"])
    print(f"dragon stand-alone |dH|_F = {dH:.3e}")
    assert dH < 1e-5
    np.testing.assert_allclose(np.asarray(X_t).sum(axis=0), g["X_mov_t_sum"], rtol=1e-6)


def test_fused_loop_equals_stepwise(gpu):
    g = load_golden("bunny")
    X_fix, X_mov = load_pair("bunny")
    nrm = full_normals(g, X_fix.shape[0])
    a = sb.register(X_fix, X_mov, normals=nrm, **g["kwargs"])
    b = sb.register(X_fix, X_mov, normals=nrm, stepwise=True, **g["kwargs"])
    assert a.iterations == b.iterations
    np.testing.assert_allclose(a.H, b.H, rtol=0, atol=1e-12)
    np.testing.assert_allclose(a.residuals, b.residuals, rtol=0, atol=1e-12)


def test_predicted_histogram_select_is_used_and_exact(gpu):
    """From the second iteration on, median/MAD come from the predictor histogram the match
    kernel fills (one gather pass instead of ~6 radix passes).  Same keep masks as NumPy."""
    for name, K in (("dragon", 1000), ("dragon", 20000)):
        X_fix, X_mov = load_pair(name)
        with _capi.Engine() as e:
            res = sb.register(X_fix, X_mov, correspondences=K, engine=e)
            assert e.phase_times()[28] >= 1.0  # last iteration: predictor histogram (1) or barrier-free kernel (2)
            lsq = e.lsq_params(np.zeros(6), np.zeros(6), np.zeros(6), 1.0)
            p = e.run_params(0.3, 1.0, 100, lsq)
            x = np.array(res.rbp.get_parameter_attributes_as_list("estimated_value"))
            # replay: two queued iterations from the solution; the second uses the fast path
            e.iterate(p, x_in=x, want_record=True)
            rec = e.iterate(p, want_record=True)
            assert e.phase_times()[28] >= 1.0
            # the same state through the stage API (radix path) must give the same statistics
            H = O.rbp_to_H(np.array(rec.x))
            xs = x.copy()
            e.iterate(p, x_in=xs, want_record=True)
            rec_a = e.iterate(p, want_record=True)      # fast path
            e.iterate(p, x_in=xs, want_record=True)
            Hm = O.rbp_to_H(np.array(e.iterate(p, x_in=xs, want_record=True).x))  # state after 1 iteration
            idx, d = e.match(Hm)                         # resets the predictor -> radix path
            keep, n_kept, st = e.reject(0.3)
            # (Hm is rebuilt with NumPy's sin/cos, the device used CUDA's: distances agree to ~1e-16)
            assert n_kept == rec_a.n_kept
            np.testing.assert_allclose([st[0], st[1]], [rec_a.median, rec_a.mad], rtol=1e-9, atol=1e-18)
            S1 = res.normals[3].astype(np.float64) >= 0.3
            assert st[0] == np.median(d[S1]) and st[1] == np.median(np.abs(d[S1] - st[0]))


def test_last_iteration_read_back(gpu):
    """sicp_get_iteration hands back what the last iterate / time_stages iteration computed: the
    record iterate returned, the transform of its parameters, and the match and keep mask the
    stage API computes from the transform that iteration started from.  A call that changes the
    loop state makes it an error."""
    X_fix, X_mov = load_pair("dragon")
    with _capi.Engine() as e:
        e.set_clouds(X_fix, X_mov)
        e.set_selected(sb.pointcloud.subsample_indices(len(X_fix), 1000).astype(np.int64))
        e.estimate_normals(10)
        p = e.run_params(0.3, 1.0, 100, e.lsq_params(np.zeros(6), np.zeros(6), np.zeros(6), 1.0))
        with pytest.raises(_capi.SicpError, match="read back"):
            e.last_iteration()
        e.iterate(p, x_in=np.zeros(6), want_record=True)
        x_before = np.array(e.iterate(p, want_record=True).x)
        rec = e.iterate(p, want_record=True)
        got, T, idx, d, keep = e.last_iteration()
        for f in ("n_kept", "median", "mad", "mean_dist", "std_dist", "mean_res", "std_res"):
            assert getattr(got, f) == getattr(rec, f), f
        assert list(got.x) == list(rec.x)
        np.testing.assert_allclose(T, O.rbp_to_H(np.array(rec.x)), rtol=0, atol=1e-12)
        e.time_stages(p, 2, False, outer_only=True)
        got2, T2, *_ = e.last_iteration()
        np.testing.assert_allclose(T2, O.rbp_to_H(np.array(got2.x)), rtol=0, atol=1e-12)
        # (the host rebuilds H with NumPy's sin/cos: distances agree to ~1e-16, ties may pick another index)
        idx_m, d_m = e.match(O.rbp_to_H(x_before))
        same = idx == idx_m
        assert same.mean() > 0.99
        np.testing.assert_allclose(d[same], d_m[same], rtol=0, atol=1e-12)
        keep_m, n_kept, _ = e.reject(0.3)
        assert np.array_equal(keep, keep_m) and n_kept == got.n_kept
        with pytest.raises(_capi.SicpError, match="read back"):
            e.last_iteration()


def test_host_sync_batching_is_equivalent(gpu):
    """Queuing several iterations between host reads (device-side stop flag) changes nothing."""
    g = load_golden("dragon")
    X_fix, X_mov = load_pair("dragon")
    nrm = full_normals(g, X_fix.shape[0])
    a = sb.register(X_fix, X_mov, normals=nrm)
    with _capi.Engine() as e:
        e.set_option("host_sync_every", 4)
        b = sb.register(X_fix, X_mov, normals=nrm, engine=e)
    assert a.iterations == b.iterations
    assert np.array_equal(a.H, b.H)


def test_facade_side_effects(gpu):
    """SimpleICP / PointCloud drop-in behaviour: pc_mov is transformed in place, pc_fix gains
    float32 sparse normal columns and a thinned selection (reference: simpleicp.py:316,
    pointcloud.py:200-203)."""
    X_fix, X_mov = load_pair("bunny")
    pc_fix = sb.PointCloud(X_fix, columns=["x", "y", "z"])
    pc_mov = sb.PointCloud(X_mov, columns=["x", "y", "z"], copy=True)
    icp = sb.SimpleICP(verbose=False)
    icp.add_point_clouds(pc_fix, pc_mov)
    H, X_t, rbp, res = icp.run(max_overlap_distance=1)
    assert H.shape == (4, 4) and X_t.shape == X_mov.shape
    np.testing.assert_allclose(X_t, O.transform_by_H(X_mov, H), rtol=0, atol=1e-12)
    assert np.array_equal(pc_mov.X, X_t)
    assert pc_fix.num_selected_points == 1000
    assert str(pc_fix["planarity"].dtype) == "Sparse[float32, nan]"
    assert np.isfinite(pc_fix["nx"].to_numpy()[pc_fix.idx_selected]).all()
    assert isinstance(rbp, sb.RigidBodyParameters)
    np.testing.assert_allclose(rbp.H, H, rtol=0, atol=1e-15)
    assert len(res) > 6
    g = load_golden("bunny")
    assert np.linalg.norm(H - g["H"]) < 1e-4
    # second run reuses the stored normal columns (reference hook simpleicp.py:176-178)
    pc_mov2 = sb.PointCloud(X_mov, columns=["x", "y", "z"], copy=True)
    pc_fix.select_all_points()
    icp.add_point_clouds(pc_fix, pc_mov2)
    with pytest.raises(Exception):
        # stored normals only cover the previously selected points: NaN planarity elsewhere
        # drops every newly selected point -> fewer than 6 correspondences is possible but not
        # guaranteed; accept either outcome, the call must not crash the process
        icp.run(max_overlap_distance=1, min_planarity=2.0)


def test_errors(gpu):
    X_fix, X_mov = load_pair("bunny")
    with pytest.raises(sb.SimpleICPException, match="do not overlap within max_overlap_distance = 0.50000"):
        sb.simpleicp(X_fix, X_mov + 1000.0, max_overlap_distance=0.5)
    with pytest.raises(sb.SimpleICPException, match="Too few correspondences"):
        sb.simpleicp(X_fix, X_mov, min_planarity=2.0)
    with pytest.raises(_capi.SicpError):
        with _capi.Engine() as e:
            e.match(np.eye(4))  # before set_clouds


def test_transform(gpu):
    rng = np.random.default_rng(1)
    for n in (1, 2, 1001, 100000):
        X = rng.normal(size=(n, 3)) * 100
        H = O.rbp_to_H([0.3, -0.2, 0.5, 10.0, -20.0, 30.0])
        with _capi.Engine() as e:
            e.set_clouds(X[:1], X)
            Y = e.transform(H)
            Z = np.empty_like(X)
            np.testing.assert_allclose(Y, O.transform_by_H(X, H), rtol=0, atol=1e-12)
            # round trip: transform of the transformed cloud by the inverse
            e.set_clouds(X[:1], Y)
            Z = e.transform(np.linalg.inv(H))
        np.testing.assert_allclose(Z, X, rtol=0, atol=1e-11)


def test_large_k_multi_block_path(gpu):
    """K > 4096 switches the reject/solve kernel to its cooperative multi-block form; lock-step
    against the oracle on dragon with 20 000 correspondences (normals from the oracle)."""
    X_fix, X_mov = load_pair("dragon")
    tr = O.Trace()
    H_o, _, x_o, sig_o, res_o = O.simpleicp(X_fix, X_mov, correspondences=20000, trace=tr)
    nrm = [np.full(X_fix.shape[0], np.nan, dtype=np.float32) for _ in range(4)]
    for a in range(3):
        nrm[a][tr.idx_sel] = tr.normals[:, a]
    nrm[3][tr.idx_sel] = tr.planarity
    with _capi.Engine() as e:
        e.set_clouds(X_fix, X_mov)
        e.set_selected(tr.idx_sel)
        e.set_normals(tr.normals[:, 0], tr.normals[:, 1], tr.normals[:, 2], tr.planarity)
        for it in tr.iterations:
            idx, d = e.match(it.H_in)
            keep, n_kept, st = e.reject(0.3)
            keep_o, med_o, mad_o = O.reject(d, tr.planarity, 0.3)
            assert np.array_equal(keep, keep_o)
            assert st[0] == med_o and st[1] == mad_o
            if np.array_equal(idx, it.pc2_idx):
                assert np.array_equal(keep, it.keep)
    res = sb.register(X_fix, X_mov, correspondences=20000, normals=tuple(nrm))
    print(f"K=20000: |dH|_F = {np.linalg.norm(res.H - H_o):.3e}, it {res.iterations} vs {len(tr.iterations)}")
    assert np.linalg.norm(res.H - H_o) < 1e-6
    # the stop rule thresholds the relative change of a mean that is ~0 (SURVEY.md §0.7): the
    # iteration count may move by a few, the fixed point may not
    assert abs(res.iterations - len(tr.iterations)) <= 4


def test_full_size_properties(gpu):
    """BASELINE.json C3 size (1M <-> 1M, K = 100 000), size-independent properties:
    recovers the known transform, grid and brute-force engines agree exactly, the converged
    state is a fixed point, median/MAD equal NumPy's on the device distances."""
    X_fix, X_mov, H_true = O.c3_pair(1_000_000)
    with _capi.Engine() as e:
        res = sb.register(X_fix, X_mov, correspondences=100_000, engine=e)
        assert res.converged and res.iterations < 30
        assert np.linalg.norm(res.H - H_true) < 2e-2
        # the grid engine (all 100k queries) against the TMA brute-force engine on a sample
        idx_g, d_g = e.match(res.H)
        keep, n_kept, st = e.reject(0.3)
        S1 = res.normals[3].astype(np.float64) >= 0.3
        assert st[0] == np.median(d_g[S1])
        assert st[1] == np.median(np.abs(d_g[S1] - st[0]))
        assert np.array_equal(keep, S1 & (np.abs(d_g - st[0]) <= 3 * st[1]))
    sample = res.idx_selected[:: 100_000 // 2048][:2048]
    with _capi.Engine() as e2:
        e2.set_option("nn_engine", _capi.NN_BRUTE)
        e2.set_clouds(X_fix, X_mov)
        e2.set_selected(sample)
        pos = np.searchsorted(res.idx_selected, sample)
        e2.set_normals(*[a[pos] for a in res.normals])
        idx_b, d_b = e2.match(res.H)
    assert np.array_equal(idx_b, idx_g[pos])
    np.testing.assert_allclose(d_b, d_g[pos], rtol=0, atol=1e-13)
    # fixed point: restarting from the solution changes nothing beyond the solver tolerance
    x = np.array(res.rbp.get_parameter_attributes_as_list("estimated_value"))
    obs_deg = x.copy()
    obs_deg[:3] *= 180 / np.pi
    res2 = sb.register(X_fix, X_mov, correspondences=100_000, rbp_observed_values=tuple(obs_deg),
                       normals=None)
    assert res2.iterations <= 6 and np.linalg.norm(res2.H - res.H) < 2e-4


def test_cli_matches_reference_flags(gpu, tmp_path):
    """sicp_cli: the reference CLIs' flag set (c++/src/simpleicp-cli.cpp:15-35) on .xyz files;
    prints the reference's table, H and the `Finished in` line scripts/benchmark.sh greps."""
    import re
    import subprocess

    from conftest import REPO

    cli = REPO / "simpleicp_b200" / "sicp_cli"
    assert cli.exists()
    for name, extra in (("dragon", []), ("bunny", ["-o", "1"])):
        g = load_golden(name)
        X_fix, X_mov = load_pair(name)
        f1, f2, fo = tmp_path / f"{name}1.xyz", tmp_path / f"{name}2.xyz", tmp_path / f"{name}_out.xyz"
        sb.write_xyz(f1, X_fix, decimals=4, header=False)
        sb.write_xyz(f2, X_mov, decimals=4, header=True)
        r = subprocess.run([str(cli), "-f", str(f1), "-m", str(f2), "-c", "1000", "-n", "10", "-p", "0.3",
                            "-i", "1", "-x", "100", "--out", str(fo)] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        rows = re.findall(r"^\[\s*(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\]$", r.stdout, re.M)
        H = np.array(rows, dtype=float)
        assert H.shape == (4, 4)
        assert np.abs(H - g["H"]).max() < (2e-6 if name == "dragon" else 2e-5)
        assert re.search(r"Finished in \d+\.\d{3} seconds!", r.stdout)
        assert "Iteration | correspondences" in r.stdout and "orig:0" in r.stdout
        X_t = sb.read_xyz(fo)
        np.testing.assert_allclose(X_t, O.transform_by_H(X_mov, g["H"]), atol=2e-4)
    bad = subprocess.run([str(cli), "-f", str(tmp_path / "nope.xyz"), "-m", str(f2)], capture_output=True, text=True)
    assert bad.returncode == 1 and "Caught exception" in bad.stderr


def test_batch_of_pairs_matches_individual_runs(gpu):
    """simpleicp_batch (concurrent engines on separate streams) == one register() per pair; the
    slab tiler produces independent registrations that all recover the common transform."""
    pairs = []
    for i in range(6):
        Xf = O.surface(40_000, 10_000 + 2 * i, extent=30.0)
        Ht = O.rbp_to_H([0.004 * (i + 1), -0.003, 0.005, 0.05, -0.03 * i, 0.02])
        Xm = O.transform_by_H(O.surface(40_000, 10_001 + 2 * i, extent=30.0), np.linalg.inv(Ht))
        pairs.append((Xf, Xm))
    table = sb.simpleicp_batch(pairs, concurrency=3, engine="pool")
    assert table.shape == (6, 20)
    table_b = sb.simpleicp_batch(pairs)  # batched engine
    np.testing.assert_allclose(table_b[:, :16], table[:, :16], rtol=0, atol=1e-12)
    assert np.array_equal(table_b[:, 16:18], table[:, 16:18])
    for i, (Xf, Xm) in enumerate(pairs):
        r = sb.register(Xf, Xm)
        np.testing.assert_allclose(table[i, :16].reshape(4, 4), r.H, rtol=0, atol=1e-12)
        assert table[i, 16] == r.iterations and table[i, 17] == r.records[-1]["n_kept"]
    X_fix, X_mov, H_true = O.c3_pair(200_000)
    slabs = sb.tile_slabs(X_fix, X_mov, 4, overlap=5.0)
    tab = sb.simpleicp_batch(slabs, correspondences=2000)
    for i in range(4):
        assert np.linalg.norm(tab[i, :16].reshape(4, 4) - H_true) < 5e-2


@pytest.mark.parametrize("K", [4096, 4097])
def test_kernel_switch_boundary(gpu, K):
    """K = 4096 runs the single-block reject/solve kernel, 4097 the cooperative one: both must
    reproduce the oracle (its normals injected) including iteration and kept counts."""
    X_fix, X_mov = load_pair("dragon")
    tr = O.Trace()
    H_o, _, x_o, sig_o, res_o = O.simpleicp(X_fix, X_mov, correspondences=K, trace=tr)
    nrm = [np.full(X_fix.shape[0], np.nan, dtype=np.float32) for _ in range(4)]
    for a in range(3):
        nrm[a][tr.idx_sel] = tr.normals[:, a]
    nrm[3][tr.idx_sel] = tr.planarity
    res = sb.register(X_fix, X_mov, correspondences=K, normals=tuple(nrm))
    assert np.array_equal(res.idx_selected, tr.idx_sel)
    assert np.linalg.norm(res.H - H_o) < 1e-6
    assert abs(res.iterations - len(tr.iterations)) <= 3
    if res.iterations == len(tr.iterations):
        assert abs(res.records[-1]["n_kept"] - int(tr.iterations[-1].keep.sum())) <= 2


def test_small_and_ragged_inputs(gpu):
    """Tiny clouds, more requested correspondences than points, one-point movable cloud."""
    rng = np.random.default_rng(3)
    # 200-point patches of a curved surface, K larger than the cloud -> every point selected
    def patch(n, seed):
        r = np.random.default_rng(seed)
        x, y = r.uniform(0, 1, n), r.uniform(0, 1, n)
        return np.column_stack((x, y, 0.2 * np.sin(3 * x) * np.cos(2 * y) + 0.05 * x * y))
    Xf = patch(200, 1)
    Ht = O.rbp_to_H([0.01, -0.02, 0.015, 0.01, -0.005, 0.008])
    Xm = O.transform_by_H(patch(300, 2), np.linalg.inv(Ht))
    H_o, Xt_o, x_o, sig_o, res_o = O.simpleicp(Xf, Xm, correspondences=5000, neighbors=8)
    res = sb.register(Xf, Xm, correspondences=5000, neighbors=8)
    assert res.idx_selected.size == 200
    assert np.linalg.norm(res.H - H_o) < 1e-3  # normals: handful of borderline-sign cases on 200 points
    # neighbours = number of points (every neighbourhood is the whole cloud)
    with _capi.Engine() as e:
        e.set_clouds(Xf[:12], Xm)
        e.set_selected(None)
        nx, ny, nz, pl = e.estimate_normals(12)
        assert np.isfinite(nx).all() and np.allclose(np.abs(nx), np.abs(nx[0]), atol=1e-6)
        with pytest.raises(_capi.SicpError, match="neighbors"):
            e.estimate_normals(13)
        with pytest.raises(_capi.SicpError):
            e.estimate_normals(1)
    # a single movable point: every query matches it; too few *distinct* constraints is the
    # solver's problem, not a crash
    with _capi.Engine() as e:
        e.set_clouds(Xf, Xm[:1])
        e.set_selected(None)
        e.estimate_normals(8)
        idx, d = e.match(np.eye(4))
        assert (idx == 0).all() and np.isfinite(d).all()
    # empty clouds are rejected at the boundary
    with _capi.Engine() as e:
        with pytest.raises(_capi.SicpError):
            e.set_clouds(np.zeros((0, 3)), Xm)
        with pytest.raises(ValueError):
            e.set_clouds(np.zeros((5, 2)), Xm)


def test_degenerate_geometry_terminates(gpu):
    """Two exactly parallel planes leave three of the six parameters unobservable: the
    reference's trust-region solver returns *some* minimiser; ours must terminate with either a
    finite result or a clean exception, never hang or return NaN silently."""
    g = np.stack(np.meshgrid(np.arange(40.0), np.arange(40.0)), -1).reshape(-1, 2)
    Xf = np.column_stack((g, np.zeros(len(g))))
    Xm = np.column_stack((g + 0.25, np.full(len(g), 0.1)))
    try:
        res = sb.register(Xf, Xm, correspondences=500, max_iterations=5)
        assert np.isfinite(res.H).all()
        assert abs(res.H[2, 3] + 0.1) < 1e-6  # the observable part: the plane offset
    except sb.SimpleICPException as e:
        assert "singular" in str(e).lower() or "correspondences" in str(e).lower()


def test_single_iteration_and_fixed_parameters(gpu):
    X_fix, X_mov = load_pair("dragon")
    res = sb.register(X_fix, X_mov, max_iterations=1)
    assert res.iterations == 1 and not res.converged
    o = O.simpleicp(X_fix, X_mov, max_iterations=1, normals=(np.column_stack(res.normals[:3]), res.normals[3]))
    assert np.linalg.norm(res.H - o[0]) < 1e-5
    # only tz free: x stays at the observed values for the five fixed parameters
    w = (np.inf,) * 5 + (0.0,)
    obs = (0.5, -0.25, 1.0, 0.01, -0.02, 0.0)
    res = sb.register(X_fix, X_mov, rbp_observed_values=obs, rbp_observation_weights=w, max_iterations=3)
    x = res.rbp.get_parameter_attributes_as_list("estimated_value")
    np.testing.assert_allclose(x[:3], np.deg2rad(obs[:3]), rtol=0, atol=0)
    assert x[3] == obs[3] and x[4] == obs[4] and x[5] != 0.0
    sig = res.rbp.get_parameter_attributes_as_list("estimated_uncertainty")
    assert np.isnan(sig[:5]).all() and np.isfinite(sig[5])
    o = O.simpleicp(X_fix, X_mov, rbp_observed_values=obs, rbp_observation_weights=w, max_iterations=3,
                    normals=(np.column_stack(res.normals[:3]), res.normals[3]))
    assert abs(x[5] - o[2][5]) < 1e-6


@pytest.mark.parametrize("name,kw", [("dragon", {}), ("bunny", {"max_overlap_distance": 1.0}),
                                     ("multisensor", {"correspondences": 5000})])
def test_fused_register_equals_stage_by_stage(gpu, name, kw):
    """sicp_register (one call, movable upload overlapped with the fixed-side work) against the
    stage-by-stage sequence it is defined to equal: bit-identical results."""
    X_fix, X_mov = load_pair(name)
    eng = _capi.Engine()
    try:
        a = sb.register(X_fix, X_mov, engine=eng, want_normals=True, **kw)    # staged
        b = sb.register(X_fix, X_mov, engine=eng, want_normals=False, **kw)   # fused
        assert b.normals is None and a.normals is not None
        assert np.array_equal(a.H, b.H) and a.iterations == b.iterations and a.converged == b.converged
        assert np.array_equal(a.residuals, b.residuals)
        assert np.array_equal(np.asarray(a.X_mov_transformed), np.asarray(b.X_mov_transformed))
        assert np.array_equal(a.idx_selected, b.idx_selected)
        for ra, rb in zip(a.records, b.records):
            assert ra["n_kept"] == rb["n_kept"] and ra["mean_res"] == rb["mean_res"] and ra["std_res"] == rb["std_res"]
        # the stage-by-stage API stays usable on the state the fused call left behind
        assert eng.K == a.idx_selected.size
        nn_idx, d = eng.match(a.H)
        assert nn_idx.shape == (eng.K,)
    finally:
        eng.close()
    with pytest.raises(sb.SimpleICPException, match="do not overlap"):
        sb.simpleicp(X_fix, X_mov + 1e5, max_overlap_distance=1.0)


def test_select_n_points_on_device(gpu):
    """sicp_select_n_points = PointCloud.select_n_points (pointcloud.py:121-147): numpy linspace
    arithmetic and round-half-even; the linearised variants round half away from zero."""
    rng = np.random.default_rng(5)
    X = rng.normal(size=(5000, 3))
    with _capi.Engine() as e:
        e.set_clouds(X, X + 0.01)
        for m_idx, n in ((None, 1000), (None, 1), (None, 4999), (None, 5000), (None, 7000), (np.arange(3, 4000, 3), 77)):
            e.set_selected(m_idx)
            base = np.arange(5000) if m_idx is None else m_idx
            got = e.select_n_points(n)
            want = base if n >= base.size else base[sb.pointcloud.subsample_indices(base.size, n)]
            assert np.array_equal(got, want), (n, got[:5], want[:5])
            assert e.K == want.size
        # 10 points -> 5: linspace = 0 2.25 4.5 6.75 9; rint -> 0 2 4 7 9, C round() -> 0 2 5 7 9
        e.set_selected(np.arange(10))
        assert e.select_n_points(5).tolist() == [0, 2, 4, 7, 9]
        e.set_option("variant", 1)
        e.set_selected(np.arange(10))
        assert e.select_n_points(5).tolist() == [0, 2, 5, 7, 9]


def test_c3_converged_full_run_vs_oracle(gpu):
    """BASELINE.json configs[2] (1M <-> 1M, K = 100 000) run to convergence against the oracle:
    (a) with the oracle's normals injected — same iteration count, same kept counts, H to 1e-9;
    (b) stand-alone, normals from the GPU's dgeev walk — fraction of identical normal signs at
        K = 100 000 and the resulting H."""
    X_fix, X_mov, H_true = O.c3_pair(1_000_000)
    tr = O.Trace()
    H_o, _, x_o, sig_o, res_o = O.simpleicp(X_fix, X_mov, correspondences=100_000, trace=tr)
    kept_o = [int(it.keep.sum()) for it in tr.iterations]
    nrm = [np.full(X_fix.shape[0], np.nan, dtype=np.float32) for _ in range(4)]
    for a in range(3):
        nrm[a][tr.idx_sel] = tr.normals[:, a]
    nrm[3][tr.idx_sel] = tr.planarity
    with _capi.Engine() as e:
        a = sb.register(X_fix, X_mov, correspondences=100_000, normals=tuple(nrm), engine=e)
        kept_a = [r["n_kept"] for r in a.records]
        dHa = np.linalg.norm(a.H - H_o)
        print(f"C3 injected: |dH|_F = {dHa:.3e}, iterations {a.iterations} vs {len(kept_o)}, kept {kept_a[-2:]} vs {kept_o[-2:]}")
        assert a.iterations == len(kept_o)
        assert kept_a == kept_o
        assert dHa < 1e-9
        np.testing.assert_allclose(a.residuals, res_o, rtol=0, atol=1e-9)
        b = sb.register(X_fix, X_mov, correspondences=100_000, engine=e)
    n_gpu = np.column_stack(b.normals[:3]).astype(np.float64)
    ok = np.isfinite(tr.planarity) & (tr.planarity > 0.05)
    same_sign = (np.sum(n_gpu * tr.normals.astype(np.float64), axis=1) > 0)[ok].mean()
    exact = (np.column_stack(b.normals[:3])[ok] == tr.normals[ok]).all(axis=1).mean()
    dHb = np.linalg.norm(b.H - H_o)
    print(f"C3 stand-alone: sign agreement {same_sign:.5f}, bit-identical normals {exact:.5f}, "
          f"|dH|_F = {dHb:.3e}, iterations {b.iterations} vs {len(kept_o)}")
    assert same_sign > 0.995
    assert dHb < 1e-5  # the north-star bar, at the 1M/100k size


@pytest.mark.parametrize("name,kw", [("dragon", {}), ("bunny", {"max_overlap_distance": 1.0}),
                                     ("dragon", {"correspondences": 20000}),
                                     ("airborne", {"correspondences": 50000})])
def test_barrier_free_kernel_equals_cooperative_kernel(gpu, name, kw):
    """Iterations after the first run reject + solve in k_rs_fused (no grid barrier, residual
    statistics from the moment sums); option fused=0 forces the cooperative kernel everywhere.
    Same kept sets and iteration counts, H to 1e-11 (the sums are taken in another order)."""
    X_fix, X_mov = load_pair(name)
    with _capi.Engine() as e:
        a = sb.register(X_fix, X_mov, engine=e, **kw)
        ta = e.timings()
        e.set_option("fused", 0)
        b = sb.register(X_fix, X_mov, engine=e, **kw)
        tb = e.timings()
    print(f"{name} {kw}: fused iterations {ta['fused_iterations']} of {a.iterations}, re-run {ta['rerun_iterations']}, "
          f"|dH| = {np.linalg.norm(a.H - b.H):.2e}")
    assert tb["fused_iterations"] == 0
    if kw.get("correspondences", 1000) <= 4096:
        # one block owns the problem: every iteration (the first included) runs in k_rs_fused
        assert ta["fused_iterations"] == a.iterations and ta["rerun_iterations"] == 0
    else:
        assert ta["fused_iterations"] + ta["rerun_iterations"] == a.iterations - 1
        assert ta["fused_iterations"] >= (a.iterations - 1) // 2
    assert a.iterations == b.iterations and a.converged == b.converged
    assert [r["n_kept"] for r in a.records] == [r["n_kept"] for r in b.records]
    for ra, rb in zip(a.records, b.records):
        # exact order statistics of distances that differ by the rounding of the two summation orders
        # (1e-13 absolute: rounding of coordinates of size 1 .. 1000 through two transforms)
        np.testing.assert_allclose([ra["median"], ra["mad"]], [rb["median"], rb["mad"]], rtol=1e-9, atol=1e-13)
        # statistics from the re-centred moment sums against the direct residual pass
        np.testing.assert_allclose(ra["std_res"], rb["std_res"], rtol=1e-9, atol=1e-13)
        np.testing.assert_allclose(ra["mean_res"], rb["mean_res"], rtol=1e-7, atol=1e-13)
    np.testing.assert_allclose(a.H, b.H, rtol=0, atol=1e-11)
    np.testing.assert_allclose(a.residuals, b.residuals, rtol=0, atol=1e-11)
    np.testing.assert_allclose(a.rbp.get_parameter_attributes_as_list("estimated_uncertainty"),
                               b.rbp.get_parameter_attributes_as_list("estimated_uncertainty"), rtol=1e-6)
    # the last record carries the exact two-pass statistics of the returned residual vector
    np.testing.assert_allclose(a.records[-1]["mean_res"], a.residuals.mean(), rtol=0, atol=1e-15)
    np.testing.assert_allclose(a.records[-1]["std_res"], a.residuals.std(), rtol=1e-12)


def _surface_pairs(n_pairs, n_pts, seed0=10_000):
    pairs = []
    rng = np.random.default_rng(99)
    for i in range(n_pairs):
        n = n_pts if isinstance(n_pts, int) else n_pts[i]
        Xf = O.surface(n, seed0 + 2 * i, extent=30.0)
        x = np.concatenate((np.deg2rad(rng.uniform(-1, 1, 3)), rng.uniform(-0.2, 0.2, 3)))
        Xm = O.transform_by_H(O.surface(n + 17 * i, seed0 + 1 + 2 * i, extent=30.0), np.linalg.inv(O.rbp_to_H(x)))
        pairs.append((Xf, Xm))
    return pairs


def test_batched_engine_equals_per_pair_registration(gpu):
    """sicp_register_batch (one launch set per stage for the whole batch, a block per pair for
    reject + solve, per-pair stop flags) against sicp_register pair by pair: the per-pair kernels
    are the same device code, so iteration counts, kept counts and H are IDENTICAL."""
    pairs = _surface_pairs(9, [40_000, 25_000, 60_000, 40_000, 3_000, 40_000, 12_345, 40_000, 80_000])
    with _capi.Engine() as e:
        lsq = e.lsq_params(np.zeros(6), np.zeros(6), np.zeros(6), 1.0)
        params = e.run_params(0.3, 1.0, 100, lsq)
        res = e.register_batch(pairs, 1000, 10, params)
        tm = e.timings()
        for i, (Xf, Xm) in enumerate(pairs):
            r = sb.register(Xf, Xm, engine=e, want_normals=False)
            b = res[i]
            assert b.status == 0
            H = np.array(b.H).reshape(4, 4)
            print(f"pair {i}: it {b.iterations} vs {r.iterations}, kept {b.n_kept} vs {r.records[-1]['n_kept']}, |dH| {np.linalg.norm(H - r.H):.2e}")
            assert b.iterations == r.iterations and bool(b.converged) == r.converged
            assert b.n_kept == r.records[-1]["n_kept"]
            np.testing.assert_allclose(H, r.H, rtol=0, atol=1e-12)
            np.testing.assert_allclose(np.array(b.x), r.rbp.get_parameter_attributes_as_list("estimated_value"), rtol=0, atol=1e-12)
            np.testing.assert_allclose(np.array(b.sigma), r.rbp.get_parameter_attributes_as_list("estimated_uncertainty"), rtol=1e-9)
            np.testing.assert_allclose([b.mean_res, b.std_res], [r.residuals.mean(), r.residuals.std()], rtol=1e-9, atol=1e-15)
        # other keyword arguments travel too: observed / fixed parameters, auto weight, fewer neighbours
        lsq2 = e.lsq_params(np.array([0.001, 0, 0, 0, 0, 0.01]), np.array([0.001, 0, 0, 0, 0, 0.01]),
                            np.array([np.inf, 0, 0, 5.0, 0, 0]), None)
        params2 = e.run_params(0.2, 0.5, 30, lsq2)
        res2 = e.register_batch(pairs[:3], 700, 8, params2)
        for i, (Xf, Xm) in enumerate(pairs[:3]):
            r = sb.register(Xf, Xm, engine=e, want_normals=False, correspondences=700, neighbors=8, min_planarity=0.2,
                            min_change=0.5, max_iterations=30, distance_weights=None,
                            rbp_observed_values=(np.rad2deg(0.001), 0, 0, 0, 0, 0.01),
                            rbp_observation_weights=(np.inf, 0, 0, 5.0, 0, 0))
            assert res2[i].status == 0 and res2[i].iterations == r.iterations
            np.testing.assert_allclose(np.array(res2[i].H).reshape(4, 4), r.H, rtol=0, atol=1e-12)
            assert res2[i].x[0] == 0.001


def test_batched_engine_per_pair_status_and_front_end(gpu):
    """A pair without enough correspondences fails alone; simpleicp_batch reports it after the
    gather; bad arguments are rejected for the whole call."""
    pairs = _surface_pairs(4, 30_000)
    t = np.sort(np.random.default_rng(1).uniform(0, 30, 5000))
    line = np.column_stack((t, 2 * t, 3 * t))
    pairs[2] = (line, line + 0.01)  # points on a line: planarity ~ 0 -> every correspondence rejected
    with _capi.Engine() as e:
        lsq = e.lsq_params(np.zeros(6), np.zeros(6), np.zeros(6), 1.0)
        res = e.register_batch(pairs, 1000, 10, e.run_params(0.3, 1.0, 50, lsq))
        assert [r.status for r in res] == [0, 0, _capi.SICP_ERR_TOO_FEW_CORR, 0]
        with pytest.raises(_capi.SicpError, match="4096"):
            e.register_batch(pairs, 5000, 10, e.run_params(0.3, 1.0, 50, lsq))
    with pytest.raises(sb.batch.BatchError) as ei:
        sb.simpleicp_batch(pairs, max_iterations=50)
    assert ei.value.failed.tolist() == [2] and ei.value.table.shape == (4, 20)
    table = sb.simpleicp_batch(pairs, max_iterations=50, on_error="nan")
    assert np.isnan(table[2, :16]).all() and table[2, 16] == -_capi.SICP_ERR_TOO_FEW_CORR
    # the batched front end equals the per-pair engines
    pool = sb.simpleicp_batch(pairs, max_iterations=50, on_error="nan", engine="pool")
    ok = [0, 1, 3]
    np.testing.assert_allclose(table[ok, :16], pool[ok, :16], rtol=0, atol=1e-12)
    assert np.array_equal(table[ok, 16:18], pool[ok, 16:18])


def test_barrier_free_kernel_many_tiles_per_block(gpu):
    """K = 300 000 > 148 x 768: every block of k_rs_fused streams several TMA-staged tiles and the
    per-bin store runs at its larger capacity; results against the cooperative kernel."""
    X_fix, X_mov, H_true = O.c3_pair(400_000)
    with _capi.Engine() as e:
        a = sb.register(X_fix, X_mov, correspondences=300_000, engine=e, want_normals=False)
        ta = e.timings()
        e.set_option("fused", 0)
        b = sb.register(X_fix, X_mov, correspondences=300_000, engine=e, want_normals=False)
    print(f"K=300000: fused {ta['fused_iterations']} of {a.iterations}, re-run {ta['rerun_iterations']}, |dH| {np.linalg.norm(a.H - b.H):.2e}")
    assert ta["fused_iterations"] >= a.iterations - 2
    assert a.iterations == b.iterations and [r["n_kept"] for r in a.records] == [r["n_kept"] for r in b.records]
    np.testing.assert_allclose(a.H, b.H, rtol=0, atol=1e-11)
    np.testing.assert_allclose(a.residuals, b.residuals, rtol=0, atol=1e-11)
    assert np.linalg.norm(a.H - H_true) < 2e-2


# ---- movable-side attributes: pc_mov with normal columns (corrpts.py:157-162) and the rejection
# ---- by the angle between normals the reference declares but leaves unimplemented (:190-193)
def _mov_attr(g):
    return tuple(np.ascontiguousarray(g["mov_normals"][:, a]) for a in range(3)) + (g["mov_planarity"],)


def test_movable_side_planarity_lockstep(gpu):
    """Reference run with pc_mov.estimate_normals() called first (golden dragon_movnormals,
    captured from the unmodified reference): the keep mask of the first iteration is bit-identical
    stage by stage, and the whole run has the reference's iteration and kept counts and its H."""
    g = load_golden("dragon_movnormals")
    X_fix, X_mov = load_pair("dragon_movnormals")
    nrm = full_normals(g, X_fix.shape[0])
    with _capi.Engine() as e:
        e.set_clouds(X_fix, X_mov)
        e.set_mov_normals(*_mov_attr(g))
        e.set_selected(g["idx_sel"])
        e.set_normals(*[a[g["idx_sel"]] for a in nrm])
        idx_nn, d = e.match(np.eye(4))
        n_ties = assert_same_nn(idx_nn, g["it_pc2_idx"][0], X_fix[g["idx_sel"]], X_mov, "dragon_movnormals it 0")
        keep, n_kept, _ = e.reject(0.3)
        # the kernel against the restated branch on ITS neighbours (an exact tie may pick another,
        # equally near movable point with another planarity) ...
        keep_o, _, _ = O.reject(d, g["planarity"], 0.3, g["mov_planarity"][idx_nn])
        assert np.array_equal(keep, keep_o) and n_kept == int(keep_o.sum())
        # ... and against the reference's own mask wherever the neighbours are the reference's
        same = idx_nn == g["it_pc2_idx"][0]
        print(f"movable planarity: {n_ties} tie picks differ, kept {n_kept} vs {int(g['it_keep'][0].sum())}")
        if n_ties == 0:
            assert np.array_equal(keep, g["it_keep"][0])
        else:
            assert abs(n_kept - int(g["it_keep"][0].sum())) <= 2 * n_ties
            assert (keep[same] != g["it_keep"][0][same]).sum() <= 4 * n_ties  # median/MAD moved by the swapped members
        # clearing the attributes gives the plain dragon mask again
        e.set_mov_normals(None, None, None, None)
        e.match(np.eye(4))
        keep0 = e.reject(0.3)[0]
        assert abs(int(keep0.sum()) - int(load_golden("dragon")["it_keep"][0].sum())) <= 2
    for fused in (1, 0):
        with _capi.Engine() as e:
            e.set_option("fused", fused)
            res = sb.register(X_fix, X_mov, normals=nrm, mov_normals=_mov_attr(g), engine=e)
        kept = [r["n_kept"] for r in res.records]
        ref_kept = [int(k.sum()) for k in g["it_keep"]]
        dH = np.linalg.norm(res.H - g["H"])
        print(f"movable planarity (fused={fused}): |dH|_F = {dH:.3e}, kept {kept} vs {ref_kept}")
        assert res.iterations == len(ref_kept)
        assert max(abs(a - b) for a, b in zip(kept, ref_kept)) <= 3
        assert dH < 1e-6
        if kept[-1] == ref_kept[-1]:
            np.testing.assert_allclose(res.residuals, g["residuals"], rtol=0, atol=1e-6)


def test_movable_side_normals_through_the_class(gpu):
    """The reference's user-level route: pc_mov.estimate_normals(k) then SimpleICP.run — all
    100 000 movable normals estimated on the GPU (compared with the reference's), then used."""
    g = load_golden("dragon_movnormals")
    X_fix, X_mov = load_pair("dragon_movnormals")
    pc_fix, pc_mov = sb.PointCloud(X_fix, columns=["x", "y", "z"]), sb.PointCloud(X_mov, columns=["x", "y", "z"])
    pc_mov.estimate_normals(10)
    pl = pc_mov["planarity"].to_numpy().astype(np.float32)
    n_gpu = np.column_stack([pc_mov[c].to_numpy() for c in ("nx", "ny", "nz")]).astype(np.float32)
    np.testing.assert_allclose(pl, g["mov_planarity"], rtol=0, atol=2e-5)
    dots = np.abs(np.sum(n_gpu.astype(np.float64) * g["mov_normals"].astype(np.float64), axis=1))
    ok = g["mov_planarity"] > 0.05
    assert dots[ok].min() > 1 - 1e-6
    exact = (n_gpu == g["mov_normals"]).all(axis=1).mean()
    print(f"movable normals: bit-identical float32 rows {exact:.4f}, planarity max diff "
          f"{np.abs(pl - g['mov_planarity']).max():.2e}")
    assert exact > 0.99
    icp = sb.SimpleICP(verbose=False)
    icp.add_point_clouds(pc_fix, pc_mov)
    H, X_t, rbp, res = icp.run()
    dH = np.linalg.norm(H - g["H"])
    print(f"class run with movable normals: |dH|_F = {dH:.3e}, {len(res)} residuals vs {len(g['residuals'])}")
    assert dH < 1e-5
    assert abs(len(res) - len(g["residuals"])) <= 2
    # without the movable columns the same clouds keep more correspondences
    H0, _, _, res0 = sb.simpleicp(X_fix, X_mov)
    assert len(res0) >= len(res)


@pytest.mark.parametrize("max_angle", [5.0, 20.0, 90.0])
def test_angle_between_normals_rejection(gpu, max_angle):
    """The step the reference only declares: against the oracle's definition (applied after the
    distance rejection, |n_fix . R n_mov| >= cos(max angle)); 90 degrees is the plain movable-
    planarity run."""
    g = load_golden("dragon_movnormals")
    X_fix, X_mov = load_pair("dragon_movnormals")
    nrm = full_normals(g, X_fix.shape[0])
    tr = O.Trace()
    H_o, _, x_o, sig_o, res_o = O.simpleicp(
        X_fix, X_mov, normals=(g["normals"], g["planarity"]), mov_normals=(g["mov_normals"], g["mov_planarity"]),
        max_angle_between_normals=max_angle, trace=tr)
    with _capi.Engine() as e:
        # first iteration stage by stage: mask equality
        e.set_clouds(X_fix, X_mov)
        e.set_mov_normals(*_mov_attr(g), max_angle_deg=max_angle)
        e.set_selected(g["idx_sel"])
        e.set_normals(*[a[g["idx_sel"]] for a in nrm])
        e.match(np.eye(4))
        keep = e.reject(0.3)[0]
        assert np.array_equal(keep.astype(bool), tr.iterations[0].keep)
        res = sb.register(X_fix, X_mov, normals=nrm, mov_normals=_mov_attr(g),
                          max_angle_between_normals=max_angle, engine=e)
    kept = [r["n_kept"] for r in res.records]
    ref_kept = [int(it.keep.sum()) for it in tr.iterations]
    dH = np.linalg.norm(res.H - H_o)
    print(f"angle <= {max_angle}: |dH|_F = {dH:.3e}, kept {kept} vs {ref_kept}")
    assert kept == ref_kept
    assert dH < 1e-9
    if max_angle == 90.0:
        assert kept == [int(k.sum()) for k in g["it_keep"]]
    else:
        assert kept[0] < int(g["it_keep"][0].sum())
    with pytest.raises(sb.SimpleICPException, match="needs the normals of the movable"):
        sb.simpleicp(X_fix, X_mov, max_angle_between_normals=10.0)
