"""The batched engine with the partial-overlap filter (max_overlap_distance, simpleicp.py:150-170):
per pair the same kept set, selection, normals and loop as sicp_register with the filter, so the
same device code gives the same iterations, kept counts and H; a pair whose clouds do not overlap
fails alone with SICP_ERR_NO_OVERLAP."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from conftest import REPO, load_golden, load_pair

import simpleicp_b200 as sb
from simpleicp_b200 import _capi, synthetic
from simpleicp_b200.simpleicp import _observed_in_radians

D = 1.0  # max_overlap_distance of the synthetic pairs


def _patch_pair(n, shift, seed):
    """A 30 x 30 m patch of the synthetic surface and a second sample of it displaced by `shift`
    metres in x (about (30 - shift) / 30 of the fixed patch overlaps), moved by a small rigid
    transform."""
    rng = np.random.default_rng(seed)
    Xf = synthetic.surface(n, seed, extent=30.0)
    x = np.concatenate((np.deg2rad(rng.uniform(-1, 1, 3)), rng.uniform(-0.2, 0.2, 3)))
    Xm = synthetic.apply_H(synthetic.surface(n + 17, seed + 1, extent=30.0, x0=shift), np.linalg.inv(synthetic.H_from_rbp(x)))
    return np.ascontiguousarray(Xf), np.ascontiguousarray(Xm)


def _few_overlap_pair():
    """Fixed: a surface patch plus three isolated points 100 m above it; movable: a patch 1 km away
    plus three points next to the isolated ones.  Exactly three fixed points are within D."""
    Xf = synthetic.surface(5000, 31, extent=30.0)
    iso = np.array([[10.0, 10.0, 100.0], [20.0, 10.0, 100.0], [10.0, 20.0, 100.0]])
    Xm = synthetic.surface(5000, 32, extent=30.0, x0=1000.0)
    return np.ascontiguousarray(np.vstack((Xf, iso))), np.ascontiguousarray(np.vstack((Xm, iso + 0.05)))


# ragged sizes; pair 1 keeps ~500 points (< correspondences), pair 4 keeps 3 (< 6)
SIZES = [40_000, 3_000, 25_000, 60_000, None, 80_000, 12_345, 20_000]
SHIFTS = [10.0, 25.0, 0.0, 15.0, None, 20.0, 5.0, 12.0]


@pytest.fixture(scope="module")
def ragged_pairs():
    return [_few_overlap_pair() if n is None else _patch_pair(n, s, 20_000 + 2 * i)
            for i, (n, s) in enumerate(zip(SIZES, SHIFTS))]


def _params(e, observed_deg=(0.0,) * 6, weights=(0.0,) * 6, dw=1.0, min_planarity=0.3, min_change=1.0,
            max_iterations=100):
    obs = _observed_in_radians(observed_deg)
    lsq = e.lsq_params(obs, obs, [float(w) for w in weights], dw)
    return e.run_params(min_planarity, min_change, max_iterations, lsq)


def _assert_same_as_register(e, b, Xf, Xm, **kw):
    r = sb.register(Xf, Xm, engine=e, want_normals=False, **kw)
    H = np.array(b.H).reshape(4, 4)
    assert b.status == 0
    assert b.iterations == r.iterations and bool(b.converged) == r.converged
    assert b.n_kept == r.records[-1]["n_kept"]
    assert b.n_selected == e.K  # sicp_register's n_selected
    np.testing.assert_allclose(H, r.H, rtol=0, atol=1e-12)
    np.testing.assert_allclose(np.array(b.x), r.rbp.get_parameter_attributes_as_list("estimated_value"), rtol=0, atol=1e-12)
    np.testing.assert_allclose([b.mean_res, b.std_res], [r.residuals.mean(), r.residuals.std()], rtol=1e-9, atol=1e-15)
    return r


@pytest.mark.gpu
def test_batched_overlap_equals_per_pair_registration(gpu, ragged_pairs):
    """Ragged batch of partly overlapping pairs, filter from H0 = I and from H0 != I (observed
    values): every pair equals sicp_register with the filter; the pair with 3 kept points fails
    alone with TOO_FEW_CORR, as sicp_register does."""
    pairs = ragged_pairs
    with _capi.Engine() as e:
        for observed in ((0.0,) * 6, (0.05, -0.03, 0.02, 0.1, -0.05, 0.02)):
            res = e.register_batch(pairs, 1000, 10, _params(e, observed), D)
            assert e.timings()["overlap_ms"] > 0
            for i, (Xf, Xm) in enumerate(pairs):
                b = res[i]
                print(f"obs {observed[0]}: pair {i}: status {b.status} it {b.iterations} n_selected {b.n_selected} kept {b.n_kept}")
                if i == 4:
                    assert b.status == _capi.SICP_ERR_TOO_FEW_CORR and b.n_selected == 3
                    with pytest.raises(sb.SimpleICPException):
                        sb.register(Xf, Xm, engine=e, want_normals=False, max_overlap_distance=D,
                                    rbp_observed_values=observed)
                    continue
                _assert_same_as_register(e, b, Xf, Xm, max_overlap_distance=D, rbp_observed_values=observed)
                if i == 1:
                    assert 0 < b.n_selected < 1000  # K = the kept count
                else:
                    assert b.n_selected == 1000


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bunny", "multisensor"])
def test_batched_overlap_reference_configs(gpu, name):
    """The reference's partial-overlap configurations (max_overlap_distance = 1) through the
    batched engine: K = min(correspondences, |idx_overlap|), H as sicp_register."""
    g = load_golden(name)
    kw = g["kwargs"]
    X_fix, X_mov = load_pair(name)
    corr, nb = kw.get("correspondences", 1000), kw.get("neighbors", 10)
    with _capi.Engine() as e:
        p = _params(e, kw.get("rbp_observed_values", (0.0,) * 6), kw.get("rbp_observation_weights", (0.0,) * 6),
                    kw.get("distance_weights", 1), kw.get("min_planarity", 0.3), kw.get("min_change", 1.0),
                    kw.get("max_iterations", 100))
        b = e.register_batch([(X_fix, X_mov)], corr, nb, p, kw["max_overlap_distance"])[0]
        assert b.status == 0
        assert b.n_selected == min(corr, len(g["idx_overlap"]))
        r = sb.register(X_fix, X_mov, engine=e, want_normals=False, **kw)
        assert b.iterations == r.iterations and b.n_kept == r.records[-1]["n_kept"]
        np.testing.assert_allclose(np.array(b.H).reshape(4, 4), r.H, rtol=0, atol=1e-12)


@pytest.mark.gpu
def test_batched_overlap_pair_without_overlap_fails_alone(gpu):
    pairs = [_patch_pair(n, s, 30_000 + 2 * i) for i, (n, s) in enumerate(zip([30_000, 20_000, 40_000, 25_000], [10.0, 5.0, 8.0, 15.0]))]
    pairs[2] = (pairs[2][0], pairs[2][1] + np.array([1000.0, 0.0, 0.0]))
    ok = [0, 1, 3]
    with _capi.Engine() as e:
        res = e.register_batch(pairs, 1000, 10, _params(e), D)
        alone = e.register_batch([pairs[i] for i in ok], 1000, 10, _params(e), D)
    assert [r.status for r in res] == [0, 0, _capi.SICP_ERR_NO_OVERLAP, 0]
    assert res[2].n_selected == 0 and res[2].iterations == 0
    for j, i in enumerate(ok):
        a, b = res[i], alone[j]
        assert (a.iterations, a.converged, a.n_kept, a.n_selected) == (b.iterations, b.converged, b.n_kept, b.n_selected)
        np.testing.assert_allclose(np.array(a.H), np.array(b.H), rtol=0, atol=1e-12)
        np.testing.assert_allclose([a.mean_res, a.std_res], [b.mean_res, b.std_res], rtol=1e-12, atol=1e-15)
    with pytest.raises(sb.batch.BatchError) as ei:
        sb.simpleicp_batch(pairs, max_overlap_distance=D)
    assert ei.value.failed.tolist() == [2]
    assert ei.value.table[2, 16] == -_capi.SICP_ERR_NO_OVERLAP
    table = sb.simpleicp_batch(pairs, max_overlap_distance=D, on_error="nan")
    pool = sb.simpleicp_batch(pairs, max_overlap_distance=D, on_error="nan", engine="pool")
    assert pool[2, 16] == table[2, 16] == -_capi.SICP_ERR_NO_OVERLAP
    np.testing.assert_allclose(table[ok, :16], pool[ok, :16], rtol=0, atol=1e-12)
    assert np.array_equal(table[ok, 16:18], pool[ok, 16:18])


@pytest.mark.gpu
def test_simpleicp_batch_routes_overlap_to_batched_engine(gpu, ragged_pairs):
    pairs = [p for i, p in enumerate(ragged_pairs) if i != 4]
    table = sb.simpleicp_batch(pairs, max_overlap_distance=D, max_iterations=50)
    assert sb.batch._BATCH_ENGINES[0].timings()["overlap_ms"] > 0
    pool = sb.simpleicp_batch(pairs, max_overlap_distance=D, max_iterations=50, engine="pool")
    np.testing.assert_allclose(table[:, :16], pool[:, :16], rtol=0, atol=1e-12)
    assert np.array_equal(table[:, 16:18], pool[:, 16:18])


@pytest.mark.gpu
def test_batched_overlap_off_means_off(gpu, ragged_pairs):
    """inf, -1 and 0 run the batch without the filter."""
    pairs = [p for i, p in enumerate(ragged_pairs) if i != 4]
    with _capi.Engine() as e:
        ref = e.register_batch(pairs, 1000, 10, _params(e, max_iterations=30))
        assert e.timings()["overlap_ms"] == 0
        for d in (np.inf, -1.0, 0.0):
            res = e.register_batch(pairs, 1000, 10, _params(e, max_iterations=30), d)
            for (Xf, _), a, b in zip(pairs, res, ref):
                assert a.status == b.status == 0
                assert a.n_selected == min(1000, Xf.shape[0])
                assert (a.iterations, a.n_kept, a.n_selected) == (b.iterations, b.n_kept, b.n_selected)
                np.testing.assert_allclose(np.array(a.H), np.array(b.H), rtol=0, atol=1e-12)


def test_overlap_filter_is_batchable():
    assert sb.batch._batchable({"max_overlap_distance": 1.0, "correspondences": 1000})
    assert sb.batch._batchable({"max_overlap_distance": np.inf})
    assert not sb.batch._batchable({"max_overlap_distance": 1.0, "correspondences": 5000})


def test_pair_result_layout_matches_header(tmp_path):
    """sizeof(sicp_pair_result) and the offsets of n_selected / n_kept, as gcc sees the header,
    equal the ctypes mirror."""
    src = tmp_path / "layout.c"
    src.write_text(r"""
#include <stdio.h>
#include <stddef.h>
#include "sicp_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(sicp_pair_result), offsetof(sicp_pair_result, n_selected),
         offsetof(sicp_pair_result, n_kept), offsetof(sicp_pair_result, std_res));
  return 0;
}
""")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(REPO / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(_capi.PairResult), _capi.PairResult.n_selected.offset, _capi.PairResult.n_kept.offset,
                   _capi.PairResult.std_res.offset]
