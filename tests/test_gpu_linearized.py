"""GPU parity tests of the linearised variant (SURVEY.md section 8f rank 3): the CUDA path through
the C ABI against oracle/linearized_oracle.py (the restatement of the C++ driver).

The restatement itself is pinned to the UNMODIFIED C++ sources (tests/test_cpp_reference_pin.py,
CPU); ``test_against_the_compiled_cpp_reference`` below additionally compares the CUDA path with
that compiled reference's own per-iteration output directly (tests/golden/cppref_*.npz).

Tolerances, and why:
  * injected normals (the oracle's, rounded to the float32 the library stores): the two sides do
    the same arithmetic in a different order -> iteration count, kept counts identical; residual
    statistics and H to 1e-9 (normal-equation solve vs SVD, moment sums vs row sums);
  * own normals: the eigenvector SIGN convention differs (LAPACK dsyevd in the oracle, dgeev
    emulation on the GPU).  The estimate does not depend on it; the median of the signed distances
    does, so kept counts move by a few and H agrees to the north star's 1e-5 only.
"""
import numpy as np
import pytest

from conftest import load_pair
from oracle import linearized_oracle as LO
from oracle import simpleicp_oracle as O

import simpleicp_b200 as sb
from simpleicp_b200 import _capi, linearized

pytestmark = pytest.mark.gpu


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def noisy_pair(n, seed=0):
    """A C3-style undulating surface pair with 1 cm noise (SURVEY.md section 8d), small."""
    X_fix = O.surface(n, 1234 + seed, extent=30.0)
    H_true = O.rbp_to_H(np.array([np.radians(0.3), np.radians(-0.2), np.radians(0.5), 0.15, -0.10, 0.05]))
    X_mov = O.transform_by_H(O.surface(n, 5678 + seed, extent=30.0), np.linalg.inv(H_true))
    return X_fix, X_mov


CASES = {
    "dragon": dict(pair=lambda: load_pair("dragon"), kw=dict()),
    "multisensor": dict(pair=lambda: load_pair("multisensor"), kw=dict()),
    "surface_K6000": dict(pair=lambda: noisy_pair(60_000), kw=dict(correspondences=6000)),  # K > 4096: cooperative path
}


@pytest.mark.parametrize("compose", ["dH*H", "H*dH"])
@pytest.mark.parametrize("name", list(CASES))
def test_lockstep_injected_normals(gpu, name, compose):
    X_fix, X_mov = CASES[name]["pair"]()
    kw = CASES[name]["kw"]
    pre = LO.simpleicp_linearized(X_fix, X_mov, max_iterations=1, **kw)  # only for normals + selection
    n32, p32 = f32(pre.normals), f32(pre.planarity)
    ref = LO.simpleicp_linearized(X_fix, X_mov, normals=n32, planarity=p32,
                                  compose="post" if compose == "H*dH" else "pre", **kw)
    res = sb.simpleicp_linearized(X_fix, X_mov, compose=compose,
                                  normals=(n32[:, 0], n32[:, 1], n32[:, 2], p32), **kw)
    assert np.array_equal(res.idx_selected, ref.idx_fix)
    assert res.iterations == len(ref.iterations) and res.converged == ref.converged
    assert res.records[0]["n_kept"] == ref.orig.n_kept
    assert res.records[0]["mean_dist"] == pytest.approx(ref.orig.mean, abs=1e-12)
    assert res.records[0]["std_dist"] == pytest.approx(ref.orig.std, rel=1e-10)
    for rec, it in zip(res.records, ref.iterations):
        assert rec["n_kept"] == it.n_kept
        assert rec["mean_res"] == pytest.approx(it.mean, abs=1e-9)
        assert rec["std_res"] == pytest.approx(it.std, abs=1e-9)
        np.testing.assert_allclose(rec["x"], it.x, atol=1e-9, rtol=0)
    assert np.linalg.norm(res.H - ref.H) < 1e-9
    assert np.linalg.norm(res.T - ref.T) < 1e-9
    if compose == "dH*H":
        assert np.array_equal(res.H, res.T)
    Xt = O.transform_by_H(X_mov, ref.T)
    np.testing.assert_allclose(np.asarray(res.X_mov_transformed), Xt, atol=1e-8, rtol=0)
    # the screen table is the C++ driver's
    assert res.table.splitlines()[:len(LO.format_table(ref).splitlines())] == LO.format_table(ref).splitlines() \
        or _tables_agree(res.table, LO.format_table(ref))


CPPREF = {  # fixture -> input pair (oracle/make_golden_cpp.py: c++/run_simpleicp.sh + two flag variations)
    "dragon": "dragon",
    "bunny": "bunny",
    "airborne": "airborne",
    "dragon_k5000": "dragon",   # K = 5000 > 4096: the multi-block kernels
    "bunny_maxit3": "bunny",    # leaves through max_iterations, no convergence line
}


@pytest.mark.parametrize("name", list(CPPREF))
def test_against_the_compiled_cpp_reference(gpu, name):
    """The CUDA path against the per-iteration output of the unmodified C++ reference (compiled
    from the reference's c++/src by oracle/Makefile, run by oracle/make_golden_cpp.py).  The
    reference run's normals are handed over (rounded to the float32 the library stores): the
    eigenvector sign is implementation defined on both sides.  Measured on the CPU restatement,
    that rounding moves H by < 1e-9 on these inputs and no kept count at all, so: selection,
    iteration count and every kept count EXACT, residual statistics 1e-7, dH-chain and reported
    H = H * dH 1e-7, screen table identical."""
    from conftest import GOLD

    g = dict(np.load(GOLD / f"cppref_{name}.npz"))
    p = eval(str(g["params_repr"]), {"inf": np.inf})
    X_fix, X_mov = load_pair(CPPREF[name])
    n32, p32 = f32(g["normals"]), f32(g["planarity"])
    res = sb.simpleicp_linearized(X_fix, X_mov, p["correspondences"], p["neighbors"], p["min_planarity"],
                                  p["max_overlap_distance"], p["min_change"], p["max_iterations"],
                                  compose="H*dH", normals=(n32[:, 0], n32[:, 1], n32[:, 2], p32))
    assert np.array_equal(res.idx_selected, g["idx_fix"])
    assert res.iterations == len(g["n_kept"]) and res.converged == bool(g["converged"])
    assert [r["n_kept"] for r in res.records[:res.iterations]] == g["n_kept"].tolist()
    assert res.records[0]["mean_dist"] == pytest.approx(float(g["initial_mean"][0]), abs=1e-7)
    assert res.records[0]["std_dist"] == pytest.approx(float(g["initial_std"][0]), abs=1e-7)
    T = np.eye(4)
    for i in range(res.iterations):
        rec = res.records[i]
        assert rec["mean_res"] == pytest.approx(float(g["mean"][i]), abs=1e-7)
        assert rec["std_res"] == pytest.approx(float(g["std"][i]), abs=1e-7)
        dH = np.eye(4)
        dH[:3, :3] = LO.euler_angles_to_rotation_matrix(*rec["x"][:3])
        dH[:3, 3] = rec["x"][3:]
        assert np.abs(dH - g["dH"][i]).max() < 1e-7
        T = g["dH"][i] @ T
    assert np.abs(res.H - g["H_api"]).max() < 1e-7      # what SimpleICP() returned
    assert np.abs(res.T - T).max() < 1e-7               # what its cloud was moved by
    np.testing.assert_allclose(np.asarray(res.X_mov_transformed), O.transform_by_H(X_mov, T), atol=1e-5, rtol=0)
    assert _tables_agree(res.table, str(g["cli_screen"]))
    shown = np.array([[float(v) for v in ln.strip("[]").split()]
                      for ln in str(g["cli_screen"]).splitlines() if ln.startswith("[")])
    assert np.abs(shown - res.H).max() < 1e-6           # the reference CLI's printed matrix


def _tables_agree(a, b):
    """Same rows up to the sign of a printed zero ("-0.0000" vs "0.0000")."""
    la = [ln.replace("-0.0000", " 0.0000") for ln in a.splitlines() if "|" in ln]
    lb = [ln.replace("-0.0000", " 0.0000") for ln in b.splitlines() if "|" in ln]
    return la == lb


@pytest.mark.parametrize("name", ["dragon", "surface_K6000"])
def test_own_normals_chain(gpu, name):
    """Stand-alone run, decomposed: (1) the library's normals equal the float64 restatement's up
    to sign and float32 rounding; (2) with THOSE normals handed to the restatement the two runs
    agree like the lock-step test; (3) against the restatement's own float64 / other-sign normals
    the result moves only at the level the data's noise allows (1e-5 on the noise-free pair)."""
    X_fix, X_mov = CASES[name]["pair"]()
    kw = CASES[name]["kw"]
    res = sb.simpleicp_linearized(X_fix, X_mov, want_normals=True, **kw)      # stage by stage
    fused = sb.simpleicp_linearized(X_fix, X_mov, **kw)                       # one sicp_register call
    assert np.array_equal(res.T, fused.T) and res.iterations == fused.iterations
    assert np.array_equal(res.idx_selected, fused.idx_selected)
    assert np.array_equal(np.asarray(res.X_mov_transformed), np.asarray(fused.X_mov_transformed))
    ref64 = LO.simpleicp_linearized(X_fix, X_mov, compose="pre", **kw)
    n_gpu = np.stack([np.asarray(a, dtype=np.float64) for a in res.normals[:3]], axis=1)
    p_gpu = np.asarray(res.normals[3], dtype=np.float64)
    sgn = np.sign(np.einsum("ij,ij->i", n_gpu, ref64.normals))
    assert np.abs(n_gpu - sgn[:, None] * ref64.normals).max() < 5e-6  # float32 store + ill-conditioned eigenvectors
    assert np.abs(p_gpu - ref64.planarity).max() < 2e-5
    ref = LO.simpleicp_linearized(X_fix, X_mov, compose="pre", normals=n_gpu, planarity=p_gpu, **kw)
    assert res.iterations == len(ref.iterations)
    for rec, it in zip(res.records, ref.iterations):
        assert rec["n_kept"] == it.n_kept
        assert rec["mean_res"] == pytest.approx(it.mean, abs=1e-9)
        assert rec["std_res"] == pytest.approx(it.std, abs=1e-9)
    assert np.linalg.norm(res.T - ref.T) < 1e-9
    assert res.converged and ref64.converged
    assert abs(res.iterations - len(ref64.iterations)) <= 2
    assert np.linalg.norm(res.T - ref64.T) < (1e-5 if name == "dragon" else 2e-4)


def test_overlap_filter_and_cli_defaults(gpu):
    X_fix, X_mov = load_pair("bunny")
    ref = LO.simpleicp_linearized(X_fix, X_mov, max_overlap_distance=1.0, compose="pre")
    res = sb.simpleicp_linearized(X_fix, X_mov, max_overlap_distance=1.0)
    assert np.array_equal(res.idx_selected, ref.idx_fix)
    assert np.linalg.norm(res.T - ref.T) < 1e-4  # noisy scans, sign-dependent rejection sets
    with pytest.raises(RuntimeError, match="do not overlap"):
        sb.simpleicp_linearized(X_fix, X_mov + 1e4, max_overlap_distance=1.0)


def test_variant_is_an_engine_option_and_is_reset(gpu):
    X_fix, X_mov = load_pair("dragon")
    eng = _capi.Engine()
    try:
        a = sb.register(X_fix, X_mov, engine=eng)
        sb.simpleicp_linearized(X_fix, X_mov, engine=eng)
        b = sb.register(X_fix, X_mov, engine=eng)  # back to the default variant, bit-identical
        assert np.array_equal(a.H, b.H) and a.iterations == b.iterations
        # observed / fixed parameters do not exist in the linearised drivers
        eng.set_option("variant", linearized.VARIANT_LINEARIZED)
        lsq = eng.lsq_params([0] * 6, [0] * 6, [0, 0, 0, np.inf, 0, 0], 1.0)
        with pytest.raises(_capi.SicpError, match="no observed or fixed"):
            eng.run(eng.run_params(0.3, 1.0, 10, lsq))
        with pytest.raises(_capi.SicpError, match="variant"):
            eng.set_option("variant", 3)
    finally:
        eng.close()


def test_cli_variant_cpp_prints_the_cpp_driver_output(gpu, tmp_path):
    """sicp_cli --variant cpp on .xyz files: the table, H (= H * dH) and transformed cloud of the
    C++ reference CLI's own algorithm (c++/src/simpleicp-cli.cpp + simpleicp.cpp)."""
    import re
    import subprocess

    from conftest import REPO

    cli = REPO / "simpleicp_b200" / "sicp_cli"
    X_fix, X_mov = load_pair("dragon")
    f1, f2, fo = tmp_path / "d1.xyz", tmp_path / "d2.xyz", tmp_path / "out.xyz"
    sb.write_xyz(f1, X_fix, decimals=4, header=False)
    sb.write_xyz(f2, X_mov, decimals=4, header=False)
    ref = LO.simpleicp_linearized(X_fix, X_mov, compose="post")
    pat = r"^\[\s*(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\]$"
    for variant in ("linearized", "cpp"):
        r = subprocess.run([str(cli), "-f", str(f1), "-m", str(f2), "--variant", variant, "--out", str(fo)],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        H = np.array(re.findall(pat, r.stdout, re.M), dtype=float)
        if variant == "linearized":
            assert np.abs(H - ref.T).max() < 2e-5  # dH * H: the applied transform, printed to 6 decimals
        else:
            # H * dH multiplies the same increments in the other order: it is NOT the applied
            # transform and depends on the path (which the normal-sign convention perturbs)
            assert np.abs(H - ref.H).max() < 5e-3 and np.abs(H - ref.T).max() > 1e-3
        shown = re.findall(r"^\s+(\d+) \|\s+(\d+) \|", r.stdout, re.M)
        assert abs(len(shown) - (len(ref.iterations) - 1)) <= 1  # the converging iteration is not printed
        assert "Convergence criteria fulfilled -> stop iteration!" in r.stdout
        # either way the cloud written is the one the loop really moved
        np.testing.assert_allclose(sb.read_xyz(fo), O.transform_by_H(X_mov, ref.T), atol=2e-4)
    bad = subprocess.run([str(cli), "-f", str(f1), "-m", str(f2), "--variant", "nope"], capture_output=True, text=True)
    assert bad.returncode == 1 and "unknown variant" in bad.stderr


def test_reference_cpp_cli_linked_against_the_library(gpu, tmp_path):
    """INTEGRATION.md section 5 as a running program: the reference's own, unmodified CLI main()
    (c++/src/simpleicp-cli.cpp) linked with integration/cpp/simpleicp_b200_binding.cpp -- the
    reference's SimpleICP() signature implemented on the C ABI -- instead of its CPU sources
    (oracle/Makefile -> oracle/_ref/simpleicp_cpp_b200, built where the reference checkout is readable).  Its
    screen output must be the library's linearised run, and agree with the CPU build of the same
    CLI (tests/golden/cppref_dragon.npz) as far as the eigenvector sign convention allows."""
    import re
    import subprocess

    from conftest import GOLD, REPO

    exe = REPO / "oracle" / "_ref" / "simpleicp_cpp_b200"
    if not exe.exists():
        pytest.skip("oracle/_ref/simpleicp_cpp_b200 not built (needs the reference checkout at build time)")
    X_fix, X_mov = load_pair("dragon")
    f1, f2 = tmp_path / "dragon1.xyz", tmp_path / "dragon2.xyz"
    sb.write_xyz(f1, X_fix, decimals=4, header=False)
    sb.write_xyz(f2, X_mov, decimals=4, header=False)
    r = subprocess.run([str(exe), "--fixed", str(f1), "--movable", str(f2)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    ours = sb.simpleicp_linearized(X_fix, X_mov, compose="H*dH")
    assert _tables_agree(r.stdout, ours.table)
    pat = r"^\[\s*(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\s+(-?[\d.]+)\]$"
    H = np.array(re.findall(pat, r.stdout, re.M), dtype=float)
    assert np.abs(H - ours.H).max() < 1e-6                      # same library run, printed to 6 decimals
    for line in ("Create point cloud objects ...", "Select points for correspondences in fixed point cloud ...",
                 "Estimate normals of selected points ...", "Start iterations ...",
                 "Convergence criteria fulfilled -> stop iteration!", "Estimated transformation matrix H:"):
        assert line in r.stdout
    assert re.search(r"^Finished in \d+\.\d{3} seconds!$", r.stdout, re.M)  # what scripts/benchmark.sh:45-51 parses
    # against the CPU build of the same CLI: same registration, other eigenvector signs
    g = dict(np.load(GOLD / "cppref_dragon.npz"))
    shown = re.findall(r"^\s+(\d+) \|\s+(\d+) \|", r.stdout, re.M)
    assert abs(len(shown) - (len(g["n_kept"]) - 1)) <= 1
    assert np.abs(H - g["H_api"]).max() < 5e-3                   # H * dH depends on the path
    T = np.eye(4)
    for dH in g["dH"]:
        T = dH @ T
    assert np.abs(ours.T - T).max() < 1e-5                       # the applied transform does not
    # the reference CLI's error path (simpleicp.cpp:26-36 caught at simpleicp-cli.cpp:60-64)
    far = tmp_path / "far.xyz"
    sb.write_xyz(far, X_mov + 1e4, decimals=4, header=False)
    bad = subprocess.run([str(exe), "--fixed", str(f1), "--movable", str(far), "--max_overlap_distance", "1"],
                         capture_output=True, text=True, timeout=300)
    assert bad.returncode == 1
    assert "Caught exception: Point clouds do not overlap within max_overlap_distance = 1.00000." in bad.stderr
