"""Pins oracle/linearized_oracle.py (the restatement of the linearised simpleICP variant) to the
UNMODIFIED C++ reference: tests/golden/cppref_<name>.npz were written by
oracle/make_golden_cpp.py from the reference's c++/src compiled by oracle/Makefile against the
stand-in dependency headers in oracle/cpp_standin (Eigen, nanoflann and cxxopts are not in the
image).  Configurations: the four command lines of c++/run_simpleicp.sh:11-41 (dragon, airborne,
terrestrial, bunny with --max_overlap_distance 1) plus two with non-default flags.

What is compared, and how tightly:
  * selection (overlap filter count, LinSpaced + round picks)          -- exact;
  * normals up to sign 1e-9, planarity 1e-9 (Jacobi stand-in vs LAPACK dsyevd) wherever the
    k-nearest-neighbour SET is unique (no tie at the k-th distance) and the two smallest
    eigenvalues are separated;
  * with the C++ run's normals injected, every iteration: nearest neighbours (equal up to
    exact-distance ties), signed distances 1e-11, kept sets EXACT, residual mean / std 1e-11,
    dH and H = H * dH 1e-11, iteration count and convergence flag exact;
  * the screen table of the restatement equals the reference CLI's output character by character
    (up to the sign of a printed zero).
The stand-alone restatement (its own eigenvector signs) is compared loosely: the sign of a normal
flips the sign of that correspondence's distance, which moves the median the rejection is
centred on (documented in the oracle's header).
"""
import shutil
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import load_pair

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "oracle"))
import linearized_oracle as lo  # noqa: E402
import make_golden_cpp as mg  # noqa: E402

GOLD = ROOT / "tests" / "golden"
DATA = {"dragon_k5000": "dragon", "bunny_maxit3": "bunny"}
NAMES = ["dragon", "bunny", "airborne", "terrestrial", "dragon_k5000", "bunny_maxit3", "multisensor"]


def load_cppref(name):
    g = dict(np.load(GOLD / f"cppref_{name}.npz"))
    g["params"] = eval(str(g["params_repr"]), {"inf": np.inf})
    return g


def oracle_kwargs(p):
    mo = p["max_overlap_distance"]
    return dict(correspondences=p["correspondences"], neighbors=p["neighbors"], min_planarity=p["min_planarity"],
                max_overlap_distance=(mo if mo > 0 else np.inf), min_change=p["min_change"],
                max_iterations=p["max_iterations"])


def screen_rows(text):
    return [ln.replace("-0.0000", " 0.0000") for ln in text.splitlines() if " | " in ln]


@pytest.mark.parametrize("name", NAMES)
def test_restatement_in_lockstep_with_the_cpp_reference(name):
    g = load_cppref(name)
    X_fix, X_mov = load_pair(DATA.get(name, name))
    kw = oracle_kwargs(g["params"])

    # selection and normals, computed by the restatement itself
    pre = lo.simpleicp_linearized(X_fix, X_mov, **dict(kw, max_iterations=1))
    assert np.array_equal(pre.idx_fix, g["idx_fix"])
    if g["params"]["max_overlap_distance"] > 0:
        assert lo.select_in_range(X_fix, X_mov, g["params"]["max_overlap_distance"]).size == int(g["n_in_range"])
    # a neighbourhood whose k-th and (k+1)-th neighbours are equally far has no unique k-NN set
    from scipy import spatial
    k = g["params"]["neighbors"]
    dk, _ = spatial.cKDTree(X_fix).query(X_fix[g["idx_fix"]], k=k + 1)
    unique = dk[:, k] - dk[:, k - 1] > 1e-12
    assert unique.mean() > 0.5  # terrestrial (mm-quantised scan): 44 % of the neighbourhoods tie
    assert np.abs(pre.planarity - g["planarity"])[unique].max() < 1e-9
    # eigenvector agreement is bounded by the gap between the two smallest eigenvalues
    dots = np.abs(np.einsum("ij,ij->i", pre.normals, g["normals"]))
    assert np.abs(dots - 1)[unique & (g["planarity"] > 0.05)].max() < 1e-9

    # the loop, with the reference run's normals and -- where several movable points are equally
    # near -- its pick among them (verified below to be a nearest neighbour)
    r = lo.simpleicp_linearized(X_fix, X_mov, compose="post", normals=g["normals"], planarity=g["planarity"],
                                keep_arrays=True, matches=g["idx_mov_all"], **kw)
    assert len(r.iterations) == len(g["n_kept"]) and r.converged == bool(g["converged"])
    assert r.orig.n_kept == g["n_kept"][0]
    assert r.orig.mean == pytest.approx(g["initial_mean"][0], abs=1e-12)
    assert r.orig.std == pytest.approx(g["initial_std"][0], abs=1e-12)
    H = np.eye(4)
    q = X_fix[g["idx_fix"]]
    for i, it in enumerate(r.iterations):
        moved = X_mov @ it.T_before[:3, :3].T + it.T_before[:3, 3]
        d_own = np.linalg.norm(moved[it.idx_mov_own] - q, axis=1)
        d_ref = np.linalg.norm(moved[g["idx_mov_all"][i]] - q, axis=1)
        differ = it.idx_mov_own != g["idx_mov_all"][i]
        assert differ.mean() < 0.1 and np.abs(d_own - d_ref).max() < 1e-12
        assert np.abs(it.dists - g["dists_all"][i]).max() < 1e-11
        kept_ref = g["idx_fix_kept"][i]
        assert np.array_equal(g["idx_fix"][it.keep], kept_ref[kept_ref >= 0])
        assert it.n_kept == g["n_kept"][i]
        assert it.mean == pytest.approx(g["mean"][i], abs=1e-11)
        assert it.std == pytest.approx(g["std"][i], abs=1e-11)
        dH = np.eye(4)
        dH[:3, :3] = lo.euler_angles_to_rotation_matrix(*it.x[:3])
        dH[:3, 3] = it.x[3:]
        H = H @ dH
        assert np.abs(dH - g["dH"][i]).max() < 1e-11
        assert np.abs(H - g["H"][i]).max() < 1e-11
    assert np.abs(r.H - g["H_api"]).max() < 1e-11
    assert np.array_equal(g["H"][-1], g["H_api"])  # the stage pass IS the run SimpleICP() made

    # the screen output: same table, same H to the 6 printed decimals
    assert screen_rows(lo.format_table(r)) == screen_rows(str(g["cli_screen"]))
    shown = [ln for ln in str(g["cli_screen"]).splitlines() if ln.startswith("[")]
    H_shown = np.array([[float(v) for v in ln.strip("[]").split()] for ln in shown])
    assert np.abs(H_shown - r.H).max() < 1e-6
    assert ("Convergence criteria fulfilled -> stop iteration!" in str(g["cli_screen"])) == r.converged


def test_lockstep_is_tight_where_no_ties_occur():
    """dragon has a handful of duplicated points (exact ties); the tie-free iterations and the
    airborne pair must agree to rounding, not to the loose bound the tie branch above allows."""
    for name in ("dragon", "airborne"):
        g = load_cppref(name)
        X_fix, X_mov = load_pair(name)
        r = lo.simpleicp_linearized(X_fix, X_mov, compose="post", normals=g["normals"], planarity=g["planarity"],
                                    **oracle_kwargs(g["params"]))
        assert [it.n_kept for it in r.iterations] == g["n_kept"].tolist()
        assert np.abs(np.array([it.std for it in r.iterations]) - g["std"]).max() < 1e-12
        assert np.abs(r.H - g["H_api"]).max() < 1e-12


def test_standalone_restatement_reaches_the_same_registration():
    """Own eigenvector signs (LAPACK's instead of the stand-in's): another rejection path, the same
    registration.  The applied transform T = ... dH2 dH1 is compared, not the path-dependent
    H = dH1 dH2 ... the C++ driver prints."""
    for name, tol in (("dragon", 1e-5), ("airborne", 5e-3)):
        g = load_cppref(name)
        X_fix, X_mov = load_pair(name)
        r = lo.simpleicp_linearized(X_fix, X_mov, compose="pre", **oracle_kwargs(g["params"]))
        T = np.eye(4)
        for dH in g["dH"]:
            T = dH @ T
        assert r.converged and abs(len(r.iterations) - len(g["dH"])) <= 2
        assert np.abs(r.T - T).max() < tol


@pytest.mark.skipif(mg.REF is None or shutil.which("g++") is None,
                    reason="needs g++ and a readable pglira/simpleICP checkout (oracle/make_golden_cpp.py)")
def test_fixture_is_reproduced_by_the_recipe(tmp_path):
    """Re-run the recipe: build oracle/_ref from the reference's C++ sources and compare the
    dragon fixture field by field -- the committed numbers are the compiled reference's."""
    cli, driver = mg.build()
    fix, mov, flags = mg.CONFIGS["dragon"]
    X_fix, X_mov = load_pair("dragon")
    j, screen = mg.run_driver(driver, X_fix, X_mov, flags)
    assert screen == mg.run_cli(cli, fix, mov, flags)
    fresh = mg.pack(j, screen, screen, dict(mg.DEFAULTS))
    g = dict(np.load(GOLD / "cppref_dragon.npz"))
    for key in ("H_api", "idx_fix", "normals", "planarity", "idx_mov_all", "dists_all", "idx_fix_kept", "n_kept",
                "mean", "std", "dH", "H"):
        assert np.array_equal(fresh[key], g[key]), key
    assert str(fresh["cli_screen"]) == str(g["cli_screen"])
    # the reference CLI's own error path (simpleicp.cpp:26-36 -> simpleicp-cli.cpp:60-64)
    far = tmp_path / "far.xyz"
    np.savetxt(far, X_mov[:2000] + 1e4, fmt="%.4f")
    r = subprocess.run([str(cli), "--fixed", str(mg.REF / "data" / "dragon1.xyz"), "--movable", str(far),
                        "--max_overlap_distance", "1"], capture_output=True, text=True)
    assert r.returncode == 1 and "Point clouds do not overlap within max_overlap_distance" in r.stderr
