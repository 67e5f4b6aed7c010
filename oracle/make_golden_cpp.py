"""Generate tests/golden/cppref_<name>.npz by running the UNMODIFIED C++ reference.

Needs g++ and a checkout of pglira/simpleICP (DEFAULT_REFERENCE, or the one $SIMPLEICP_REFERENCE
names):

    python oracle/make_golden_cpp.py            # dragon, bunny, airborne, terrestrial (+ extras)

The C++ tree (c++/src of that checkout) is the definition of the LINEARISED simpleICP variant
(SURVEY.md section 8f rank 3).  Its sources are compiled where they lie -- never copied -- by
oracle/Makefile into oracle/_ref/ against stand-in headers for the three third-party libraries
the image lacks (oracle/cpp_standin: the used subset of Eigen's, nanoflann's and cxxopts'
documented interfaces; see the header of cpp_standin/Eigen/Dense for what that does and does not
pin), exactly as oracle/lmfit_standin does for the Python package.

Two programs are run per configuration:

  * oracle/_ref/simpleicp_cpp -- the reference's own CLI main() -- with the command lines of
    c++/run_simpleicp.sh on the .xyz files under data/ of the checkout: its screen output
    (iteration table to 4 decimals, H to 6) is stored verbatim (minus the wall-clock line);
  * oracle/_ref/simpleicp_cpp_driver (oracle/cpp_driver.cpp) -- calls the reference's
    SimpleICP() for H with 17 digits and then replays the same sequence of calls on the
    reference's PointCloud / CorrPts objects to record every stage with full precision; it
    fails unless both passes end in the bit-identical H.

tests/test_cpp_reference_pin.py checks oracle/linearized_oracle.py against these files (and
re-runs this recipe where the checkout is readable); tests/test_gpu_linearized.py checks the
CUDA path against the same files.
"""
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parents[1]
# where the fixtures were generated from; $SIMPLEICP_REFERENCE names another checkout
DEFAULT_REFERENCE = "/root/reference"


def reference_root():
    """The pglira/simpleICP checkout to build the reference from; None where its C++ sources are
    absent or cannot be read (a directory the user may not enter is the same as none)."""
    root = Path(os.environ.get("SIMPLEICP_REFERENCE") or DEFAULT_REFERENCE)
    try:
        return root if (root / "c++" / "src" / "simpleicp.cpp").is_file() else None
    except OSError:
        return None


REF = reference_root()
GOLD = REPO / "tests" / "golden"
OUT = REPO / "oracle" / "_ref"
sys.path.insert(0, str(REPO / "tests"))

# name -> (fixed, movable, CLI flags).  The first four are c++/run_simpleicp.sh:11-41 verbatim;
# the next two add a non-default correspondences / neighbors / min_planarity combination and the
# max_iterations exit (no convergence message).
CONFIGS = {
    "dragon": ("dragon1.xyz", "dragon2.xyz", {}),
    "airborne": ("airborne_lidar1.xyz", "airborne_lidar2.xyz", {}),
    "terrestrial": ("terrestrial_lidar1.xyz", "terrestrial_lidar2.xyz", {}),
    "bunny": ("bunny_part1.xyz", "bunny_part2.xyz", {"max_overlap_distance": 1}),
    "dragon_k5000": ("dragon1.xyz", "dragon2.xyz",
                     {"correspondences": 5000, "neighbors": 15, "min_planarity": 0.5, "min_change": 0.1}),
    "bunny_maxit3": ("bunny_part1.xyz", "bunny_part2.xyz", {"max_overlap_distance": 1, "max_iterations": 3}),
    # a small pair of the Python test file (python/simpleicp/tests/test_simpleicp.py:66-80) with the flag
    # the C++ CLI has for it: fewer selectable points than correspondences (SelectNPts is a no-op), 32
    # iterations.  (webots without its initial transform -- the C++ CLI has no such flag -- stays at
    # the identity on a lattice full of equidistant neighbours: not kept.)
    "multisensor": ("multisensor_lidar.xyz", "multisensor_radar.xyz", {"max_overlap_distance": 1}),
}
DEFAULTS = dict(correspondences=1000, neighbors=10, min_planarity=0.3, max_overlap_distance=-1.0,
                min_change=1.0, max_iterations=100)  # c++/src/simpleicp-cli.cpp:20-35


def build():
    subprocess.run(["make", "-C", str(REPO / "oracle"), f"REF={REF}/c++/src"], check=True,
                   stdout=subprocess.DEVNULL)
    return OUT / "simpleicp_cpp", OUT / "simpleicp_cpp_driver"


def run_cli(cli, fix, mov, flags):
    cmd = [str(cli), "--fixed", str(REF / "data" / fix), "--movable", str(REF / "data" / mov)]
    for k, v in flags.items():
        cmd += [f"--{k}", repr(v) if isinstance(v, float) else str(v)]
    out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
    return "\n".join(ln for ln in out.splitlines() if not ln.startswith("Finished in"))


def run_driver(driver, X_fix, X_mov, flags):
    p = dict(DEFAULTS)
    p.update(flags)
    with tempfile.TemporaryDirectory() as tmp:
        f, m, o = Path(tmp) / "fix.f64", Path(tmp) / "mov.f64", Path(tmp) / "out.json"
        np.ascontiguousarray(X_fix, dtype=np.float64).tofile(f)
        np.ascontiguousarray(X_mov, dtype=np.float64).tofile(m)
        r = subprocess.run([str(driver), str(f), str(m), str(len(X_fix)), str(len(X_mov)),
                            str(p["correspondences"]), str(p["neighbors"]), repr(float(p["min_planarity"])),
                            repr(float(p["max_overlap_distance"])), repr(float(p["min_change"])),
                            str(p["max_iterations"]), str(o)], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"driver failed ({r.returncode}): {r.stderr[-500:]}")
        lines = r.stdout.splitlines()
        screen = lines[lines.index("### SimpleICP() begin") + 1:lines.index("### SimpleICP() end")]
        return json.loads(o.read_text()), "\n".join(ln for ln in screen if not ln.startswith("Finished in"))


def pack(j, cli_screen, api_screen, params):
    its = j["iterations"]
    n = len(its)
    K = len(j["idx_fix"])
    kept = np.full((n, K), -1, dtype=np.int64)
    for i, it in enumerate(its):
        kept[i, :len(it["idx_fix_kept"])] = it["idx_fix_kept"]
    return dict(
        H_api=np.array(j["H_api"]),
        n_in_range=np.int64(j["n_in_range"]),
        idx_fix=np.array(j["idx_fix"], dtype=np.int64),
        normals=np.column_stack([j["nx"], j["ny"], j["nz"]]),
        planarity=np.array(j["planarity"]),
        idx_mov_all=np.array([it["idx_mov_all"] for it in its], dtype=np.int64),
        dists_all=np.array([it["dists_all"] for it in its]),
        idx_fix_kept=kept,  # rows padded with -1
        n_kept=np.array([it["n_kept"] for it in its], dtype=np.int64),
        initial_mean=np.array([it["initial_mean"] for it in its]),
        initial_std=np.array([it["initial_std"] for it in its]),
        mean=np.array([it["mean"] for it in its]),
        std=np.array([it["std"] for it in its]),
        dH=np.array([it["dH"] for it in its]),
        H=np.array([it["H"] for it in its]),
        converged=np.bool_(j["converged"]),
        cli_screen=np.str_(cli_screen),
        params_repr=np.str_(repr(params)),
        recipe=np.str_("oracle/make_golden_cpp.py: unmodified c++/src of pglira/simpleICP compiled by "
                       "oracle/Makefile against oracle/cpp_standin"),
    )


def main(names):
    from conftest import load_pair  # the committed lossless input fixtures (== the .xyz files)

    if REF is None:
        sys.exit(f"no readable pglira/simpleICP checkout at {DEFAULT_REFERENCE}: set SIMPLEICP_REFERENCE")

    cli, driver = build()
    for name in names:
        fix, mov, flags = CONFIGS[name]
        data = {"dragon_k5000": "dragon", "bunny_maxit3": "bunny"}.get(name, name)
        X_fix, X_mov = load_pair(data)
        cli_screen = run_cli(cli, fix, mov, flags)
        j, api_screen = run_driver(driver, X_fix, X_mov, flags)
        # the committed input fixture is the .xyz file: the CLI (reading the file with the
        # reference's own parser) and the driver (reading the fixture) print the same screen
        assert cli_screen == api_screen, f"{name}: CLI and driver screens differ"
        assert j["stage_pass_equals_api"]
        p = dict(DEFAULTS)
        p.update(flags)
        np.savez_compressed(GOLD / f"cppref_{name}.npz", **pack(j, cli_screen, api_screen, p))
        print(f"{name}: {len(j['iterations'])} iterations, converged={j['converged']}, "
              f"kept={[it['n_kept'] for it in j['iterations']]}")
        print(cli_screen.split("Estimated transformation matrix H:")[1])


if __name__ == "__main__":
    main(sys.argv[1:] or list(CONFIGS))
