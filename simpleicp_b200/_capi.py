"""ctypes binding of libsicp_b200.so (the C ABI declared in include/sicp_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc; if that is impossible
an ImportError is raised, and creating an Engine without a CUDA device raises SicpError.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional, Sequence

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libsicp_b200.so"

SICP_OK, SICP_ERR_BAD_ARG, SICP_ERR_NO_OVERLAP, SICP_ERR_TOO_FEW_CORR = 0, 1, 2, 3
SICP_ERR_CUDA, SICP_ERR_SINGULAR, SICP_ERR_STATE = 4, 5, 6
ABI_VERSION = 2  # include/sicp_b200.h: SICP_ABI_VERSION
NN_AUTO, NN_GRID, NN_BRUTE = 0, 1, 2
SIGN_DGEEV, SIGN_CANONICAL = 0, 1

# every symbol include/sicp_b200.h declares (tests check the library exports all of them)
SYMBOLS = (
    "sicp_abi_version", "sicp_create", "sicp_destroy", "sicp_last_error", "sicp_set_option",
    "sicp_set_clouds", "sicp_set_selected", "sicp_select_in_range", "sicp_estimate_normals",
    "sicp_set_normals", "sicp_set_mov_normals", "sicp_get_knn", "sicp_match", "sicp_reject", "sicp_solve",
    "sicp_uncertainties", "sicp_run", "sicp_get_transform", "sicp_get_residuals", "sicp_iterate", "sicp_transform",
    "sicp_select_n_points", "sicp_register",
    "sicp_register_batch", "sicp_get_timings", "sicp_time_stages", "sicp_get_iteration", "sicp_get_phase_times",
    "sicp_xyz_load", "sicp_xyz_free", "sicp_xyz_save", "sicp_io_last_error",
)


class LsqParams(C.Structure):
    _fields_ = [("x0", C.c_double * 6), ("observed", C.c_double * 6),
                ("obs_weight", C.c_double * 6), ("distance_weight", C.c_double)]


class RunParams(C.Structure):
    _fields_ = [("min_planarity", C.c_double), ("min_change", C.c_double),
                ("max_iterations", C.c_int32), ("reserved", C.c_int32), ("lsq", LsqParams)]


class RegisterParams(C.Structure):
    _fields_ = [("correspondences", C.c_int64), ("neighbors", C.c_int32), ("reserved", C.c_int32),
                ("max_overlap_distance", C.c_double), ("run", RunParams)]


class IterRecord(C.Structure):
    _fields_ = [("n_kept", C.c_int64), ("median", C.c_double), ("mad", C.c_double),
                ("mean_dist", C.c_double), ("std_dist", C.c_double), ("x", C.c_double * 6),
                ("mean_res", C.c_double), ("std_res", C.c_double), ("distance_weight", C.c_double),
                ("lm_iterations", C.c_int32), ("n_bruteforce", C.c_int32)]


class RunResult(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("converged", C.c_int32), ("x", C.c_double * 6),
                ("H", C.c_double * 16), ("sigma", C.c_double * 6), ("n_residuals", C.c_int64),
                ("loop_ms", C.c_double)]


class Timings(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("upload_ms", "grid_mov_ms", "grid_fix_ms", "overlap_ms",
                                          "normals_ms", "match_ms", "reject_solve_ms",
                                          "transform_ms")] + [("kernel_launches", C.c_int64),
                                                            ("fused_iterations", C.c_int64),
                                                            ("rerun_iterations", C.c_int64)]


class PairResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("iterations", C.c_int32), ("converged", C.c_int32),
                ("n_selected", C.c_int32), ("n_kept", C.c_int64), ("H", C.c_double * 16),
                ("x", C.c_double * 6), ("sigma", C.c_double * 6), ("mean_res", C.c_double),
                ("std_res", C.c_double)]


class SicpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libsicp_b200 error {code}: {message}")
        self.code = code
        self.message = message


_lib = None


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if needed) the CUDA library.  Never falls back to a CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("SICP_B200_LIB")  # diagnostics: an experimental build of the same ABI
    if override:
        lib_path = Path(override)
        if not lib_path.exists():
            raise ImportError(f"SICP_B200_LIB={override} does not exist")
    else:
        lib_path = LIB_PATH
    if not override:
        if build_if_missing:
            # digest-checked and cheap when up to date: a library left over from older sources is
            # rebuilt instead of being loaded against newer ctypes struct layouts.  Where nvcc is
            # absent (a box that only received the built .so) the existing library is used and the
            # ABI version check below is the guard.
            from . import _build

            try:
                _build.build()
            except RuntimeError:
                if not LIB_PATH.exists():
                    raise ImportError(f"{LIB_PATH} is missing and cannot be built (nvcc not found)")
        elif not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing; run `python -m simpleicp_b200._build`")
    lib = C.CDLL(str(lib_path))
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.sicp_abi_version.restype = i32
    if lib.sicp_abi_version() != ABI_VERSION:
        raise ImportError(f"{lib_path} has ABI version {lib.sicp_abi_version()}, this binding needs "
                          f"{ABI_VERSION}: rebuild with `python -m simpleicp_b200._build --force`")
    lib.sicp_last_error.restype = C.c_char_p
    lib.sicp_last_error.argtypes = [vp]
    sigs = {
        "sicp_create": [i32, vp, C.POINTER(vp)],
        "sicp_destroy": [vp],
        "sicp_set_option": [vp, C.c_char_p, dbl],
        "sicp_set_clouds": [vp, vp, i64, vp, i64],
        "sicp_set_selected": [vp, vp, i64],
        "sicp_select_in_range": [vp, C.POINTER(dbl), dbl, vp, C.POINTER(i64)],
        "sicp_estimate_normals": [vp, i32, vp, vp, vp, vp],
        "sicp_set_normals": [vp, vp, vp, vp, vp],
        "sicp_set_mov_normals": [vp, vp, vp, vp, vp, C.c_double],
        "sicp_get_knn": [vp, vp, vp],
        "sicp_match": [vp, C.POINTER(dbl), vp, vp],
        "sicp_reject": [vp, dbl, vp, C.POINTER(i64), C.POINTER(dbl)],
        "sicp_solve": [vp, C.POINTER(LsqParams), C.POINTER(dbl), C.POINTER(dbl), vp,
                       C.POINTER(dbl), C.POINTER(dbl)],
        "sicp_uncertainties": [vp, C.POINTER(dbl)],
        "sicp_run": [vp, C.POINTER(RunParams), C.POINTER(RunResult), C.POINTER(IterRecord)],
        "sicp_get_transform": [vp, C.POINTER(C.c_double)],
        "sicp_get_residuals": [vp, vp, i64, C.POINTER(i64)],
        "sicp_iterate": [vp, C.POINTER(RunParams), C.POINTER(dbl), C.POINTER(IterRecord)],
        "sicp_transform": [vp, C.POINTER(dbl), vp],
        "sicp_select_n_points": [vp, i64, vp],
        "sicp_register": [vp, vp, i64, vp, i64, C.POINTER(RegisterParams), C.POINTER(RunResult),
                          C.POINTER(IterRecord), vp, C.POINTER(i64)],
        "sicp_register_batch": [vp, i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(vp), C.POINTER(i64),
                                C.POINTER(RegisterParams), C.POINTER(PairResult)],
        "sicp_get_timings": [vp, C.POINTER(Timings)],
        "sicp_time_stages": [vp, C.POINTER(RunParams), i32, i32, C.POINTER(dbl)],
        "sicp_get_iteration": [vp, C.POINTER(IterRecord), C.POINTER(dbl), vp, vp, vp],
        "sicp_get_phase_times": [vp, C.POINTER(dbl)],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = i32
    lib.sicp_xyz_load.argtypes = [C.c_char_p, C.POINTER(C.POINTER(dbl)), C.POINTER(i64)]
    lib.sicp_xyz_load.restype = i32
    lib.sicp_xyz_free.argtypes = [C.POINTER(dbl)]
    lib.sicp_xyz_free.restype = None
    lib.sicp_xyz_save.argtypes = [C.c_char_p, vp, i64, i32, i32]
    lib.sicp_xyz_save.restype = i32
    lib.sicp_io_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def read_xyz(path) -> np.ndarray:
    """Fast multi-threaded .xyz reader (x y z per line, '/'/'#' comment lines skipped); the
    doubles equal what np.genfromtxt parses from the same text."""
    lib = load_library()
    p = C.POINTER(C.c_double)()
    n = C.c_int64(0)
    rc = lib.sicp_xyz_load(str(path).encode(), C.byref(p), C.byref(n))
    if rc != SICP_OK:
        raise OSError(lib.sicp_io_last_error().decode())
    try:
        return np.ctypeslib.as_array(p, shape=(int(n.value), 3)).copy()
    finally:
        lib.sicp_xyz_free(p)


def write_xyz(path, X, decimals: int = 3, header: bool = True) -> None:
    """CloudCompare-style text file like the reference's PointCloud.write_xyz."""
    lib = load_library()
    X = np.ascontiguousarray(X, dtype=np.float64)
    if X.ndim != 2 or X.shape[1] != 3:
        raise ValueError("X must have 3 columns!")
    rc = lib.sicp_xyz_save(str(path).encode(), X.ctypes.data, X.shape[0], int(decimals), int(header))
    if rc != SICP_OK:
        raise OSError(lib.sicp_io_last_error().decode())


def _ptr(a) -> Optional[int]:
    """Raw address of a NumPy array or a torch tensor (host or CUDA); None passes NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(f"unsupported buffer type {type(a)}")


def _as_f64_xyz(X):
    """(n,3) float64 C-contiguous view/copy of a NumPy array or torch tensor."""
    if isinstance(X, np.ndarray) or not hasattr(X, "data_ptr"):
        X = np.ascontiguousarray(X, dtype=np.float64)
        if X.ndim != 2 or X.shape[1] != 3:
            raise ValueError("X must have 3 columns!")
        return X
    import torch

    if X.dim() != 2 or X.shape[1] != 3:
        raise ValueError("X must have 3 columns!")
    return X.to(torch.float64).contiguous()


def _d6(v: Sequence[float]):
    return (C.c_double * 6)(*[float(x) for x in v])


def _d16(H) -> "C.Array":
    H = np.asarray(H, dtype=np.float64).reshape(16)
    return (C.c_double * 16)(*H.tolist())


def current_stream_ptr(device: int) -> int:
    """torch's current CUDA stream on `device` (PyTorch owns streams and user-visible buffers);
    the legacy default stream when torch is not importable."""
    try:
        import torch

        if torch.cuda.is_available():
            return int(torch.cuda.current_stream(device).cuda_stream)
    except ImportError:
        pass
    return 0


def current_device() -> int:
    try:
        import torch

        if torch.cuda.is_available():
            return int(torch.cuda.current_device())
    except ImportError:
        pass
    return 0


def pinned_empty(shape, dtype) -> np.ndarray:
    """Host output buffer in pinned memory (through torch) so D2H copies run at link speed."""
    try:
        import torch

        if torch.cuda.is_available():
            tdt = {np.float64: torch.float64, np.float32: torch.float32, np.int64: torch.int64,
                   np.uint8: torch.uint8}[np.dtype(dtype).type]
            return torch.empty(shape, dtype=tdt, pin_memory=True).numpy()
    except (ImportError, RuntimeError):
        pass
    return np.empty(shape, dtype=dtype)


class Engine:
    """Thin object wrapper over one sicp_ctx."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.device = device
        st = current_stream_ptr(device) if stream is None else stream
        rc = self._lib.sicp_create(device, C.c_void_p(st), C.byref(self._h))
        if rc != SICP_OK:
            msg = self._lib.sicp_last_error(None).decode()
            self._h = C.c_void_p()
            raise SicpError(rc, msg)
        self.n_fix = self.n_mov = self.K = 0

    # -- plumbing
    def _check(self, rc: int):
        if rc != SICP_OK:
            raise SicpError(rc, self._lib.sicp_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.sicp_destroy(self._h)
            self._h = C.c_void_p()

    @property
    def alive(self) -> bool:
        return bool(getattr(self, "_h", None))

    def reset_options(self):
        """Back to the library defaults (used when a cached engine is handed out again)."""
        self._check(self._lib.sicp_set_option(self._h, b"defaults", 0.0))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_option(self, key: str, value: float):
        self._check(self._lib.sicp_set_option(self._h, key.encode(), float(value)))

    # -- stages
    def set_clouds(self, X_fix, X_mov):
        Xf, Xm = _as_f64_xyz(X_fix), _as_f64_xyz(X_mov)
        self.n_fix, self.n_mov = int(Xf.shape[0]), int(Xm.shape[0])
        self._check(self._lib.sicp_set_clouds(self._h, _ptr(Xf), self.n_fix, _ptr(Xm), self.n_mov))
        self.K = 0

    def set_selected(self, idx=None):
        if idx is None:
            self._check(self._lib.sicp_set_selected(self._h, None, self.n_fix))
            self.K = self.n_fix
        else:
            idx = np.ascontiguousarray(idx, dtype=np.int64)
            self._check(self._lib.sicp_set_selected(self._h, _ptr(idx), idx.size))
            self.K = int(idx.size)

    def select_in_range(self, H0, max_range: float) -> np.ndarray:
        keep = np.empty(self.K, dtype=np.uint8)
        n = C.c_int64(0)
        self._check(self._lib.sicp_select_in_range(self._h, _d16(H0), float(max_range), _ptr(keep),
                                                   C.byref(n)))
        return keep.astype(bool)

    def estimate_normals(self, neighbors: int, download: bool = True):
        if not download:
            self._check(self._lib.sicp_estimate_normals(self._h, int(neighbors), None, None, None, None))
            return None
        out = np.empty((4, self.K), dtype=np.float32)
        self._check(self._lib.sicp_estimate_normals(
            self._h, int(neighbors), out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data,
            out[3].ctypes.data))
        return out[0], out[1], out[2], out[3]

    def set_normals(self, nx, ny, nz, planarity):
        a = [np.ascontiguousarray(v, dtype=np.float32) for v in (nx, ny, nz, planarity)]
        for v in a:
            if v.size != self.K:
                raise ValueError("normal arrays must have one entry per selected point")
        self._check(self._lib.sicp_set_normals(self._h, *[_ptr(v) for v in a]))

    def set_mov_normals(self, nx, ny, nz, planarity, max_angle_deg=None):
        """Movable-side attributes (sicp_set_mov_normals): n_mov floats each, NaN = not estimated;
        ``set_mov_normals(None, None, None, None)`` clears them.  ``max_angle_deg`` switches the
        rejection by the angle between the normals on (degrees, like the facade's other angles)."""
        if nx is None and ny is None and nz is None and planarity is None:
            self._check(self._lib.sicp_set_mov_normals(self._h, None, None, None, None, -1.0))
            return
        a = [np.ascontiguousarray(v, dtype=np.float32) for v in (nx, ny, nz, planarity)]
        for v in a:
            if v.size != self.n_mov:
                raise ValueError("movable normal arrays must have one entry per movable point")
        ang = -1.0 if max_angle_deg is None else float(np.deg2rad(max_angle_deg))
        self._check(self._lib.sicp_set_mov_normals(self._h, *[_ptr(v) for v in a], ang))

    def get_knn(self, k: int):
        """Neighbour lists of the last estimate_normals (needs set_option("keep_knn", 1) before it)."""
        idx = np.empty((self.K, k), dtype=np.int64)
        d2 = np.empty((self.K, k), dtype=np.float64)
        self._check(self._lib.sicp_get_knn(self._h, _ptr(idx), _ptr(d2)))
        return idx, d2

    def match(self, H):
        idx = np.empty(self.K, dtype=np.int64)
        d = np.empty(self.K, dtype=np.float64)
        self._check(self._lib.sicp_match(self._h, _d16(H), _ptr(idx), _ptr(d)))
        return idx, d

    def reject(self, min_planarity: float):
        keep = np.empty(self.K, dtype=np.uint8)
        n = C.c_int64(0)
        stats = (C.c_double * 4)()
        self._check(self._lib.sicp_reject(self._h, float(min_planarity), _ptr(keep), C.byref(n), stats))
        return keep.astype(bool), int(n.value), list(stats)

    @staticmethod
    def lsq_params(x0, observed, obs_weight, distance_weight) -> LsqParams:
        p = LsqParams()
        p.x0 = _d6(x0)
        p.observed = _d6(observed)
        p.obs_weight = _d6(obs_weight)
        p.distance_weight = float("nan") if distance_weight is None else float(distance_weight)
        return p

    def solve(self, x0, observed, obs_weight, distance_weight, n_kept: int):
        p = self.lsq_params(x0, observed, obs_weight, distance_weight)
        x = (C.c_double * 6)()
        H = (C.c_double * 16)()
        stats = (C.c_double * 2)()
        w = C.c_double(0)
        res = np.empty(n_kept, dtype=np.float64)
        self._check(self._lib.sicp_solve(self._h, C.byref(p), x, H, _ptr(res), stats, C.byref(w)))
        return np.array(x), np.array(H).reshape(4, 4), res, list(stats), float(w.value)

    def uncertainties(self) -> np.ndarray:
        s = (C.c_double * 6)()
        self._check(self._lib.sicp_uncertainties(self._h, s))
        return np.array(s)

    @staticmethod
    def run_params(min_planarity, min_change, max_iterations, lsq: LsqParams) -> RunParams:
        p = RunParams()
        p.min_planarity = float(min_planarity)
        p.min_change = float(min_change)
        p.max_iterations = int(max_iterations)
        p.lsq = lsq
        return p

    def run(self, params: RunParams):
        out = RunResult()
        log = (IterRecord * int(params.max_iterations))()
        self._check(self._lib.sicp_run(self._h, C.byref(params), C.byref(out), log))
        n = C.c_int64(0)
        res = np.empty(int(out.n_residuals), dtype=np.float64)
        self._check(self._lib.sicp_get_residuals(self._h, _ptr(res), res.size, C.byref(n)))
        return out, [log[i] for i in range(out.iterations)], res

    def select_n_points(self, n: int, want_idx: bool = True):
        """PointCloud.select_n_points on the device; returns the resulting selection (int64)."""
        k = min(int(n), self.K if self.K else self.n_fix)
        idx = np.empty(k, dtype=np.int64) if want_idx else None
        self._check(self._lib.sicp_select_n_points(self._h, int(n), None if idx is None else _ptr(idx)))
        self.K = k
        return idx

    def register_fused(self, X_fix, X_mov, correspondences, neighbors, max_overlap_distance,
                       params: RunParams, transform_out=None):
        """SimpleICP.run as one library call (sicp_register): uploads, selection, normals, the
        loop and the final transform, with the movable upload overlapped with the fixed-side work."""
        Xf, Xm = _as_f64_xyz(X_fix), _as_f64_xyz(X_mov)
        self.n_fix, self.n_mov = int(Xf.shape[0]), int(Xm.shape[0])
        rp = RegisterParams()
        rp.correspondences = int(correspondences)
        rp.neighbors = int(neighbors)
        rp.max_overlap_distance = float(max_overlap_distance)
        rp.run = params
        out = RunResult()
        log = (IterRecord * int(params.max_iterations))()
        if transform_out is None:
            transform_out = pinned_empty((self.n_mov, 3), np.float64)
        nsel = C.c_int64(0)
        self._check(self._lib.sicp_register(self._h, _ptr(Xf), self.n_fix, _ptr(Xm), self.n_mov, C.byref(rp),
                                            C.byref(out), log, _ptr(transform_out), C.byref(nsel)))
        self.K = int(nsel.value)
        n = C.c_int64(0)
        res = np.empty(int(out.n_residuals), dtype=np.float64)
        self._check(self._lib.sicp_get_residuals(self._h, _ptr(res), res.size, C.byref(n)))
        return out, [log[i] for i in range(out.iterations)], res, transform_out

    def register_batch(self, pairs, correspondences, neighbors, params: RunParams, max_overlap_distance=-1.0):
        """sicp_register_batch: SimpleICP.run for every (X_fix, X_mov) of `pairs` with one set of
        kernel launches per stage for the whole batch.  Clouds are NumPy arrays (pinned ones
        upload at link speed) or CUDA tensors; nothing is copied on the host.  A finite
        `max_overlap_distance` > 0 filters every pair's fixed points as sicp_register does.
        Returns the ctypes array of PairResult (status per pair)."""
        n = len(pairs)
        keep = [(_as_f64_xyz(a), _as_f64_xyz(b)) for a, b in pairs]  # keeps converted copies alive
        fp = (C.c_void_p * n)(*[_ptr(a) for a, _ in keep])
        mp = (C.c_void_p * n)(*[_ptr(b) for _, b in keep])
        nf = (C.c_int64 * n)(*[int(a.shape[0]) for a, _ in keep])
        nm = (C.c_int64 * n)(*[int(b.shape[0]) for _, b in keep])
        rp = RegisterParams()
        rp.correspondences = int(correspondences)
        rp.neighbors = int(neighbors)
        rp.max_overlap_distance = float(max_overlap_distance)
        rp.run = params
        out = (PairResult * n)()
        self._check(self._lib.sicp_register_batch(self._h, n, fp, nf, mp, nm, C.byref(rp), out))
        return out

    def get_transform(self) -> np.ndarray:
        """The 4 x 4 transform the last run/solve applied to the movable cloud."""
        T = (C.c_double * 16)()
        self._check(self._lib.sicp_get_transform(self._h, T))
        return np.array(T).reshape(4, 4)

    def iterate(self, params: RunParams, x_in=None, want_record: bool = False):
        rec = IterRecord() if want_record else None
        self._check(self._lib.sicp_iterate(
            self._h, C.byref(params), None if x_in is None else _d6(x_in),
            C.byref(rec) if rec is not None else None))
        return rec

    def transform(self, H, out=None):
        """X_mov transformed by H.  `out` may be a CUDA torch tensor (n_mov, 3) float64."""
        if out is None:
            out = pinned_empty((self.n_mov, 3), np.float64)
        self._check(self._lib.sicp_transform(self._h, _d16(H), _ptr(out)))
        return out

    def time_stages(self, params: RunParams, reps: int, flush_l2: bool, outer_only: bool = False) -> dict:
        """Average device milliseconds per iteration of each kernel group (CUDA events).
        outer_only: only the events around the whole iteration (no bubbles from the inner ones)."""
        ms = (C.c_double * 4)()
        self._check(self._lib.sicp_time_stages(self._h, C.byref(params), int(reps),
                                               (1 if flush_l2 else 0) | (2 if outer_only else 0), ms))
        return {"match_grid": ms[0], "bruteforce_pass": ms[1], "reject_solve": ms[2], "iteration": ms[3]}

    def last_iteration(self):
        """What the last iterate / time_stages iteration computed, read back without running
        anything: (record, 4 x 4 cumulative transform, matched movable index, point-to-plane
        distance, keep flag), the arrays with one entry per selected point."""
        rec = IterRecord()
        T = (C.c_double * 16)()
        idx = np.empty(self.K, dtype=np.int64)
        d = np.empty(self.K, dtype=np.float64)
        keep = np.empty(self.K, dtype=np.uint8)
        self._check(self._lib.sicp_get_iteration(self._h, C.byref(rec), T, _ptr(idx), _ptr(d), _ptr(keep)))
        return rec, np.array(T).reshape(4, 4), idx, d, keep.astype(bool)

    def phase_times(self) -> list:
        """Diagnostics: block-0 phase stamps (us) of the last reject+solve kernel."""
        us = (C.c_double * 32)()
        self._check(self._lib.sicp_get_phase_times(self._h, us))
        return list(us)

    def timings(self) -> dict:
        t = Timings()
        self._check(self._lib.sicp_get_timings(self._h, C.byref(t)))
        return {n: getattr(t, n) for n, _ in Timings._fields_}
