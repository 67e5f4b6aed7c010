import ast
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
GOLD = REPO / "tests" / "golden"

TRAVEL = ("dragon", "bunny", "multisensor", "webots")
ALIAS = {"dragon_observed": "dragon", "dragon_movnormals": "dragon"}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def decode_cloud(blob, n, scale):
    """Inverse of oracle/make_golden.py::encode_cloud (delta + zig-zag + byte planes + LZMA)."""
    import lzma

    planes = np.frombuffer(lzma.decompress(blob.tobytes()), dtype=np.uint8).reshape(3, 4, n)
    Z = np.ascontiguousarray(planes.transpose(0, 2, 1)).view(np.uint32).reshape(3, n).T
    D = (Z >> 1).astype(np.int64) ^ -(Z & 1).astype(np.int64)
    return np.cumsum(D, axis=0) / float(scale)


_PAIR_CACHE = {}


def load_pair(name):
    """Input clouds of a reference test config, stored losslessly as scaled int32 (the two
    1.3 M-point lidar pairs additionally delta-coded and LZMA-compressed)."""
    name = ALIAS.get(name, name)
    if name in _PAIR_CACHE:
        return _PAIR_CACHE[name]
    z = np.load(GOLD / f"data_{name}.npz")
    if "codec" in z.files:
        pair = (decode_cloud(z["fix_blob"], int(z["n_fix"]), int(z["fix_scale"])),
                decode_cloud(z["mov_blob"], int(z["n_mov"]), int(z["mov_scale"])))
        _PAIR_CACHE[name] = pair  # decoding takes seconds: keep for the session
        return pair
    s = float(z["scale"])
    return z["fix"] / s, z["mov"] / s


def load_golden(name):
    g = dict(np.load(GOLD / f"ref_{name}.npz"))
    inf = np.inf  # noqa: F841  (used by eval below)
    g["kwargs"] = eval(str(g["kwargs_repr"]), {"inf": np.inf, "nan": np.nan})
    return g


def has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def gpu():
    if not has_gpu():
        pytest.skip("no CUDA device")
    return True
