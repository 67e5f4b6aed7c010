"""Batched registration of independent (X_fix, X_mov) pairs, sharded over GPUs.

Independent pairs share nothing (SURVEY.md §8e): each rank registers its static share on its
own GPU with the single-GPU pipeline and the only exchange is one all-gather of a fixed-size
record per pair — H (16 f64), iterations, kept correspondences, mean and std of the final
residuals — over NCCL (gloo on CPU-only hosts for the tests of the sharding logic).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

RECORD_LEN = 20  # H (16) + iterations + n_kept + mean + std


def shard_pairs(n_pairs: int, world_size: int, rank: int) -> List[int]:
    """Static round-robin assignment: pair i belongs to rank i % world_size."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("invalid rank / world_size")
    return list(range(rank, n_pairs, world_size))


def pack_record(H: np.ndarray, iterations: int, n_kept: int, mean: float, std: float) -> np.ndarray:
    r = np.empty(RECORD_LEN)
    r[:16] = np.asarray(H, dtype=float).reshape(16)
    r[16:] = (iterations, n_kept, mean, std)
    return r


def gather_records(local: np.ndarray, n_pairs: int, world_size: int, rank: int, dist=None,
                   device=None) -> np.ndarray:
    """All-gather the per-pair records.  `local` is (len(shard), RECORD_LEN) in shard order;
    returns (n_pairs, RECORD_LEN) in pair order on every rank."""
    if world_size == 1 or dist is None:
        out = np.zeros((n_pairs, RECORD_LEN))
        out[shard_pairs(n_pairs, 1, 0)] = local
        return out
    import torch

    per = (n_pairs + world_size - 1) // world_size  # equal-size slots, last ones may be padding
    buf = torch.full((per, RECORD_LEN), float("nan"), dtype=torch.float64, device=device)
    if local.shape[0]:
        buf[: local.shape[0]] = torch.from_numpy(np.ascontiguousarray(local)).to(buf.device)
    gathered = torch.empty((world_size * per, RECORD_LEN), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(gathered, buf)
    g = gathered.cpu().numpy().reshape(world_size, per, RECORD_LEN)
    out = np.zeros((n_pairs, RECORD_LEN))
    for r in range(world_size):
        ids = shard_pairs(n_pairs, world_size, r)
        out[ids] = g[r, : len(ids)]
    return out


def tile_slabs(X_fix: np.ndarray, X_mov: np.ndarray, n_slabs: int, overlap: float, axis: int = 0):
    """Cut a large pair into `n_slabs` overlapping slabs along `axis` (BASELINE.json configs[3],
    SURVEY.md section 8d C4): equal-count quantile cuts of the fixed cloud's coordinate, the same
    cuts for both clouds, every slab widened by `overlap` on both sides.  Each slab is an
    independent registration.  Returns a list of (X_fix_slab, X_mov_slab)."""
    if n_slabs < 1:
        raise ValueError("n_slabs must be >= 1")
    cuts = np.quantile(X_fix[:, axis], np.linspace(0.0, 1.0, n_slabs + 1))
    cuts[0], cuts[-1] = -np.inf, np.inf
    out = []
    for s in range(n_slabs):
        lo, hi = cuts[s] - overlap, cuts[s + 1] + overlap
        mf = (X_fix[:, axis] >= lo) & (X_fix[:, axis] < hi)
        mm = (X_mov[:, axis] >= lo) & (X_mov[:, axis] < hi)
        out.append((np.ascontiguousarray(X_fix[mf]), np.ascontiguousarray(X_mov[mm])))
    return out


# Engines (one CUDA stream + one libsicp_b200 context each) are kept between calls: creating a
# context and growing its device buffers costs far more than one small registration.
_ENGINES: dict = {}


def _engine_pool(device: int, n: int):
    import torch

    from . import _capi

    pool = _ENGINES.setdefault(int(device), [])
    with torch.cuda.device(device):
        while len(pool) < n:
            stream = torch.cuda.Stream(device=device)
            pool.append((stream, _capi.Engine(device, stream=int(stream.cuda_stream))))
    return pool


def close_engine_pool() -> None:
    """Release the engines simpleicp_batch keeps between calls."""
    for pool in _ENGINES.values():
        for _, eng in pool:
            eng.close()
    _ENGINES.clear()
    for eng in _BATCH_ENGINES.values():
        eng.close()
    _BATCH_ENGINES.clear()


def simpleicp_batch(
    pairs: Sequence[Tuple[np.ndarray, np.ndarray]] | Callable[[int], Tuple[np.ndarray, np.ndarray]],
    n_pairs: Optional[int] = None,
    *,
    rank: int = 0,
    world_size: int = 1,
    dist=None,
    device: int = 0,
    register_fn=None,
    concurrency: int = 4,
    on_error: str = "raise",
    batch_size: int = 64,
    engine: str = "batched",
    **run_kwargs,
) -> np.ndarray:
    """Register every pair; returns the (n_pairs, 20) record table on every rank.

    `pairs` is a sequence or a generator function i -> (X_fix, X_mov) (so that ranks only
    materialise their own share).  `register_fn` defaults to the GPU pipeline
    (simpleicp_b200.register on cuda:`device`); tests inject a stub to exercise the sharding and
    the collective on CPU.  On the GPU path `concurrency` engines, each on its own CUDA stream and
    driven by its own thread (the C calls release the GIL), work through the rank's share so the
    host round trips of small registrations overlap.

    `engine="batched"` (default) hands the rank's share to the library's batched engine in chunks
    of `batch_size` pairs (sicp_register_batch: one set of kernel launches per stage and per
    iteration for the whole chunk, a block per pair for reject + solve, per-pair stop flags),
    with or without the overlap filter (`max_overlap_distance`); pairs it does not cover (more
    than 4096 correspondences, debug output) and `engine="pool"` use the concurrent per-pair
    engines described above.

    A pair that cannot be registered (no overlap, fewer than 6 correspondences: ordinary
    data-dependent outcomes) gets a NaN record whose `iterations` field is minus the library's
    status code; every rank still takes part in the collective.  Afterwards `on_error="raise"`
    raises BatchError (same on every rank, `.table` holds the full table, `.failed` the pair
    numbers), `on_error="nan"` just returns the table.
    """
    if n_pairs is None:
        n_pairs = len(pairs)  # type: ignore[arg-type]
    get = pairs if callable(pairs) else (lambda i: pairs[i])  # type: ignore[index]
    mine = shard_pairs(n_pairs, world_size, rank)
    local = np.zeros((len(mine), RECORD_LEN))

    def record(res):
        last = res.records[res.iterations - 1]
        return pack_record(res.H, res.iterations, last["n_kept"], last["mean_res"], last["std_res"])

    def guarded(fn, Xf, Xm, **kw):
        try:
            return record(fn(Xf, Xm, **kw))
        except Exception as e:  # noqa: BLE001 — recorded per pair, reported after the gather
            code = getattr(getattr(e, "__cause__", None) or e, "code", None)
            msg = str(e)
            if code is None:
                code = 2 if "overlap" in msg else (3 if "correspondences" in msg else 99)
            messages.append(msg)
            return pack_record(np.full((4, 4), np.nan), -int(code), 0, np.nan, np.nan)

    messages: List[str] = []
    if register_fn is not None:
        for j, i in enumerate(mine):
            Xf, Xm = get(i)
            local[j] = guarded(register_fn, Xf, Xm, **run_kwargs)
    elif engine == "batched" and _batchable(run_kwargs):
        _run_batched(get, mine, local, device, batch_size, run_kwargs, messages)
    else:
        import threading

        import torch

        from .simpleicp import register

        run_kwargs.setdefault("want_normals", False)  # one fused sicp_register call per pair
        n_workers = max(1, min(concurrency, len(mine)))
        errors = []
        pool = _engine_pool(device, n_workers)
        todo, lock = iter(range(len(mine))), threading.Lock()

        def worker(w):
            try:
                with torch.cuda.device(device):
                    _, eng = pool[w]
                    while True:
                        with lock:  # dynamic hand-out: iteration counts (3 .. max_iterations) vary a lot
                            j = next(todo, None)
                        if j is None:
                            break
                        Xf, Xm = get(mine[j])
                        local[j] = guarded(register, Xf, Xm, engine=eng, **run_kwargs)
            except Exception as e:  # surfaced after the join
                errors.append(e)

        threads = [threading.Thread(target=worker, args=(w,)) for w in range(n_workers)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:  # not a per-pair outcome (bad generator, lost device): NaN for what is missing
            messages.append(repr(errors[0]))
            done = np.isfinite(local[:, 16]) & (local[:, 16] != 0)
            local[~done] = pack_record(np.full((4, 4), np.nan), -99, 0, np.nan, np.nan)
    dev = None
    if dist is not None and world_size > 1:
        import torch

        dev = torch.device("cuda", device) if dist.get_backend() == "nccl" else torch.device("cpu")
    table = gather_records(local, n_pairs, world_size, rank, dist, dev)
    failed = np.flatnonzero(table[:, 16] < 0)
    if failed.size and on_error == "raise":
        raise BatchError(table, failed, messages)
    return table


_BATCH_KEYS = {"correspondences", "neighbors", "min_planarity", "min_change", "max_iterations",
               "distance_weights", "rbp_observed_values", "rbp_observation_weights", "max_overlap_distance",
               "want_normals"}


def _batchable(kw) -> bool:
    """Can the batched engine serve these run() arguments?  (One block per pair: at most 4096
    correspondences; nothing that needs per-pair host interaction.)"""
    if set(kw) - _BATCH_KEYS:
        return False
    return int(kw.get("correspondences", 1000)) <= 4096 and not kw.get("want_normals", False)


_BATCH_ENGINES: dict = {}


def _run_batched(get, mine, local, device, batch_size, kw, messages):
    import torch

    from . import _capi
    from .simpleicp import _check_arguments, _observed_in_radians

    dw = kw.get("distance_weights", 1)
    obs_v = kw.get("rbp_observed_values", (0.0,) * 6)
    obs_w = kw.get("rbp_observation_weights", (0.0,) * 6)
    _check_arguments(dw, obs_v, obs_w)
    obs = _observed_in_radians(obs_v)
    with torch.cuda.device(device):
        eng = _BATCH_ENGINES.get(int(device))
        if eng is None or not eng.alive:
            eng = _BATCH_ENGINES[int(device)] = _capi.Engine(int(device))
        lsq = eng.lsq_params(obs, obs, [float(w) for w in obs_w], dw)
        params = eng.run_params(kw.get("min_planarity", 0.3), kw.get("min_change", 1.0),
                                kw.get("max_iterations", 100), lsq)
        for lo in range(0, len(mine), max(1, int(batch_size))):
            ids = range(lo, min(lo + max(1, int(batch_size)), len(mine)))
            pairs = [get(mine[j]) for j in ids]
            res = eng.register_batch(pairs, kw.get("correspondences", 1000), kw.get("neighbors", 10), params,
                                     float(kw.get("max_overlap_distance", np.inf)))
            for j, r in zip(ids, res):
                if r.status == 0:
                    local[j] = pack_record(np.array(r.H).reshape(4, 4), r.iterations, r.n_kept, r.mean_res, r.std_res)
                else:
                    messages.append(f"pair {mine[j]}: library status {r.status}")
                    local[j] = pack_record(np.full((4, 4), np.nan), -int(r.status), 0, np.nan, np.nan)


class BatchError(RuntimeError):
    """Some pairs of a batch could not be registered; `.table` is the complete record table."""

    def __init__(self, table, failed, messages):
        codes = sorted({int(-table[i, 16]) for i in failed})
        super().__init__(f"{len(failed)} of {len(table)} pairs failed (pairs {failed[:8].tolist()}"
                         f"{' ...' if len(failed) > 8 else ''}, status codes {codes})"
                         + (f"; first local message: {messages[0]}" if messages else ""))
        self.table, self.failed, self.messages = table, failed, messages
