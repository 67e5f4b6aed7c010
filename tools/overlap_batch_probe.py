"""Partial-overlap batch (GPU): the batched engine against the pool of per-pair engines on pairs
that only partly overlap, with the overlap filter on.

Workload: 64 pairs of 100 000 points like C5 (30 x 30 m patches of synthetic.surface, the C5
rigid transforms), but every movable patch is sampled 10 m further along x before the inverse
transform, so about 2/3 of each fixed patch overlaps; max_overlap_distance = 1.0.  Both engines
run in one process on the same pinned pairs, alternating, after a warm-up of each.

    python tools/overlap_batch_probe.py [--pairs 64] [--points 100000] [--rounds 5] [--out FILE]
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import simpleicp_b200 as sb  # noqa: E402
from simpleicp_b200 import synthetic  # noqa: E402


def make_pairs(n_pairs, n_pts, shift):
    import torch

    x = synthetic.c5_transforms(max(512, n_pairs))
    out = []
    for i in range(n_pairs):
        Xf = synthetic.surface(n_pts, 10_000 + 2 * i, extent=30.0)
        Xm = synthetic.apply_H(synthetic.surface(n_pts, 10_001 + 2 * i, extent=30.0, x0=shift),
                               np.linalg.inv(synthetic.H_from_rbp(x[i])))
        out.append(tuple(torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (Xf, Xm)))
    return out


def card():
    import torch

    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True, timeout=30).stdout.strip().splitlines()
        info["nvidia_smi"] = q[0] if q else None
    except Exception as e:  # noqa: BLE001 — reported, not fatal
        info["nvidia_smi"] = f"unavailable: {e!r}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--shift", type=float, default=10.0)
    ap.add_argument("--distance", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU")
    pairs = make_pairs(args.pairs, args.points, args.shift)
    kw = dict(max_overlap_distance=args.distance, on_error="nan", batch_size=args.pairs)

    def run(engine):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        table = sb.simpleicp_batch(pairs, engine=engine, **kw)
        torch.cuda.synchronize()
        return table, time.perf_counter() - t0

    for engine in ("batched", "pool"):  # warm-up: module loads, buffer growth
        run(engine)
    times = {"batched": [], "pool": []}
    tables = {}
    for _ in range(args.rounds):
        for engine in ("batched", "pool"):
            tables[engine], dt = run(engine)
            times[engine].append(dt)
    tm = sb.batch._BATCH_ENGINES[0].timings()
    a, b = tables["batched"], tables["pool"]
    ok = (a[:, 16] > 0) & (b[:, 16] > 0)
    res = {
        "workload": f"{args.pairs} pairs x {args.points} points, movable patch shifted {args.shift} m in x, "
                    f"max_overlap_distance={args.distance}, simpleicp_batch on pinned host arrays",
        "card": card(),
        "rounds": args.rounds,
        "seconds": times,
        "pairs_per_s": {k: args.pairs / statistics.median(v) for k, v in times.items()},
        "pairs_per_s_range": {k: [args.pairs / max(v), args.pairs / min(v)] for k, v in times.items()},
        "failed": {"batched": int((a[:, 16] < 0).sum()), "pool": int((b[:, 16] < 0).sum())},
        "tables_equal": {
            "status_equal": bool(np.array_equal(a[:, 16] < 0, b[:, 16] < 0)),
            "iterations_and_kept_equal": bool(np.array_equal(a[ok, 16:18], b[ok, 16:18])),
            "max_abs_dH": float(np.abs(a[ok, :16] - b[ok, :16]).max()) if ok.any() else None,
        },
        "mean_iterations": float(a[ok, 16].mean()) if ok.any() else None,
        "batched_timings_last_call": tm,
    }
    print(json.dumps(res, indent=1))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
