#!/usr/bin/env python
"""bench.py — correspondences/sec per ICP iteration on the BASELINE.json C3 workload.

    python bench.py --gpus 1 --steps 20 --warmup 3                 # B200 arm
    python bench.py --impl reference --steps 20 --warmup 3          # CPU arm (oracle port)
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs DIR   # + what the last timed step computed
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W       # weak scaling

Workload (SURVEY.md §8d, BASELINE.json configs[2]): synthetic 1M <-> 1M point pair (tilted,
undulating plane with 1 cm noise), correspondences = 100 000, all other reference defaults.
One STEP = one ICP iteration of the hot path: nearest-neighbour match of the 100 000 selected
fixed points into the 1M-point movable cloud + point-to-plane distances, planarity / median-MAD
rejection, 6-DoF least-squares solve, residual statistics and stop-rule evaluation.

value      = K * steps / (sum of the per-step device times); every step starts with a COLD L2
             (a 256 MiB buffer is overwritten between steps, outside the timed intervals),
             inputs resident in HBM.  Per-step times are CUDA-event intervals on the launching
             stream; with N ranks the slowest rank's total is used.
e2e        = the same metric through the public API call  simpleicp_b200.register(X_fix, X_mov,
             correspondences=K)  (what simpleicp() runs) on pinned HOST arrays: upload, grid
             builds, normals, the whole iteration loop, final transform and download are all
             inside the timed region.  Beside it: the same call on pageable arrays with the
             library's default engine (e2e_simpleicp_pageable) and the drop-in class
             SimpleICP().run() on pandas point clouds (e2e_class_run).
N > 1      = independent pairs, one per GPU (weak scaling); the only collective is ONE NCCL
             all-gather of the per-pair result records after the last registration.
c4 / c5    = BASELINE configs[3] and [4] measured through their public entry points
             (tile_slabs + register per slab; simpleicp_batch), spread over the N ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

METRIC = "correspondences/sec per ICP iter (1M<->1M pts)"
UNIT = "corr/s"


def workload_string(n: int, K: int) -> str:
    """Identical in both arms (the driver compares the strings)."""
    return (f"C3 synthetic surface pair {n}<->{n} per GPU, correspondences={K}, neighbors=10, "
            "min_planarity=0.3 (BASELINE.json configs[2])")


def make_pair(n: int, rank: int):
    """C3 generator (SURVEY.md §8d); rank r uses seeds shifted by 10 r (independent pairs)."""
    from simpleicp_b200 import synthetic

    return synthetic.c3_pair(n, shift=10 * rank)


def make_c5_pairs(ids, n_pts: int = 100_000, pinned: bool = False, total: int = 512):
    """Pairs `ids` of the C5 batch (SURVEY.md §8d) as host arrays (optionally pinned)."""
    from simpleicp_b200 import synthetic

    out = []
    for i in ids:
        Xf, Xm, _ = synthetic.c5_pair(i, n_pts, total)
        if pinned:
            import torch

            Xf, Xm = torch.from_numpy(Xf).pin_memory().numpy(), torch.from_numpy(Xm).pin_memory().numpy()
        out.append((Xf, Xm))
    return out


def algorithmic_bytes(n_mov: int, K: int, n_kept: int):
    """SURVEY.md §8(d): B_iter = 16 N_mov + 60 K + 48 K_kept, split by kernel."""
    match = 16 * n_mov + 44 * K          # cloud stream + query + normal + (idx, dist) out
    reject_solve = 16 * K + 48 * n_kept  # select/compaction + fp64 gathers for the solve
    return match, reject_solve


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples while the benchmark runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index: int):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            p = [v.strip() for v in line.split(",")]
            if len(p) >= 7:
                try:
                    self.samples.append((time.time(), float(p[0]), float(p[1]), p[3:7]))
                except ValueError:
                    pass

    def summary(self, t0: float, t1: float):
        if self.proc is not None:
            self.proc.terminate()
        sel = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({self.NAMES[i] for s in sel for i, v in enumerate(s[3]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median([s[1] for s in sel])), "sm_max_mhz": sel[0][2],
                "reasons": reasons, "samples": len(sel)}


# ------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------
def _reference_worker(args_tuple):
    """One reference process: the oracle port on ITS pair with its share of the host cores."""
    n, K, warmup, steps, pair_id, workers = args_tuple
    from oracle import simpleicp_oracle as O

    O.WORKERS = workers
    X_fix, X_mov, _ = _oracle_pair(O, n, pair_id)
    tr = O.Trace(light=True)
    n_it = warmup + steps
    t0 = time.perf_counter()
    O.simpleicp(X_fix, X_mov, correspondences=K, min_change=0.0, max_iterations=n_it, trace=tr)
    total = time.perf_counter() - t0
    return tr.iter_seconds, total, tr.timings.get("normals")


def _oracle_pair(O, n, pair_id):
    H_true = O.rbp_to_H([np.deg2rad(0.3), np.deg2rad(-0.2), np.deg2rad(0.5), 0.15, -0.10, 0.05])
    X_fix = O.surface(n, 1234 + 10 * pair_id)
    X_mov = O.transform_by_H(O.surface(n, 5678 + 10 * pair_id), np.linalg.inv(H_true))
    return X_fix, X_mov, H_true


def run_reference(args):
    """CPU arm: the oracle port of the reference's algorithm (NumPy + SciPy cKDTree + TRF), the
    same SciPy calls the reference makes, on this host's cores.  One step = one ICP iteration.
    With --gpus N it registers N independent pairs side by side (N processes, the cores split
    between them) — the like-for-like counterpart of the N-GPU weak-scaling run."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_proc = max(1, int(args.gpus))
    workers = max(1, cores // n_proc)
    jobs = [(args.points, args.correspondences, args.warmup, args.steps, r, workers if n_proc > 1 else -1)
            for r in range(n_proc)]
    t0 = time.perf_counter()
    if n_proc == 1:
        results = [_reference_worker(jobs[0])]
    else:
        import multiprocessing as mp

        with mp.get_context("spawn").Pool(n_proc) as pool:
            results = pool.map(_reference_worker, jobs)
    wall = time.perf_counter() - t0
    n_it = args.warmup + args.steps
    loops = [float(np.sum(it_s[args.warmup:])) for it_s, _, _ in results]
    totals = [tot for _, tot, _ in results]
    steps = len(results[0][0][args.warmup:])
    value = n_proc * args.correspondences * steps / max(loops)
    e2e = n_proc * args.correspondences * n_it / max(totals)
    sample = (f"{n_it} ICP iterations (first {args.warmup} untimed) of the oracle port on "
              f"{n_proc} full C3 pair(s) side by side ({n_proc} process(es), {workers if n_proc > 1 else cores} cKDTree "
              f"worker threads each), K={args.correspondences}; tree build, transforms, eig loop and TRF solve are "
              "single-threaded as in the reference")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * max(loops) / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_string(args.points, args.correspondences), "l2": "n/a (CPU)",
                   "pairs_side_by_side": n_proc},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "setup_s": {"normals": results[0][2], "total": max(totals), "wall": wall},
    }), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local: int):
    """Pinned buffers are first-touched by this process: run it on the GPU's own NUMA node."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={local}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out  # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text())
        if node < 0:
            return None
        cpus = []
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:  # noqa: BLE001 — best effort, containers often hide the topology
        return None


def run_c4(sb, eng, rank, world, local):
    """BASELINE configs[3]: the airborne pair cut into 8 overlapping slabs along x (25 m overlap,
    SURVEY.md §8d C4), one registration per slab, slabs dealt round-robin to the ranks."""
    import torch

    fixture = REPO / "tests" / "golden" / "data_airborne.npz"
    if not fixture.exists():
        return None
    sys.path.insert(0, str(REPO / "tests"))
    from conftest import load_golden, load_pair

    X_fix, X_mov = load_pair("airborne")
    H_ref = load_golden("airborne")["H"]
    slabs = sb.tile_slabs(X_fix, X_mov, 8, overlap=25.0)
    mine = list(range(rank, 8, world))
    pinned = [(torch.from_numpy(slabs[s][0]).pin_memory().numpy(), torch.from_numpy(slabs[s][1]).pin_memory().numpy())
              for s in mine]
    out = []
    for (Xf, Xm) in pinned[:1]:
        sb.register(Xf, Xm, engine=eng, want_normals=False)  # warm-up (buffer growth)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s, (Xf, Xm) in zip(mine, pinned):
        t1 = time.perf_counter()
        r = sb.register(Xf, Xm, engine=eng, want_normals=False)
        out.append({"slab": s, "n_fix": int(Xf.shape[0]), "n_mov": int(Xm.shape[0]), "iterations": r.iterations,
                    "ms": 1e3 * (time.perf_counter() - t1), "H_frobenius_vs_whole_cloud_reference": float(np.linalg.norm(r.H - H_ref))})
    torch.cuda.synchronize()
    return {"slabs": out, "seconds": time.perf_counter() - t0}


def run_c5(sb, rank, world, local, dist, pairs_per_gpu, n_pts):
    """BASELINE configs[4]: 64 x N independent 100k-point pairs (512 on 8 GPUs), through
    simpleicp_batch (batched engine: one launch set per stage and iteration for a rank's share,
    NCCL all-gather of the records)."""
    import torch

    n_pairs = pairs_per_gpu * world
    mine = list(range(rank, n_pairs, world))
    local_pairs = dict(zip(mine, make_c5_pairs(mine, n_pts, pinned=True, total=max(512, n_pairs))))
    get = lambda i: local_pairs[i]  # noqa: E731 — only this rank's share is ever asked for
    kw = dict(rank=rank, world_size=world, dist=dist if world > 1 else None, device=local, on_error="nan",
              batch_size=pairs_per_gpu)
    sb.simpleicp_batch(get, n_pairs, **kw)  # warm-up (buffer growth)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    table = sb.simpleicp_batch(get, n_pairs, **kw)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    from simpleicp_b200 import synthetic

    x_true = synthetic.c5_transforms(max(512, n_pairs))
    errs = [float(np.linalg.norm(table[i, :16].reshape(4, 4) - synthetic.H_from_rbp(x_true[i]))) for i in range(n_pairs)
            if table[i, 16] > 0]
    return {"pairs": n_pairs, "points_per_cloud": n_pts, "seconds": dt, "pairs_per_s": n_pairs / dt,
            "failed": int((table[:, 16] < 0).sum()), "mean_iterations": float(table[table[:, 16] > 0, 16].mean()),
            "max_H_frobenius_vs_H_true": max(errs) if errs else None,
            "api": "simpleicp_b200.simpleicp_batch(pairs, engine='batched') on pinned host arrays, records all-gathered"}


# per-correspondence entries written by --dump-outputs (28 bytes each with the sample index): a
# larger K is sampled with a fixed seed so that a dump stays under 64 MB
DUMP_MAX_ENTRIES = 1 << 21


def dump_outputs(out_dir: str, eng) -> None:
    """What the last timed step (one ICP iteration) computed, as the arrays a caller of the
    iteration receives: the cumulative transform H and parameters x after it, its residual
    statistics and, per selected fixed point, the matched movable index, the point-to-plane
    distance and the keep flag of the rejection.  Inputs are seeded, so two builds run with the
    same arguments can be compared file by file."""
    rec, H, nn_idx, dist, keep = eng.last_iteration()
    K = nn_idx.size
    sample = np.arange(K)
    if K > DUMP_MAX_ENTRIES:
        sample = np.sort(np.random.default_rng(0).choice(K, DUMP_MAX_ENTRIES, replace=False))
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {
        "H": H,
        "x": np.array(rec.x, dtype=np.float64),
        "n_kept": np.array([rec.n_kept], dtype=np.float64),
        # median and MAD of the distances, their mean and std, mean and std of the residuals after
        # the solve, distance weight of the least-squares problem
        "stats": np.array([rec.median, rec.mad, rec.mean_dist, rec.std_dist, rec.mean_res, rec.std_res,
                           rec.distance_weight], dtype=np.float64),
        "sample_index": sample.astype(np.float64),
        "match_index": nn_idx[sample].astype(np.float64),
        "distance": dist[sample],
        "kept": keep[sample].astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def _trace(msg):
    if os.environ.get("SICP_BENCH_TRACE"):
        print(f"[bench rank {os.environ.get('RANK', '0')} t={time.time() % 1000:.1f}] {msg}", file=sys.stderr, flush=True)


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local) if world > 1 else None

    _trace("numa bound, importing package")
    import simpleicp_b200 as sb
    from simpleicp_b200 import _capi, batch

    torch.cuda.set_device(local)
    if world > 1:
        # stdout carries exactly one JSON line: whatever NCCL logs (version banner, INFO lines when
        # the caller asks for them) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # (this image exports NCCL_DEBUG=VERSION, whose banner ignores NCCL_DEBUG_FILE; WARN has none)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    _trace("process group ready")
    K, n = args.correspondences, args.points

    X_fix, X_mov, H_true = make_pair(n, rank)
    Xf_pin = torch.from_numpy(X_fix).pin_memory()
    Xm_pin = torch.from_numpy(X_mov).pin_memory()
    out_pin = torch.empty((n, 3), dtype=torch.float64).pin_memory()

    _trace("inputs pinned")
    sampler = ClockSampler(local) if rank == 0 else None
    eng = _capi.Engine(local)

    # ---- setup (untimed for `value`): resident inputs, grid, selection, normals
    eng.set_clouds(Xf_pin.numpy(), Xm_pin.numpy())
    idx = sb.pointcloud.subsample_indices(n, K).astype(np.int64)
    eng.set_selected(idx)
    eng.estimate_normals(10)
    lsq = eng.lsq_params(np.zeros(6), np.zeros(6), np.zeros(6), 1.0)
    params = eng.run_params(0.3, 1.0, 100, lsq)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    _trace("setup done")
    # ---- warm-up: a real registration's worth of iterations brings the loop to its steady state
    # (the state every iteration after the first few of a registration is in), then the timed
    # region (cold L2 before every step)
    rec = eng.iterate(params, x_in=np.zeros(6), want_record=True)
    for _ in range(max(args.warmup - 1, 11)):
        rec = eng.iterate(params, want_record=True)
    launches0 = eng.timings()["kernel_launches"]
    barrier()
    # the K timed steps: one CUDA-event pair around each whole iteration (cold L2 before each)
    st_outer = eng.time_stages(params, args.steps, True, outer_only=True)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)
    launches = eng.timings()["kernel_launches"] - launches0
    # the per-kernel split of the same step, from a second set of steps with events between the
    # kernels (those events cost a few microseconds of stream bubbles, hence not in `value`)
    st = eng.time_stages(params, args.steps, True)
    st["iteration_with_inner_events"] = st["iteration"]
    st["iteration"] = st_outer["iteration"]
    path = eng.phase_times()[28]
    total_ms = st_outer["iteration"] * args.steps
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * K * args.steps / (total_ms * 1e-3)
    rec = eng.iterate(params, want_record=True)
    n_kept = int(rec.n_kept)

    _trace("cold timing done")
    # ---- same loop, warm L2, iterations queued back to back with no host sync (what sicp_run does)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        eng.iterate(params)
    e1.record()
    torch.cuda.synchronize()
    warm_ms = e0.elapsed_time(e1) / args.steps
    eng.iterate(params, want_record=True)  # lets the engine see that no query needs the fallback
    st_warm = eng.time_stages(params, args.steps, False)

    # ---- sustained load for the clock record (~1.5 s of the same step)
    t_load0 = time.time()
    while time.time() - t_load0 < 1.5:
        for _ in range(200):
            eng.iterate(params)
        torch.cuda.synchronize()
    t_load1 = time.time()

    _trace("clock window done")
    # ---- end to end through the public API on pinned host arrays
    def one_e2e():
        return sb.register(Xf_pin.numpy(), Xm_pin.numpy(), correspondences=K, engine=eng,
                           transform_out=out_pin.numpy(), want_normals=False)  # = what simpleicp() does

    one_e2e()  # warm-up (allocations)
    barrier()
    t0 = time.perf_counter()
    its = 0
    for _ in range(args.e2e_steps):
        res = one_e2e()
        its += res.iterations
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    tm = eng.timings()
    # the one collective of the multi-GPU run: the result records, gathered once after the last
    # registration (inside the reported time)
    if world > 1:
        last = res.records[res.iterations - 1]
        local_rec = batch.pack_record(res.H, res.iterations, last["n_kept"], last["mean_res"], last["std_res"])[None]
        tg = time.perf_counter()
        batch.gather_records(local_rec, world, world, rank, dist, torch.device("cuda", local))
        e2e_s += time.perf_counter() - tg
        t = torch.tensor([e2e_s, float(its)], dtype=torch.float64, device="cuda")
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        e2e_s_max, its_total = float(tmax[0].item()), float(tsum[1].item())
    else:
        e2e_s_max, its_total = e2e_s, float(its)
    e2e_value = K * its_total / e2e_s_max
    dH_true = float(np.linalg.norm(res.H - H_true))

    _trace("e2e done")
    # ---- the north-star API as a user calls it: pageable arrays, no engine argument; and the class
    extra = {}
    if world == 1:
        for _ in range(2):  # warm-up: default engine creation, pinned result buffers, upload workers
            H1, X1, rbp1, r1 = sb.simpleicp(X_fix, X_mov, correspondences=K)
        t_pg = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            H1, X1, rbp1, r1 = sb.simpleicp(X_fix, X_mov, correspondences=K)
            torch.cuda.synchronize()
            t_pg.append(time.perf_counter() - t0)
        dt = float(np.median(t_pg))
        extra["e2e_simpleicp_pageable"] = {
            "ms_per_registration": 1e3 * dt, "ms_each": [round(1e3 * t, 3) for t in t_pg],
            "value": K * res.iterations / dt, "unit": UNIT,
            "api": "simpleicp_b200.simpleicp(X_fix, X_mov, correspondences=K) on pageable NumPy arrays, library-owned engine"}
        pc_fix = sb.PointCloud(X_fix, columns=["x", "y", "z"])
        icp = sb.SimpleICP(verbose=False)
        t_cls = []
        for _ in range(2):
            pc_fix.select_all_points()
            for col in ("nx", "ny", "nz", "planarity"):
                if col in pc_fix:
                    del pc_fix[col]
            pc_mov = sb.PointCloud(X_mov, columns=["x", "y", "z"], copy=True)
            icp.add_point_clouds(pc_fix, pc_mov)
            t0 = time.perf_counter()
            Hc, Xc, rbpc, rc = icp.run(correspondences=K)
            t_cls.append(time.perf_counter() - t0)
        extra["e2e_class_run"] = {
            "ms_per_registration": 1e3 * min(t_cls), "value": K * res.iterations / min(t_cls), "unit": UNIT,
            "H_equals_functional_api": bool(np.array_equal(Hc, H1)),
            "api": "SimpleICP().add_point_clouds(PointCloud, PointCloud); .run(correspondences=K) — pandas containers, "
                   "normals stored back as columns, pc_mov transformed in place"}

    # ---- the linearised variant (SURVEY.md section 8f rank 3) on the same pair
    variants = None
    if world == 1:
        eng.set_option("variant", 1)
        eng.iterate(params, x_in=np.zeros(6), want_record=True)
        for _ in range(max(args.warmup, 11)):
            eng.iterate(params, want_record=True)
        st_lin = eng.time_stages(params, args.steps, True)
        t0 = time.perf_counter()
        rl = sb.simpleicp_linearized(Xf_pin.numpy(), Xm_pin.numpy(), correspondences=K, engine=eng,
                                     transform_out=out_pin.numpy())
        torch.cuda.synchronize()
        lin_s = time.perf_counter() - t0
        eng.set_option("variant", 0)
        variants = {"linearized": {
            "ms_per_step": st_lin["iteration"], "value": K / (st_lin["iteration"] * 1e-3), "unit": UNIT,
            "kernels_ms_cold_l2": st_lin, "e2e_ms_per_registration": 1e3 * lin_s, "e2e_iterations": rl.iterations,
            "H_frobenius_vs_H_true": float(np.linalg.norm(rl.T - H_true)),
            "api": "simpleicp_b200.simpleicp_linearized(X_fix, X_mov, correspondences=K, engine=<reused>)"}}

    _trace("variants done")
    # ---- BASELINE configs[3] and [4] through their public entry points (all ranks take part)
    c4 = c5 = None
    if not args.no_c4c5:
        try:
            c4 = run_c4(sb, eng, rank, world, local)
            if c4 is not None and world > 1:
                gathered = [None] * world
                dist.all_gather_object(gathered, c4)
                c4 = {"slabs": sorted(sum((g["slabs"] for g in gathered), []), key=lambda s: s["slab"]),
                      "seconds": max(g["seconds"] for g in gathered)}
            if c4 is not None:
                c4["config"] = "airborne_lidar1/2 (1 342 906 points each) cut into 8 slabs along x, 25 m overlap, defaults"
                c4["slabs_per_s"] = 8 / c4["seconds"]
            c5 = run_c5(sb, rank, world, local, dist, args.c5_pairs_per_gpu, args.c5_points)
        except Exception as e:  # noqa: BLE001 — the headline line must not depend on the side configs
            c5 = c5 or {"error": repr(e)}

    _trace("c4/c5 done")
    if rank != 0:
        eng.close()
        batch.close_engine_pool()
        if world > 1:
            dist.destroy_process_group()
        return

    clocks = sampler.summary(t_load0, t_load1)
    clocks["window"] = "1.5 s of back-to-back steps right after the timed region"

    # ---- roofline of the dominant kernel (cold-L2 per-launch time measured above)
    b_match, b_rs = algorithmic_bytes(n, K, n_kept)
    peaks = {}
    try:
        peaks = json.loads((REPO / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    rs_name = {2.0: "k_rs_fused", 1.0: "k_reject_solve", 0.0: "k_reject_solve"}.get(path, "k_reject_solve")
    if st["match_grid"] >= st["reject_solve"]:
        dom, dom_ms, dom_bytes = "k_match_grid_coop", st["match_grid"], b_match
    else:
        dom, dom_ms, dom_bytes = rs_name, st["reject_solve"], b_rs
    ach = dom_bytes / (dom_ms * 1e-3) / 1e9
    traffic = None
    prof = REPO / "profiles" / "ncu_traffic.json"
    if prof.exists():
        try:
            traffic = json.loads(prof.read_text()).get(dom)
        except ValueError:
            pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom_bytes, "ms_per_launch": dom_ms,
                "kernels_ms_cold_l2": st, "kernels_ms_warm_l2": st_warm,
                "reject_solve_kernel": rs_name,
                "per_kernel": {"k_match_grid_coop": {"algorithmic_bytes": b_match, "ms": st["match_grid"],
                                                     "frac": b_match / (st["match_grid"] * 1e-3) / 1e9 / peak},
                               rs_name: {"algorithmic_bytes": b_rs, "ms": st["reject_solve"],
                                         "frac": b_rs / (st["reject_solve"] * 1e-3) / 1e9 / peak}},
                "iteration_bytes": b_match + b_rs,
                "note": "the search structure is L2-resident in the real loop; see DESIGN.md for the L2/latency view"}

    # ---- CPU baseline beside it: oracle port on a bounded sample of the same workload (N = 1)
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import simpleicp_oracle as O

        tr = O.Trace()
        n_it = 3
        t0 = time.perf_counter()
        H_o, _, x_o, _, _ = O.simpleicp(X_fix, X_mov, correspondences=K, min_change=0.0, max_iterations=n_it, trace=tr)
        t_cpu = time.perf_counter() - t0
        loop = float(np.sum(tr.iter_seconds))
        cpu = {"value": K * n_it / loop, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
               "sample": f"{n_it} ICP iterations of the oracle port on the full C3 pair (K={K}); loop only "
                         f"({loop:.1f} s; normals {tr.timings['normals']:.1f} s and final transform excluded; "
                         f"whole run {t_cpu:.1f} s); cKDTree queries on all cores, the rest single-threaded"}
        # live parity check on the same inputs: 3 lock-step iterations, oracle normals injected
        full = [np.full(n, np.nan, dtype=np.float32) for _ in range(4)]
        for a in range(3):
            full[a][tr.idx_sel] = tr.normals[:, a]
        full[3][tr.idx_sel] = tr.planarity
        r3 = sb.register(X_fix, X_mov, correspondences=K, min_change=0.0, max_iterations=n_it,
                         normals=tuple(full), engine=eng)
        parity = {"H_frobenius_vs_oracle_after_3_iterations": float(np.linalg.norm(r3.H - H_o)),
                  "kept_gpu": r3.records[-1]["n_kept"], "kept_oracle": int(tr.iterations[-1].keep.sum())}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(n, K),
                   "l2": "flushed: 256 MiB buffer overwritten before every timed step",
                   "nn_engine": "grid (float64, warm-started from the previous iteration's match) + TMA brute-force fallback",
                   "kept_per_iteration": n_kept, "numa_node_bound": numa},
        "value_l2_warm_queued": world * K / (warm_ms * 1e-3),
        "ms_per_step_l2_warm_queued": warm_ms,
        "roofline": roofline, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * n * 24,
                "d2h_bytes_per_step": n * 24 + 8 * n_kept,
                "ms_per_registration": 1e3 * e2e_s_max / args.e2e_steps, "iterations": its_total / (args.e2e_steps * world),
                "registrations": args.e2e_steps,
                "api": "simpleicp_b200.register(X_fix, X_mov, correspondences=K, engine=<reused>, transform_out=<pinned>)",
                "stage_ms": {k: v for k, v in tm.items() if k.endswith("_ms")},
                "iterations_in_barrier_free_kernel": tm.get("fused_iterations"),
                "iterations_repeated_in_general_kernel": tm.get("rerun_iterations"),
                "H_frobenius_vs_H_true": dH_true, **extra},
        "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "variants": variants,
        "c4": c4, "c5": c5,
    }
    # flushed at once: the line must not sit in a pipe buffer while the process tears CUDA / NCCL down
    print(json.dumps(line), flush=True)
    eng.close()
    batch.close_engine_pool()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--correspondences", type=int, default=100_000)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4c5", action="store_true")
    ap.add_argument("--c5-pairs-per-gpu", type=int, default=64)
    ap.add_argument("--c5-points", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0 only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3 if args.impl == "b200" else 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
