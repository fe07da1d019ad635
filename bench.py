#!/usr/bin/env python
"""bench.py — throughput of the squidpy spatial-statistics hot path on B200.

Headline (BASELINE.json `metric`, quoted on configs[1]): permutations/s of `nhood_enrichment` on 1 000 000 spots,
30 clusters, k=6 hexagonal neighbour graph (nnz = 5 992 002), n_perms = 1000 per GPU, exact numpy-RNG replay.
A "step" = one pass of the permutation test: the five kernels of the 1000 permutations (fill, swap-target generation,
apply, transpose, count) PLUS the per-bin mean / std over all permutations of the job — on one GPU the device statistics
kernel, on N GPUs one NCCL all-gather of the per-permutation counts and the same statistics kernel over the gathered rows
(device tensors; `squidpy_b200._dist.stats_device`) — with graph, base labels and generator states resident in
HBM.  `e2e` = the same metric through the public API (`squidpy_b200.gr.nhood_enrichment(adata, ...)`) with host buffers.
Further top-level keys of the same JSON line (each with its own roofline / e2e / cpu_baseline):
  `fast` / `roofline_fast`  — the same workload with `rng="philox"` (keyed-bijection permutations, not the reference's draws);
  `moran`                   — configs[2]: Moran's I genes/s, 199 809 spots x 20 000 genes CSR f32 @10 %, features sharded
                              over the ranks; e2e through `sq.gr.spatial_autocorr(adata)` (column-sliced upload + all-gather);
  `co_occurrence`           — configs[3]: 500 000 points, 20 clusters, 49 radii, through `sq.gr.co_occurrence`;
  `ripley_L`                — configs[4]: 300 000 cells, 12 clusters, through `sq.gr.ripley(mode="L")`.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--skip-moran] [--skip-pairs] [--skip-cpu] [--dump-outputs DIR]
N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
--dump-outputs DIR writes what the timed calls returned in their last step (rank 0) as DIR/<name>.npy, float64, so that two
builds can be compared output for output: every input is generated from fixed seeds.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG2 = dict(rows=1000, cols=1000, n_cls=30, n_perms=1000, seed=0)
CFG3 = dict(rows=447, cols=447, n_genes=20000, density=0.1)
METRIC = "nhood_enrichment permutations/s (1M spots, 30 clusters, k=6, n_perms=1000/GPU, exact numpy-RNG replay)"
WORKLOAD = "configs[1]: 1M-spot hex grid (nnz=5992002), 30 clusters, k=6, nhood_enrichment n_perms=1000 per GPU"
CONFIG = {"workload": WORKLOAD, "n_perms_per_gpu": CFG2["n_perms"], "rng": "numpy PCG64 exact replay",
          "l2": "flushed between steps (256 MiB read+write); working set per step 2 GB > L2",
          "timing": "CUDA events per step on the launch stream, max over ranks; the step includes the mean/std statistics (N>1: NCCL all-gather of the counts + the statistics kernel)"}
# warp instructions per evaluated unordered pair of the tiled pair kernel (profiles/r01_prof_cooc_metrics.csv:
# smsp__inst_executed.sum = 2.448e10 for 200 000 points = 2.0e10 pair evaluations) and the issue peak they are held against
PAIR_WARP_INSTR = 2.448e10 / (200_000 * 199_999 / 2)
# --dump-outputs: name -> what the timed calls returned in their last step; an array larger than DUMP_ARRAY_BYTES is stored as a
# fixed, seeded sample of its rows (plus `<name>_rows`, the row indices), which keeps a dump under DUMP_TOTAL_BYTES
OUTPUTS: dict[str, np.ndarray] = {}
DUMP_ARRAY_BYTES, DUMP_TOTAL_BYTES = 8 << 20, 64 << 20


def dump_outputs(path: str) -> None:
    os.makedirs(path, exist_ok=True)
    arrays = {}
    for name, a in OUTPUTS.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > DUMP_ARRAY_BYTES:
            keep = max(1, DUMP_ARRAY_BYTES // (a.nbytes // a.shape[0]))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            a, arrays[f"{name}_rows"] = a[rows], rows.astype(np.float64)
        arrays[name] = a
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_TOTAL_BYTES, f"--dump-outputs would write {total} bytes"
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(j.get("sm_max_mhz", 1965.0))
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


def _ncu_traffic(path, kernel_hint=None):
    """dram__bytes_read.sum + dram__bytes_write.sum of the longest launch in a committed `ncu --set full` metrics csv."""
    import csv

    try:
        rows = {r[0]: r for r in csv.reader(open(os.path.join(ROOT, path)))}
        names = rows["metric"][2:]
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
        dur = [float(v) for v in rows["gpu__time_duration.sum"][2:]]
        cand = [i for i, nm in enumerate(names) if kernel_hint is None or kernel_hint in nm] or list(range(len(names)))
        col = 2 + max(cand, key=lambda i: dur[i])
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(rows[k][col]) * scale[rows[k][1]]
        return {"bytes_per_launch": tot, "kernel": names[col - 2], "source": f"{path} (ncu --set full)"}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        # In-process NVML (a few microseconds per sample).  A looping `nvidia-smi` child costs nothing on a one-GPU box, but on a
        # multi-GPU box its queries contend with every rank's kernel launches: measured at 4 GPUs, 36.6 ms per step with it and
        # 22.7 ms without (tools/dist_diag.py, same kernels, same collective).  nvidia-smi stays as the fallback.
        try:
            import pynvml

            pynvml.nvmlInit()
            handle = None
            try:
                import torch

                pr = torch.cuda.get_device_properties(self.index)
                handle = pynvml.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0")
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml, self.handle, self.halt = pynvml, handle, threading.Event()
            self.proc = "nvml"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        while True:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append([str(sm), str(mx), "%.1f" % pw] + [("Active" if rs & b else "Not Active") for b in bits])
            except Exception:
                pass
            if self.halt.wait(0.1):
                break

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        if self.proc == "nvml":
            self.halt.set()
            self.t.join(timeout=2.0)
        else:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "NVML in-process, 10 Hz" if self.proc == "nvml" else "nvidia-smi -lms 200"}


def _dist_setup():
    import torch

    rank, ws, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if ws > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, ws, local


def _barrier_sync(ws):
    import torch

    if ws > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(v: float, ws: int) -> float:
    if ws == 1:
        return v
    import torch
    import torch.distributed as dist

    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _timed_steps(fn, steps, flush, ws):
    """EXACTLY `steps` calls of fn, each bracketed by CUDA events on the current stream; mean ms, max over ranks."""
    import torch

    _barrier_sync(ws)
    tot = 0.0
    for _ in range(steps):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    _barrier_sync(ws)
    return _max_over_ranks(tot / steps, ws)


# ---------------------------------------------------------------------------------------------------------------
# CPU arms (the oracle C port of the reference algorithms on the box's host cores)
# ---------------------------------------------------------------------------------------------------------------
def _pin_openmp():
    # must happen before liboracle.so (its libgomp) is loaded: threads bound to cores, no migration between runs.  It must NOT
    # happen before torch is imported: an OpenMP runtime that sees OMP_PROC_BIND binds the thread that initialises it -- the
    # main thread of every rank -- to the first place, and every thread created afterwards inherits that one-core mask
    # (measured under torchrun: 4 ranks launching from the same core, 36.6 ms per step instead of 22.7).
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")


class _cpu_leg:
    """A CPU-baseline leg: OpenMP pinning for the oracle library only, and the main thread gets its CPU mask back afterwards
    (the OpenMP master thread is bound to the first place while it works)."""

    cores = None  # CPUs this process may use, read BEFORE the OpenMP runtime narrows the main thread's mask

    def __enter__(self):
        self.mask = os.sched_getaffinity(0)
        _cpu_leg.cores = len(self.mask)
        _pin_openmp()
        return self

    def __exit__(self, *exc):
        try:
            os.sched_setaffinity(0, self.mask)
        except OSError:
            pass
        return False


def cpu_reference_nhood(g, base, n_cls, seed, reps=3, sample=None):
    """The reference's CPU algorithm ((N,C)-scratch two-pass count + exact numpy shuffle, oracle C port) on all host cores
    (threads over permutations == joblib n_jobs=-1 semantics): `reps` repetitions of a bounded sample, min / median."""
    from oracle import ref
    from squidpy_b200._rng import spawn_states

    cores = _cpu_leg.cores or len(os.sched_getaffinity(0))
    ref.nhood_perm_counts(g.indptr, g.indices, base, n_cls, spawn_states(seed, cores), n_threads=cores)  # warm-up
    t0 = time.perf_counter()
    ref.nhood_perm_counts(g.indptr, g.indices, base, n_cls, spawn_states(seed, 1), n_threads=1)
    t1 = time.perf_counter() - t0
    p_s = sample or int(max(cores, min(4 * cores, 8.0 / max(t1, 1e-3) * cores * 0.5)))
    rates = []
    for r in range(reps):
        t0 = time.perf_counter()
        ref.nhood_perm_counts(g.indptr, g.indices, base, n_cls, spawn_states(seed + r, p_s), n_threads=cores)
        rates.append(p_s / (time.perf_counter() - t0))
    return {"value": float(np.median(rates)), "unit": "permutations/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x {p_s} permutations of the same 1M-spot workload on {cores} OpenMP threads (OMP_PROC_BIND=close, OMP_PLACES=cores); median of {reps}",
            "min": float(min(rates)), "max": float(max(rates)), "serial_value": 1.0 / t1}


def run_reference(args, rank, ws):
    """--impl reference: the reference's own CPU path (oracle port; the Python/numba reference cannot travel to the GPU
    box) on the host cores, same config/metric; each step = a bounded sample (512 of the 1000 permutations)."""
    if rank != 0:
        return
    _cpu_leg.cores = len(os.sched_getaffinity(0))  # before the OpenMP runtime is loaded
    _pin_openmp()
    from oracle import ref
    from squidpy_b200._rng import spawn_states
    from tools import synth

    g = synth.hex_graph(CFG2["rows"], CFG2["cols"])
    base = synth.categorical_labels(g.shape[0], CFG2["n_cls"], seed=0).cat.codes.to_numpy().astype(np.uint32)
    cores = _cpu_leg.cores or len(os.sched_getaffinity(0))
    p_s = max(cores, min(512, 4 * cores))
    for _ in range(max(args.warmup, 1)):
        ref.nhood_perm_counts(g.indptr, g.indices, base, CFG2["n_cls"], spawn_states(0, cores), n_threads=cores)
    t0 = time.perf_counter()
    ref.nhood_perm_counts(g.indptr, g.indices, base, CFG2["n_cls"], spawn_states(0, 1), n_threads=1)
    serial = 1.0 / (time.perf_counter() - t0)
    rates = []
    t_all = time.perf_counter()
    for k in range(args.steps):
        t0 = time.perf_counter()
        counts = ref.nhood_perm_counts(g.indptr, g.indices, base, CFG2["n_cls"], spawn_states(k, p_s), n_threads=cores)
        rates.append(p_s / (time.perf_counter() - t0))
    OUTPUTS["nhood_counts"] = counts
    dt = time.perf_counter() - t_all
    val = args.steps * p_s / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "permutations/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 labels / u32 counts", "data": "synthetic", "config": CONFIG,
            "cpu_baseline": {"value": val, "unit": "permutations/s", "cores": cores, "kind": "port",
                             "sample": f"{p_s} of the 1000 permutations per step x {args.steps} steps, {cores} OpenMP threads over permutations (joblib n_jobs=-1 semantics), OMP_PROC_BIND=close OMP_PLACES=cores",
                             "per_step_min": float(min(rates)), "per_step_median": float(np.median(rates)), "per_step_max": float(max(rates)),
                             "serial_value": serial},
            "e2e": {"value": val, "unit": "permutations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs)


def _fit_extrapolate(ns, secs, n_target):
    """power-law fit t = a * n^b through the measured points, evaluated at n_target"""
    b = float(np.polyfit(np.log(ns), np.log(secs), 1)[0]) if len(ns) > 1 else 2.0
    return float(secs[-1] * (n_target / ns[-1]) ** b), b


# ---------------------------------------------------------------------------------------------------------------
def bench_moran(ctx, rank, ws, steps, warmup, flush, skip_cpu):
    """configs[2]: 199 809 spots x 20 000 genes CSR float32 @10 %, mode='moran'; features sharded over ranks (strong)."""
    import squidpy_b200 as sq
    from sklearn.preprocessing import normalize

    from squidpy_b200._dist import shard_range
    from squidpy_b200.gr import AutocorrPlan
    from tools import synth

    g = synth.hex_graph(CFG3["rows"], CFG3["cols"])
    n, G = g.shape[0], CFG3["n_genes"]
    lo, hi = shard_range(G, rank, ws)
    t0 = time.perf_counter()
    x = synth.expression_csr(n, G, density=CFG3["density"], coords=synth.hex_coords(CFG3["rows"], CFG3["cols"]), seed=100)
    t_gen = time.perf_counter() - t0
    ad = synth.make_adata(synth.hex_coords(CFG3["rows"], CFG3["cols"]), g, None, X=x)
    # ---- e2e: the plugin call with host buffers (graph copy + float32 row normalisation, column-sliced staged upload of this
    # rank's features, device re-layout, kernel, download, all-gather under torchrun, p-values, FDR, sort)
    sq.gr.spatial_autocorr(ad, mode="moran", copy=True)  # warm-up (pinned staging buffers, memory pool, scipy caches)
    reps = []
    for _ in range(2):
        _barrier_sync(ws)
        t0 = time.perf_counter()
        df = sq.gr.spatial_autocorr(ad, mode="moran", copy=True)
        _barrier_sync(ws)
        reps.append(_max_over_ranks(time.perf_counter() - t0, ws))
    t_e2e = min(reps)
    # ---- device-timed: matrix resident in HBM, one launch per step
    gn = g.copy()
    normalize(gn, norm="l1", axis=1, copy=False)
    plan = AutocorrPlan(gn, ctx)
    plan.load(x, obs_major=True, cols=(lo, hi))
    for _ in range(warmup):
        plan.run_async("moran")
    l0 = ctx.launches
    ms = _timed_steps(lambda: plan.run_async("moran"), steps, flush, ws)
    launches = (ctx.launches - l0) // max(steps, 1)
    score = plan.download()
    OUTPUTS["moran_I"] = score
    nnz_x = int(np.diff(x.indptr).sum()) if ws == 1 else int(x.nnz * (hi - lo) / G)
    algo_bytes = 8 * x.nnz + 8 * (G + 1) + 8 * g.nnz + 4 * (n + 1) + 8 * G  # whole call, SURVEY 8(d)
    peak, _, _ = _peaks()
    ach = algo_bytes / (ms / 1e3) / 1e9
    out = {"metric": "Moran's I genes/s (199 809 spots x 20 000 genes CSR f32 @10%, features sharded over GPUs)", "value": G / (ms / 1e3),
           "unit": "genes/s", "ms_per_step": ms, "scaling": "strong", "genes_per_rank": hi - lo, "nnz_x": int(x.nnz), "nnz_x_rank0_approx": nnz_x,
           "e2e": {"value": G / t_e2e, "unit": "genes/s", "seconds": t_e2e, "seconds_all": reps,
                   "h2d_bytes_per_step": int((x.data.nbytes + x.indices.nbytes) * (hi - lo) / G + 8 * (n + 1) + 12 * g.nnz),
                   "d2h_bytes_per_step": int(8 * (hi - lo)),
                   "note": "sq.gr.spatial_autocorr(adata, mode='moran', copy=True): pageable scipy buffers; every rank uploads only its feature slice; one all-gather of the scores"},
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes_per_step": int(algo_bytes),
                        "traffic": _ncu_traffic("profiles/r02_prof_moran_metrics.csv", "ac_sparse"),
                        "kernel": "ac_sparse_kernel (one launch per call; per-feature bitmap + rank lookups in shared memory, packed 64-byte W rows)",
                        "note": "the kernel is bound by L1/shared-memory wavefronts (one W-row gather + 8 bitmap look-ups per stored observation), not by DRAM: see DESIGN.md 3.2"},
           "finite_scores": int(np.isfinite(score).sum()), "max_I": float(np.nanmax(score)), "gpu_launches": int(launches), "synth_seconds": t_gen,
           "df_head_I": [float(v) for v in df["I"].to_numpy()[:3]]}
    if rank == 0 and ws == 1:
        # permutation variant at scale (SURVEY 8f-4): X stays resident, one launch per permutation
        t0 = time.perf_counter()
        sq.gr.spatial_autocorr(ad, mode="moran", n_perms=100, seed=0, copy=True)
        out["n_perms_100_seconds"] = time.perf_counter() - t0
        if not skip_cpu:
            try:
              with _cpu_leg():
                from oracle import ref

                cores = _cpu_leg.cores or len(os.sched_getaffinity(0))
                ns = 2 * cores
                sub = x[:, :ns].T.tocsr()
                ref.morans_i(gn, sub[:cores], n_threads=cores)
                t0 = time.perf_counter()
                exp = ref.morans_i(gn, sub, n_threads=cores)
                dt = time.perf_counter() - t0
                out["cpu_baseline"] = {"value": ns / dt, "unit": "genes/s", "cores": cores, "kind": "port",
                                       "sample": f"{ns} genes of the same matrix, scanpy-style restatement (oracle C, OpenMP over genes), {dt:.2f}s"}
                out["parity_max_abs_err_sample"] = float(np.nanmax(np.abs(score[:ns] - exp)))
            except Exception as e:  # pragma: no cover
                out["cpu_baseline"] = {"error": repr(e)}
    plan.close()
    return out


def bench_cooc(ctx, rank, ws, skip_cpu):
    """configs[3]: 500 000 uniform points, 20 clusters, interval=50 (L = 49) through sq.gr.co_occurrence."""
    import pandas as pd

    import squidpy_b200 as sq
    from tools import synth

    rng = np.random.default_rng(4)
    n = 500_000
    pts = rng.random((n, 2)) * 2.0e4
    labels = pd.Series(pd.Categorical.from_codes(rng.integers(0, 20, n), categories=[f"c{i:02d}" for i in range(20)]))
    ad = synth.make_adata(pts, None, labels)
    small = synth.make_adata(pts[:20000], None, pd.Series(labels.values[:20000]))
    sq.gr.co_occurrence(small, "cluster", copy=True)  # warm-up
    reps, kms = [], []
    for _ in range(2):
        _barrier_sync(ws)
        ctx.profile_reset()
        t0 = time.perf_counter()
        occ, iv = sq.gr.co_occurrence(ad, "cluster", copy=True)
        _barrier_sync(ws)
        reps.append(_max_over_ranks(time.perf_counter() - t0, ws))
    OUTPUTS["cooc_occ"], OUTPUTS["cooc_interval"] = occ, iv
    ctx.profile(True)
    ctx.profile_reset()
    sq.gr.co_occurrence(ad, "cluster", copy=True)
    ctx.sync()
    k_ms = _max_over_ranks(ctx.profile_get("pairs")[0], ws)
    ctx.profile(False)
    dt = min(reps)
    pairs = float(n) * (n - 1)
    _, _, sm_mhz = _peaks()
    issue_peak = 148 * 4 * sm_mhz * 1e6  # warp instructions / s: 148 SMs x 4 schedulers x 1 per clock
    ach = (pairs / 2) * PAIR_WARP_INSTR / (k_ms / 1e3)
    out = {"metric": "co_occurrence ordered pairs/s (500k points, 20 clusters, 49 radii)", "value": pairs / dt, "unit": "ordered pairs/s",
           "e2e": {"value": pairs / dt, "unit": "ordered pairs/s", "seconds": dt, "seconds_all": reps, "h2d_bytes_per_step": int(n * 12), "d2h_bytes_per_step": int(20 * 20 * 49 * 8),
                   "note": "sq.gr.co_occurrence(adata, 'cluster', copy=True) with host buffers"},
           "kernel_ms": k_ms, "kernel_pairs_per_s": pairs / (k_ms / 1e3), "scaling": "strong (pair tiles round-robin over ranks, one int64 all-reduce)",
           "roofline": {"bound": "fp32_issue", "achieved": ach / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-instr/s", "frac": ach / issue_peak,
                        "note": f"n(n-1)/2 pair evaluations x {PAIR_WARP_INSTR:.3f} warp instructions per pair (ncu smsp__inst_executed of the same kernel, profiles/r01_prof_cooc_metrics.csv) / (148 SM x 4 x {sm_mhz:.0f} MHz); each point is re-used ~1000x from shared memory, DRAM traffic ~ 0"},
           "finite": bool(np.isfinite(occ).all()), "interval_len": int(len(iv))}
    if rank == 0 and ws == 1 and not skip_cpu:
        try:
          with _cpu_leg():
            from oracle import ref
            from squidpy_b200.gr._ppatterns import _find_min_max

            cores = _cpu_leg.cores or len(os.sched_getaffinity(0))
            p32 = pts.astype(np.float32)
            labs = labels.cat.codes.to_numpy().astype(np.int32)
            tmin, tmax = _find_min_max(p32)
            thr = np.linspace(tmin, tmax, 50, dtype=np.float32)[1:] ** 2
            ns, secs = [20000, 40000], []
            for m in ns:
                t0 = time.perf_counter()
                ref.occur_count(p32[:m, 0], p32[:m, 1], thr, labs[:m], 20, n_threads=cores)
                secs.append(time.perf_counter() - t0)
            t_full, expo = _fit_extrapolate(ns, secs, n)
            out["cpu_baseline"] = {"value": pairs / t_full, "unit": "ordered pairs/s", "cores": cores, "kind": "port",
                                   "sample": f"oracle C port of _occur_count at n={ns} ({secs[0]:.2f}s, {secs[1]:.2f}s) on {cores} threads, fitted exponent {expo:.2f}, EXTRAPOLATED to n=500000 ({t_full:.0f}s)"}
        except Exception as e:  # pragma: no cover
            out["cpu_baseline"] = {"error": repr(e)}
    return out


def bench_ripley(ctx, rank, ws, skip_cpu):
    """configs[4]: 300 000 MERFISH-shaped cells, 12 clusters, ripley(mode='L', n_steps=50, n_simulations=100, n_observations=1000)."""
    import squidpy_b200 as sq
    from tools import synth

    n = 300_000
    pts = synth.thomas_points(n, seed=5)
    labels = synth.dirichlet_labels(n, 12, seed=5)
    ad = synth.make_adata(pts, None, labels)
    kw = dict(mode="L", n_steps=50, n_simulations=100, n_observations=1000, seed=0, copy=True)
    sq.gr.ripley(ad, "cluster", **kw)  # warm-up
    reps = []
    for _ in range(3):
        _barrier_sync(ws)
        t0 = time.perf_counter()
        res = sq.gr.ripley(ad, "cluster", **kw)
        _barrier_sync(ws)
        reps.append(_max_over_ranks(time.perf_counter() - t0, ws))
    OUTPUTS.update(ripley_L_stat=res["L_stat"]["stats"].to_numpy(), ripley_sims_stat=res["sims_stat"]["stats"].to_numpy(), ripley_bins=res["bins"],
                   ripley_pvalues=res["pvalues"])
    ctx.profile(True)
    ctx.profile_reset()
    sq.gr.ripley(ad, "cluster", **kw)
    ctx.sync()
    k_ms = _max_over_ranks(ctx.profile_get("pairs")[0], ws)
    ctx.profile(False)
    lab = labels.cat.codes.to_numpy()
    sizes = np.bincount(lab, minlength=12).astype(np.float64)
    pairs = float((sizes**2).sum() + 100 * 1000.0**2)
    dt = float(np.median(reps))
    out = {"metric": "Ripley L ordered pairs/s (300k cells, 12 clusters + 100 simulations of 1000 points, float64, 50 radii)", "value": pairs / dt,
           "unit": "ordered pairs/s",
           "e2e": {"value": pairs / dt, "unit": "ordered pairs/s", "seconds": dt, "seconds_all": reps, "h2d_bytes_per_step": int((n + 100_000) * 16), "d2h_bytes_per_step": int(112 * 50 * 8),
                   "note": "sq.gr.ripley(adata, 'cluster', mode='L', n_simulations=100, n_observations=1000, seed=0): convex hull + the 100 host-RNG point-process simulations (numpy stream parity) are inside; median of 3"},
           "kernel_ms": k_ms, "kernel_pairs_per_s": pairs / (k_ms / 1e3), "largest_cluster": int(sizes.max()), "scaling": "strong (pair tiles round-robin over ranks, one int64 all-reduce)",
           "pvalues_finite": bool(np.isfinite(res["pvalues"]).all())}
    if rank == 0 and ws == 1 and not skip_cpu:
        try:
          with _cpu_leg():
            from oracle import ref

            cores = _cpu_leg.cores or len(os.sched_getaffinity(0))
            big = pts[lab == int(np.argmax(sizes))]
            sup = res["bins"]
            ns, secs = [15000, 30000], []
            for m in ns:
                t0 = time.perf_counter()
                ref.pair_counts(big[:m], sup, n_threads=cores)
                secs.append(time.perf_counter() - t0)
            rate = ns[-1] ** 2 / secs[-1]  # brute force is exactly quadratic: pairs/s carries over
            out["cpu_baseline"] = {"value": rate, "unit": "ordered pairs/s", "cores": cores, "kind": "port",
                                   "sample": f"oracle brute-force restatement of KDTree.two_point_correlation at m={ns} ({secs[0]:.2f}s, {secs[1]:.2f}s) on {cores} threads; the reference itself uses one thread of a dual-tree KDTree (SURVEY 6: ~0.07 G pairs/s)"}
        except Exception as e:  # pragma: no cover
            out["cpu_baseline"] = {"error": repr(e)}
    return out


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--all", action="store_true", help="(kept for compatibility: everything runs by default)")
    ap.add_argument("--skip-moran", action="store_true")
    ap.add_argument("--skip-pairs", action="store_true")
    ap.add_argument("--skip-fast", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--perms", type=int, default=CFG2["n_perms"])
    ap.add_argument("--shuffle-threads", type=int, default=0)
    ap.add_argument("--shuffle-algo", type=int, default=-1)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed calls returned in their last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    if args.impl == "reference":
        rank, ws = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
        run_reference(args, rank, ws)
        return

    import torch

    import squidpy_b200 as sq
    from squidpy_b200._dist import stats_device
    from squidpy_b200._rng import spawn_states
    from squidpy_b200.gr import NhoodPlan
    from tools import synth

    rank, ws, local = _dist_setup()
    # the library launches on a torch-owned stream made current here, so torch.cuda.Event timing and the NCCL collectives
    # are ordered with its kernels (torch's default stream has handle 0, which the C ABI reads as "create your own stream")
    bench_stream = torch.cuda.Stream()
    torch.cuda.set_stream(bench_stream)
    ctx = sq.Context(local, bench_stream.cuda_stream)
    sq.set_default_context(ctx)  # sq.gr.* below run on the same context / stream
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush():
        flush_buf.add_(1)  # 256 MiB read+write > 126 MB L2

    g = synth.hex_graph(CFG2["rows"], CFG2["cols"])
    n, n_cls, P = g.shape[0], CFG2["n_cls"], args.perms
    labels = synth.categorical_labels(n, n_cls, seed=0)
    base = labels.cat.codes.to_numpy().astype(np.uint32)
    plan = NhoodPlan(g.indptr, g.indices, n_cls, ctx)
    if args.shuffle_threads:
        plan.set_option("shuffle_threads", args.shuffle_threads)
    plan.set_option("shuffle_algo", args.shuffle_algo)
    plan.set_base(base)
    observed = plan.count(base)
    states = spawn_states(CFG2["seed"], P * ws, rank * P, (rank + 1) * P)  # this rank's generators of the N*P-permutation job
    stat = torch.empty((2, n_cls * n_cls), dtype=torch.float64, device="cuda")
    last = {}

    def step():
        plan.run_async()
        if ws == 1:
            plan.stats_dev(stat[0].data_ptr(), stat[1].data_ptr())
        else:
            last["mean"], last["std"] = stats_device(plan, P * ws, True)

    def run_mode(fast: bool):
        if fast:
            plan.upload_philox(CFG2["seed"], rank * P, P)
        else:
            plan.upload(states)
        for _ in range(args.warmup):
            step()
        l0 = ctx.launches
        ms = _timed_steps(step, args.steps, flush, ws)
        launches = (ctx.launches - l0) // max(args.steps, 1)
        if ws == 1:
            m, s = stat.cpu().numpy()
        else:
            m, s = last["mean"].ravel(), last["std"].ravel()
        counts = plan.download()
        assert (counts.reshape(P, -1).sum(axis=1, dtype=np.int64) == g.nnz).all(), "count checksum failed"
        tag = "nhood_fast" if fast else "nhood"
        OUTPUTS.update({f"{tag}_counts": counts, f"{tag}_mean": m.reshape(n_cls, n_cls), f"{tag}_std": s.reshape(n_cls, n_cls)})
        # per-kernel-class CUDA-event times of ONE step (launches synchronised, not part of the timed region)
        ctx.profile(True)
        ctx.profile_reset()
        plan.run_async()
        ctx.sync()
        kms = {k: ctx.profile_get(k)[0] for k in ("fill", "misc", "shuffle", "transpose", "count")}
        ctx.profile(False)
        kms["jgen"] = kms.pop("misc")
        return ms, launches, kms, m.copy(), s.copy()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step, launches, kms, mean_x, std_x = run_mode(False)
    clocks = sampler.stop() if rank == 0 else None
    value = ws * P / (ms_step / 1e3)
    peak, peak_src, _ = _peaks()
    bpp = plan.bytes_per_perm
    dom = max(kms, key=kms.get)
    step_gbs = bpp * P / (ms_step / 1e3) / 1e9  # per GPU
    roofline = {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                "traffic": _ncu_traffic("profiles/r02_prof_nhood_metrics.csv", "apply") or _ncu_traffic("profiles/r01_prof_nhood_metrics.csv"),
                "kernel": "nhood permutation step = fill + jgen + shuffle (apply) + transpose + count + stats (one launch each per 1000 permutations); dominant: nhood_apply_list_kernel",
                "algorithmic_bytes_per_perm": int(bpp), "bytes_formula": "4*nnz + 4*(N+1) + 8*N + 4*C^2 (SURVEY.md 8d, reference dtypes)", "peak_source": peak_src,
                "kernel_ms": kms, "dominant_kernel": dom, "dominant_share": kms[dom] / max(sum(kms.values()), 1e-9)}

    fast = roofline_fast = None
    if not args.skip_fast:
        ms_f, launches_f, kms_f, mean_f, std_f = run_mode(True)
        gbs_f = bpp * P / (ms_f / 1e3) / 1e9
        kms_f = {"philox_labels": kms_f["shuffle"], "count": kms_f["count"]}
        with np.errstate(divide="ignore", invalid="ignore"):
            dm = np.abs(mean_f - mean_x) / (std_x / np.sqrt(P * ws))
            ds = np.abs(std_f - std_x) / std_x * np.sqrt(2 * P * ws)
        fast = {"metric": METRIC.replace("exact numpy-RNG replay", "rng='philox' keyed-bijection permutations"), "value": ws * P / (ms_f / 1e3),
                "unit": "permutations/s", "ms_per_step": ms_f, "gpu_launches": int(launches_f), "kernel_ms": kms_f,
                "validation_vs_exact": {"frac_bins_dmean_below_4": float(np.nanmean(dm < 4.0)), "frac_bins_dstd_below_4": float(np.nanmean(ds < 4.0)),
                                        "max_abs_dmean_in_sigma_over_sqrtP": float(np.nanmax(dm)), "max_rel_dstd_times_sqrt2P": float(np.nanmax(ds)),
                                        "bound": "SURVEY 8(d): |d mean| < 4 sigma/sqrt(P), |d std|/std < 4/sqrt(2P) per bin; both arms are P-sample estimates, so the difference of two has sqrt(2) of that spread and the maximum over 900 bins reaches ~4.5-5"},
                "note": "NOT the reference's permutations: same null distribution, different draws; z-scores agree to O(P^-1/2)"}
        roofline_fast = {"bound": "hbm", "achieved": gbs_f, "peak": peak, "unit": "GB/s", "frac": gbs_f / peak, "algorithmic_bytes_per_perm": int(bpp),
                         "kernel": "nhood_philox_labels_kernel + nhood_count_recs_kernel + stats", "kernel_ms": kms_f,
                         "note": "algorithmic bytes use the reference dtypes (u32 labels written + read per permutation); the kernels move u8 labels, so the effective figure can exceed the DRAM peak"}
        plan.upload(states)

    # ---- e2e through the public API with host buffers (H2D + kernels + statistics + D2H inside the timed region)
    ad = synth.make_adata(np.zeros((n, 2)), g, labels)
    e2e_steps = max(1, min(args.steps, 3))

    def api(rng_mode):
        return sq.gr.nhood_enrichment(ad, "cluster", n_perms=P * ws, seed=CFG2["seed"], copy=True, rng=rng_mode)

    def time_api(rng_mode):
        api(rng_mode)
        _barrier_sync(ws)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            res = api(rng_mode)
        _barrier_sync(ws)
        return _max_over_ranks((time.perf_counter() - t0) / e2e_steps, ws), res

    t_e2e, res = time_api("numpy")
    OUTPUTS["nhood_zscore"] = res.zscore
    h2d = int(g.indptr.nbytes + g.indices.nbytes + 2 * base.nbytes + states.nbytes)
    d2h = int(3 * n_cls * n_cls * 8)  # observed counts + mean + std (the per-permutation counts stay on the device)
    e2e = {"value": ws * P / t_e2e, "unit": "permutations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "seconds_per_call": t_e2e,
           "note": "sq.gr.nhood_enrichment(adata, n_perms=1000*N, seed, copy=True): CSR + labels + PCG64 states H2D (pageable scipy/numpy buffers), kernels, device statistics (N>1: NCCL all-gather of the per-permutation counts + the statistics kernel), z-scores"}
    assert np.isfinite(res.zscore).all() and (res.counts == observed).all()
    with np.errstate(divide="ignore", invalid="ignore"):
        z_dev = (observed.ravel() - mean_x) / std_x
    e2e["zscore_equals_device_step"] = bool(np.array_equal(z_dev, res.zscore.ravel()))
    if fast is not None:
        t_f, _ = time_api("philox")
        fast["e2e"] = {"value": ws * P / t_f, "unit": "permutations/s", "seconds_per_call": t_f, "h2d_bytes_per_step": int(h2d - states.nbytes), "d2h_bytes_per_step": d2h}

    # ---- configs[4] nhood part: 300 000 MERFISH-shaped cells, kNN(6) graph (built on the GPU), n_perms = 10 000 IN TOTAL,
    # sharded over the ranks (strong scaling; 1 250 permutations per GPU at N = 8)
    cfg5 = None
    try:
        from squidpy_b200.gr import KNNBuilder

        P5 = 10000
        pts5 = synth.thomas_points(300_000, seed=5)
        lab5 = synth.dirichlet_labels(300_000, 12, seed=5).cat.codes.to_numpy().astype(np.uint32)
        t0 = time.perf_counter()
        adj5, _ = KNNBuilder(n_neighs=6, ctx=ctx).build(pts5)
        t_graph = time.perf_counter() - t0
        lo5, hi5 = rank * -(-P5 // ws), min(P5, (rank + 1) * -(-P5 // ws))
        plan5 = NhoodPlan(adj5.indptr, adj5.indices, 12, ctx)
        plan5.set_base(lab5)
        plan5.upload(spawn_states(CFG2["seed"], P5, lo5, hi5))

        def step5():
            plan5.run_async()
            if ws == 1:
                plan5.stats_dev(stat5[0].data_ptr(), stat5[1].data_ptr())
            else:
                stats_device(plan5, P5, True)

        stat5 = torch.empty((2, 144), dtype=torch.float64, device="cuda")
        step5()
        ms5 = _timed_steps(step5, max(1, min(args.steps, 3)), flush, ws)
        if ws == 1:
            OUTPUTS["nhood_cfg5_mean"], OUTPUTS["nhood_cfg5_std"] = stat5.cpu().numpy().reshape(2, 12, 12)
        cfg5 = {"metric": "nhood_enrichment permutations/s (configs[4]: 300k cells, 12 clusters, kNN k=6 directed graph, n_perms=10000 in total)",
                "value": P5 / (ms5 / 1e3), "unit": "permutations/s", "ms_per_step": ms5, "scaling": "strong", "perms_per_rank": hi5 - lo5,
                "graph_build_seconds": t_graph, "nnz": int(adj5.nnz),
                "note": "kNN graph built with sqb_knn_2d; directed graph -> full-CSR count kernel (no symmetric shortcut); step = kernels + statistics (+ collective)"}
        plan5.close()
    except Exception as e:  # pragma: no cover
        cfg5 = {"error": repr(e)}

    moran = cooc = rip = None
    if not args.skip_moran:
        try:
            moran = bench_moran(ctx, rank, ws, max(1, min(args.steps, 5)), 1, flush, args.skip_cpu)
        except Exception as e:  # pragma: no cover
            moran = {"error": repr(e)}
    if not args.skip_pairs:
        for name, fn in (("cooc", bench_cooc), ("rip", bench_ripley)):
            try:
                r = fn(ctx, rank, ws, args.skip_cpu)
            except Exception as e:  # pragma: no cover
                r = {"error": repr(e)}
            if name == "cooc":
                cooc = r
            else:
                rip = r

    if rank == 0:
        cpu = None
        if not args.skip_cpu and ws == 1:  # the CPU baseline is timed on rank 0 at N = 1 only
            try:
                with _cpu_leg():
                    cpu = cpu_reference_nhood(g, base, n_cls, CFG2["seed"])
            except Exception as e:  # pragma: no cover
                cpu = {"error": repr(e)}
        line = {"metric": METRIC, "value": value, "unit": "permutations/s", "n_gpus": ws, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 labels / u32 counts", "data": "synthetic",
                "config": dict(CONFIG, shuffle_algo=args.shuffle_algo) if args.shuffle_algo != -1 else CONFIG,
                "collective": None if ws == 1 else "NCCL all_gather of the per-permutation counts (uint32[P, C*C] per rank, device tensors) + the statistics kernel over the gathered rows (inside the timed step)",
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "fast": fast, "roofline_fast": roofline_fast, "nhood_cfg5_strong": cfg5, "moran": moran, "co_occurrence": cooc, "ripley_L": rip}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs)
    plan.close()
    if ws > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
