#!/usr/bin/env python
"""bench.py -- queries/sec of the flat-search hot path on B200 (BASELINE.json metric).

Headline workload at every N: BASELINE configs[1] -- synthetic 1M x 384 fp32 rows, flat L2, 1024 queries, k=10.
A "step" is one index.search() over the whole query batch; every measurement below times --steps of them.  Inputs come
from fixed seeds, so --dump-outputs DIR (the headline's last timed result) is comparable between builds and runs.

  value      device-resident: queries / results are CUDA tensors, timed with CUDA events
  e2e        the same search through the C-ABI with HOST (pinned) buffers: H2D of the queries and D2H of (D, I) are
             inside the timed region
  roofline   the dominant kernel (K2 tcgen05 tensor scan; K1 streaming scan at nq = 1) timed per launch with CUDA
             events on its own stream inside the library
  parity_check   untimed: the first queries of the timed batch against the C oracle over the same synthetic rows
  cpu_baseline   the CPU restatement of IndexFlat (oracle/) on the box's host cores, bounded sample (rank 0)
  series     N = 1 only: the other batch sizes of configs[1] and BASELINE configs[2] (10M x 768 IP, k=100; batch
             1 / 32 / 4096), each with its own roofline and a parity spot check
  c4         BASELINE configs[3] at this N: 12.5M x 384 bf16 rows PER GPU (100M over 8), batch 4096, k=10

N > 1 (torchrun): the 1M rows are row-sharded over the ranks (contiguous ranges) and the query batch grows with N
(1024 x N queries, replicated on every rank), so per-GPU work is constant ("weak"): every rank searches its shard
for the whole batch and ONE kernel per rank exchanges the per-rank top-k lists over NVLink peer memory and merges
them (B200FLAT_EXCHANGE=nccl: one NCCL all-gather + merge kernel).  value = all queries answered / max-over-ranks
time.  --impl reference times the CPU restatement instead (faiss-cpu itself cannot be installed here: no wheel, no
network -- see DESIGN.md), with the thread count set here, not inherited from torchrun's OMP_NUM_THREADS=1.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (rows, d, nq, k, metric, normalize, storage)
    "c2": dict(n=1_000_000, d=384, nq=1024, k=10, metric=1, normalize=False, storage="fp32",
               label="synthetic 1Mx384 fp32 flat L2, 1024 queries, k=10 (BASELINE configs[1])"),
    "c2_nq1": dict(n=1_000_000, d=384, nq=1, k=10, metric=1, normalize=False, storage="fp32",
                   label="synthetic 1Mx384 fp32 flat L2, 1 query, k=10 (small-batch series)"),
    "c2_nq4": dict(n=1_000_000, d=384, nq=4, k=10, metric=1, normalize=False, storage="fp32",
                   label="synthetic 1Mx384 fp32 flat L2, 4 queries, k=10 (small-batch series)"),
    "c2_nq8": dict(n=1_000_000, d=384, nq=8, k=10, metric=1, normalize=False, storage="fp32",
                   label="synthetic 1Mx384 fp32 flat L2, 8 queries, k=10 (small-batch series)"),
    "c2_nq128": dict(n=1_000_000, d=384, nq=128, k=10, metric=1, normalize=False, storage="fp32",
                     label="synthetic 1Mx384 fp32 flat L2, 128 queries, k=10 (small-batch series)"),
    "c2_nq4096": dict(n=1_000_000, d=384, nq=4096, k=10, metric=1, normalize=False, storage="fp32",
                      label="synthetic 1Mx384 fp32 flat L2, 4096 queries, k=10 (large-batch series)"),
    "c2_nq32": dict(n=1_000_000, d=384, nq=32, k=10, metric=1, normalize=False, storage="fp32",
                    label="synthetic 1Mx384 fp32 flat L2, 32 queries, k=10 (small-batch series)"),
    "c2_shard4": dict(n=250_000, d=384, nq=4096, k=10, metric=1, normalize=False, storage="fp32",
                      label="synthetic 250k x 384 fp32 flat L2, 4096 queries, k=10 (one rank's share of the N = 4 weak-scaling point)"),
    "c2_shard8": dict(n=125_000, d=384, nq=8192, k=10, metric=1, normalize=False, storage="fp32",
                      label="synthetic 125k x 384 fp32 flat L2, 8192 queries, k=10 (one rank's share of the N = 8 weak-scaling point)"),
    "c3_nq1": dict(n=10_000_000, d=768, nq=1, k=100, metric=0, normalize=True, storage="fp32",
                   label="synthetic 10Mx768 flat inner-product (normalized), batch 1, k=100 (BASELINE configs[2])"),
    "c3_nq32": dict(n=10_000_000, d=768, nq=32, k=100, metric=0, normalize=True, storage="fp32",
                    label="synthetic 10Mx768 flat inner-product (normalized), batch 32, k=100 (BASELINE configs[2])"),
    "c3_nq4096": dict(n=10_000_000, d=768, nq=4096, k=100, metric=0, normalize=True, storage="fp32",
                      label="synthetic 10Mx768 flat inner-product (normalized), batch 4096, k=100 (BASELINE configs[2])"),
    "c4shard": dict(n=12_500_000, d=384, nq=4096, k=10, metric=1, normalize=False, storage="bf16", per_gpu=True,
                    label="synthetic 100Mx384 bf16 flat L2 row-sharded 12.5M rows per GPU (BASELINE configs[3]), 4096 queries, k=10, fp32 re-rank"),
    "c4shard_nq1": dict(n=12_500_000, d=384, nq=1, k=10, metric=1, normalize=False, storage="bf16", per_gpu=True,
                        label="synthetic 12.5Mx384 bf16 flat L2 per GPU (config 4 shard), 1 query, k=10"),
    "c4shard_nq32": dict(n=12_500_000, d=384, nq=32, k=10, metric=1, normalize=False, storage="bf16", per_gpu=True,
                         label="synthetic 12.5Mx384 bf16 flat L2 per GPU (config 4 shard), 32 queries, k=10"),
}
for _k, _w in WORKLOADS.items():
    _w["key"] = _k.split("_nq")[0]
SEED_DB, SEED_Q = 1234, 5678


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return dict(hbm=float(j["hbm_gbs"]), tf=float(j["bf16_tflops"]), tf_sus=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])),
                        src="measured")
        except Exception:
            pass
    return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    """Samples SM clocks / throttle reasons during the timed regions: NVML every ~2 ms (nvidia-smi every
    100 ms as the fallback when the NVML binding is missing)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NVML_BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop = threading.Event()
        self._t = None
        self.source = "nvidia-smi"

    def _sample_nvml(self, nv, h, mx, get_reasons):
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            self.mx.append(mx)
            bits = int(get_reasons(h))
            for name, bit in self.NVML_BITS.items():
                if bits & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _run_nvml(self, nv, h):
        mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while True:   # at least one sample even when the whole run is shorter than the thread's start-up
            self._sample_nvml(nv, h, mx, get_reasons)
            if self._stop.wait(0.002):
                break
        self._sample_nvml(nv, h, mx, get_reasons)

    def _run_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 8:
                    self.sm.append(float(parts[0]))
                    self.mx.append(float(parts[1]))
                    for name, val in zip(names, parts[4:8]):
                        if val.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            # NVML enumerates physical devices: map through CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.source = "nvml"
            self._t = threading.Thread(target=self._run_nvml, args=(nv, h), daemon=True)
        except Exception:
            self._t = threading.Thread(target=self._run_smi, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": self.source}


L2_BYTES = 126e6
FLUSH_BYTES = 256 << 20
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, D, I):
    """--dump-outputs: one search result as out_dir/distances.npy (float32) and out_dir/labels.npy (float64, exact for
    every label below 2**53), so that two builds can be compared output for output.  A result larger than DUMP_BYTES is
    cut to a fixed, seeded sample of its query rows, whose indices go to out_dir/query_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    D = np.asarray(D, np.float32)
    I = np.asarray(I).astype(np.float64)
    nq, k = D.shape
    row_bytes = k * (4 + 8) + 8
    if nq * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(SEED_Q).choice(nq, DUMP_BYTES // row_bytes, replace=False))
        D, I = D[rows], I[rows]
        np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), D)
    np.save(os.path.join(out_dir, "labels.npy"), I)


def host_threads() -> int:
    """Host threads this process may use (NOT what OMP_NUM_THREADS says: torchrun exports OMP_NUM_THREADS=1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def shard_rows(wl, world):
    """(rows_total, rows_per_gpu, nq_total) of a workload at `world` GPUs."""
    if wl.get("per_gpu"):        # config 4: every GPU holds n rows (the database grows with N), batch fixed
        return wl["n"] * world, wl["n"], wl["nq"]
    return wl["n"], -(-wl["n"] // world), wl["nq"] * world   # the same rows sharded, the batch grows with N (weak)


def workload_config(wl, world, nq_total=None):
    """The workload-defining part of `config`: printed verbatim by BOTH arms (repo and --impl reference)."""
    rows_total, rows_per_gpu, nq = shard_rows(wl, world)
    if nq_total is not None:
        nq = nq_total
    d = wl["d"]
    dpad = (d + 63) // 64 * 64
    scan_bytes = rows_per_gpu * dpad * 2
    flush = scan_bytes < 2 * L2_BYTES
    if flush:
        l2 = ("L2 flushed before every timed step (a %d MB buffer is overwritten; the bf16 scan copy is only %.0f MB per GPU, "
              "L2 126 MB); steps are timed one by one with CUDA events and summed" % (FLUSH_BYTES >> 20, scan_bytes / 1e6))
    else:
        l2 = "inputs larger than L2 (bf16 scan copy %.0f MB per GPU, L2 126 MB)" % (scan_bytes / 1e6)
    if world == 1:
        sharding = "single GPU"
    elif wl.get("per_gpu"):
        sharding = ("%d rows on each of %d GPUs (contiguous global ranges), batch %d replicated; per-rank top-k exchanged and "
                    "merged by one kernel per rank over NVLink peer memory (12 nq k bytes per rank)" % (rows_per_gpu, world, nq))
    else:
        sharding = ("rows in contiguous ranges over %d GPUs, batch %d = %d x N replicated; per-rank top-k exchanged and merged "
                    "by one kernel per rank over NVLink peer memory (12 nq k bytes per rank)" % (world, nq, wl["nq"]))
    label = wl["label"]
    if nq_total is not None and nq != (wl["nq"] if wl.get("per_gpu") else wl["nq"] * world):   # another batch size on the same rows (series)
        label = "%s [batch %d]" % (label, nq)
    return {"workload": label, "rows_total": rows_total, "rows_per_gpu": rows_per_gpu, "d": d, "nq": nq, "k": wl["k"],
            "metric": "L2" if wl["metric"] == 1 else "IP", "normalized": bool(wl["normalize"]), "storage": wl["storage"],
            "l2_policy": l2, "sharding": sharding}


def metric_name(wl):
    return "queries/sec @k=%d (flat %s, %d-d)" % (wl["k"], "L2" if wl["metric"] == 1 else "IP", wl["d"])


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that touch oracle/): cpu_baseline, --impl reference, the parity checkers
# ---------------------------------------------------------------------------------------------------------------------
def _cpu_step_fn(orc, wl, xb, xq, threads):
    if xq.shape[0] < 20:   # faiss: nq < 20 -> the seq path, one thread per query
        return lambda: orc.c_search(xb, xq, wl["k"], wl["metric"], algo=0, nthreads=threads)
    return lambda: orc.torch_search_blas(xb, xq, wl["k"], wl["metric"], nthreads=threads)


def cpu_baseline(wl, nq_total, budget_s=20.0):
    """Times the CPU restatement of IndexFlat on a bounded sample of the workload, all host threads."""
    import oracle as orc

    t0 = time.time()
    n = wl["n"] if not wl.get("per_gpu") else wl["n"]
    n_cpu = min(n, 1_000_000)
    xb = orc.c_synth_rows(SEED_DB, 0, n_cpu, wl["d"], wl["normalize"])
    threads = host_threads()
    if nq_total < 20:
        nq_s = nq_total
        xq = orc.c_synth_rows(SEED_Q, 0, nq_s, wl["d"], wl["normalize"])
        fn = _cpu_step_fn(orc, wl, xb, xq, threads)
        fn()
        t = time.time()
        fn()
        dt = time.time() - t
        note = "C restatement, seq path (nq<20: one thread per query, as faiss)"
        cores = min(threads, nq_s)
    else:
        nq_s = min(nq_total, 128)
        xq_all = orc.c_synth_rows(SEED_Q, 0, min(nq_total, 4096), wl["d"], wl["normalize"])
        orc.torch_search_blas(xb[:20000], xq_all[:32], wl["k"], wl["metric"], nthreads=threads)  # thread-pool / MKL warm-up
        t = time.time()
        orc.torch_search_blas(xb, xq_all[:nq_s], wl["k"], wl["metric"], nthreads=threads)
        dt = time.time() - t
        while dt < budget_s / 4 and nq_s < xq_all.shape[0]:   # grow the sample while it stays within the budget
            nq_s = min(xq_all.shape[0], nq_s * 4)
            t = time.time()
            orc.torch_search_blas(xb, xq_all[:nq_s], wl["k"], wl["metric"], nthreads=threads)
            dt = time.time() - t
        note = "BLAS (torch CPU/MKL sgemm) restatement of faiss's blas path (sgemm blocks + expanded form + clamp)"
        cores = threads
    qps = nq_s / dt * (n_cpu / n)  # rows scale linearly; only != 1 when the host cannot hold n rows
    sample = f"{nq_s} of {nq_total} queries x {n_cpu} of {n} rows, {note}; setup {time.time() - t0 - dt:.1f}s"
    if n_cpu != n:
        sample += " (q/s linearly extrapolated in rows)"
    return {"value": round(qps, 2), "unit": "queries/sec", "cores": int(cores), "kind": "port", "sample": sample}


def cpu_baseline_isolated(workload, wl, nq_total, budget_s):
    """cpu_baseline() in a fresh interpreter without the launcher's thread caps: inside the GPU arm's own process (CUDA
    context, NCCL threads, an intra-op pool first used under torchrun's OMP_NUM_THREADS=1) the same sgemm ran at 3-10 % of
    its speed (N = 2: 149 q/s, N = 8: 44 q/s, against ~1500 q/s for `--impl reference` on the same hosts)."""
    env = {k_: v for k_, v in os.environ.items()
           if k_ not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "RANK", "LOCAL_RANK", "WORLD_SIZE")}
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-baseline-only", "--workload", workload, "--nq", str(nq_total),
           "--cpu-budget", str(budget_s)]
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
        line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)
    except Exception as exc:   # never lose the GPU line to the CPU leg
        return {"value": None, "unit": "queries/sec", "cores": host_threads(), "kind": "port",
                "sample": "cpu_baseline subprocess failed: %s" % exc}


def run_reference(args, wl, rank, world):
    """--impl reference: the CPU restatement of the reference's IndexFlat path on the host cores.  The thread count is
    set HERE (all threads this process may use), never inherited from the launcher; the reference's own configured
    mode (OMP_NUM_THREADS=1, 2-cli-rag-search.py:15-19) is reported beside it."""
    if rank != 0:
        return
    import oracle as orc

    threads = host_threads()
    rows_total, _, nq_total = shard_rows(wl, world)
    n = rows_total if not wl.get("per_gpu") else wl["n"]
    n_cpu = min(n, 1_000_000)
    xb = orc.c_synth_rows(SEED_DB, 0, n_cpu, wl["d"], wl["normalize"])
    nq_s = nq_total if nq_total < 20 else min(nq_total, 1024)   # one step = up to 1024 queries (~1 s of sgemm on 16 cores)
    xq = orc.c_synth_rows(SEED_Q, 0, nq_s, wl["d"], wl["normalize"])
    step = _cpu_step_fn(orc, wl, xb, xq, threads)
    for _ in range(max(args.warmup, 1)):
        step()
    t = time.time()
    for _ in range(args.steps):
        D, I = step()
    dt = (time.time() - t) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, D, I)
    qps = nq_s / dt * (n_cpu / n)
    cores = threads if nq_s >= 20 else min(threads, nq_s)
    # the reference's own configuration: one thread; a smaller sample keeps it bounded
    nq_1 = nq_s if nq_s < 20 else min(nq_s, 64)
    step1 = _cpu_step_fn(orc, wl, xb, xq[:nq_1], 1)
    step1()
    t = time.time()
    step1()
    qps_1 = nq_1 / (time.time() - t) * (n_cpu / n)
    path = "C restatement, seq path" if nq_s < 20 else "MKL sgemm blas path"
    sample = (f"{nq_s} of {nq_total} queries x {n_cpu} of {n} rows per step; CPU restatement of IndexFlat (faiss-cpu unavailable), "
              f"{path}; threads set by bench.py = {cores} (launcher's OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS', 'unset')} ignored)")
    line = {
        "impl": "reference", "metric": metric_name(wl), "value": round(qps, 2), "unit": "queries/sec",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, world),
        "cpu_baseline": {"value": round(qps, 2), "unit": "queries/sec", "cores": int(cores), "kind": "port", "sample": sample,
                         "one_thread": {"value": round(qps_1, 2), "cores": 1,
                                        "sample": f"{nq_1} queries x {n_cpu} rows, the reference's configured OMP_NUM_THREADS=1"}},
        "e2e": {"value": round(qps, 2), "unit": "queries/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def parity_full(wl, xq_host, D, I, nchk):
    """Whole-database check (n <= 1M): the first nchk queries against the C oracle's seq path over the same rows."""
    import oracle as orc

    xb_host = orc.c_synth_rows(SEED_DB, 0, wl["n"], wl["d"], wl["normalize"])
    D_ref, I_ref = orc.c_search(xb_host, xq_host[:nchk], wl["k"], wl["metric"], algo=1, nthreads=host_threads())
    r = orc.recall_and_errors(D[:nchk], I[:nchk], D_ref, I_ref, wl["metric"])
    r.update({"mode": "full database vs C oracle (seq path)", "queries": int(nchk), "rows": int(wl["n"])})
    return r


def parity_sampled(wl, ix, rows_local, xq_host, D, I, nchk, window=1_000_000):
    """Databases the host cannot hold / the oracle cannot finish (10M+ rows): size-independent sampled exactness.
      * window: the oracle's top-k over the first `window` rows (read back from the index: the authoritative rows);
        a window row that beats the k-th returned neighbour must be in the result, and returned labels inside the
        window must be the oracle's
      * every returned distance recomputed in float64 (rank-0-resident labels: from the stored rows, 1e-5; labels on
        other ranks: from the regenerated fp32 rows -- bf16 storage then differs by its rounding, tolerance 2e-2)
      * order: ascending (L2) / descending (IP)"""
    import oracle as orc

    k, metric, d = wl["k"], wl["metric"], wl["d"]
    W = int(min(window, rows_local))
    xwin = ix.reconstruct_n(0, W)
    Dw, Iw = orc.c_search(xwin, xq_host[:nchk], k, metric, algo=1, nthreads=host_threads())
    sign = 1.0 if metric == 1 else -1.0
    viol, rel_local, rel_remote, sorted_ok = 0, 0.0, 0.0, True
    for qi in range(nchk):
        got = {int(i) for i in I[qi] if i >= 0}
        kth = sign * float(D[qi, k - 1])
        tol = 1e-5 * max(abs(kth), 10.0)
        for j in range(k):
            if Iw[qi, j] >= 0 and sign * float(Dw[qi, j]) < kth - tol and int(Iw[qi, j]) not in got:
                viol += 1       # a window row better than the k-th returned neighbour is missing
        want = {int(i) for i in Iw[qi] if i >= 0}
        for j in range(k):
            lab = int(I[qi, j])
            if 0 <= lab < W and lab not in want and sign * float(D[qi, j]) < sign * float(Dw[qi, k - 1]) - tol:
                viol += 1       # a returned window label the oracle does not have
        keys = sign * D[qi].astype(np.float64)
        sorted_ok = sorted_ok and bool(np.all(np.diff(keys) >= -1e-6 * np.maximum(np.abs(keys[1:]), 1.0)))
        q64 = xq_host[qi].astype(np.float64)
        for j in range(k):
            lab = int(I[qi, j])
            if lab < 0:
                continue
            local = lab < rows_local
            row = (ix.reconstruct(lab) if local else orc.c_synth_rows(SEED_DB, lab, 1, d, wl["normalize"])[0]).astype(np.float64)
            exact = float(((row - q64) ** 2).sum()) if metric == 1 else float(row @ q64)
            rel = abs(exact - float(D[qi, j])) / max(abs(exact), 10.0)
            if local:
                rel_local = max(rel_local, rel)
            else:
                rel_remote = max(rel_remote, rel)
    ok = viol == 0 and sorted_ok and rel_local <= 1e-5 and rel_remote <= (2e-2 if wl["storage"] == "bf16" else 1e-5)
    return {"mode": "sampled: oracle over a row window + recomputed distances", "queries": int(nchk), "window_rows": W,
            "window_violations": int(viol), "recall": 1.0 if viol == 0 else 0.0, "sorted": bool(sorted_ok),
            "max_rel_err": float(rel_local), "max_rel_err_remote_labels_vs_unrounded_rows": float(rel_remote), "ok": bool(ok)}


# ---------------------------------------------------------------------------------------------------------------------
# the GPU arm
# ---------------------------------------------------------------------------------------------------------------------
class Ctx:
    """One workload's index (this rank's shard) plus what every batch size measured on it shares."""

    def __init__(self, env, wl, algo_name="auto", slack=0):
        b2f, torch = env["b2f"], env["torch"]
        from rag_faiss_embedding_b200.sharded import ShardedIndexFlat, partition_rows

        self.env, self.wl = env, wl
        rank, world, local_rank = env["rank"], env["world"], env["local_rank"]
        self.rows_total, _, _ = shard_rows(wl, world)
        if wl.get("per_gpu"):
            self.lo, self.hi = rank * wl["n"], (rank + 1) * wl["n"]
        else:
            self.lo, self.hi = partition_rows(wl["n"], world)[rank]
        self.algo = {"auto": b2f.ALGO_AUTO, "scan": b2f.ALGO_SCAN, "tensor": b2f.ALGO_TENSOR}[algo_name]
        self.storage = b2f.STORE_BF16 if wl["storage"] == "bf16" else b2f.STORE_F32
        self.ix = b2f.IndexFlat(wl["d"], wl["metric"], storage=self.storage, device=local_rank)
        self.ix.reserve(self.hi - self.lo)
        self.ix.add_synthetic(SEED_DB, self.lo, self.hi - self.lo, wl["normalize"])   # on the device, bit-identical to the oracle
        self.ix.set_search_params(algo=self.algo, id_offset=self.lo, profile=True, slack=slack)
        self.sh = None
        if world > 1:
            self.sh = ShardedIndexFlat(wl["d"], wl["metric"], local_index=self.ix)
            self.sh.segments.append(self.lo, self.hi - self.lo)
            self.sh.set_total(self.rows_total)

    def close(self):
        self.sh = None
        self.ix = None
        self.env["torch"].cuda.synchronize()


def measure(ctx, nq, steps, warmup, do_e2e=True, parity="auto", nchk=4, dump_dir=None):
    """One batch size on one index: device-resident value, e2e through host buffers, roofline of the dominant kernel,
    parity spot check; with dump_dir, rank 0 writes the result of the last timed device step there.  Collective at
    world > 1.  Returns the record on rank 0 (None elsewhere)."""
    env, wl, ix, sh = ctx.env, ctx.wl, ctx.ix, ctx.sh
    b2f, torch, dist = env["b2f"], env["torch"], env["dist"]
    from rag_faiss_embedding_b200.encoder import synth_rows

    rank, world, dev, peaks = env["rank"], env["world"], env["dev"], env["peaks"]
    d, k = wl["d"], wl["k"]
    cfg = workload_config(wl, world, nq)
    flush = cfg["l2_policy"].startswith("L2 flushed")
    flush_buf = env.get("flush_buf")
    if flush and flush_buf is None:
        flush_buf = env["flush_buf"] = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=dev)

    # queries from the library's own counter-based generator (bit-identical to the oracle's)
    xq_host = synth_rows(SEED_Q, 0, nq, d, wl["normalize"], device=env["local_rank"]).cpu().numpy()
    xq_pin = torch.from_numpy(xq_host).pin_memory()
    D_pin = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    I_pin = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    xq_dev = xq_pin.to(dev)
    D_dev = torch.empty((nq, k), dtype=torch.float32, device=dev)
    I_dev = torch.empty((nq, k), dtype=torch.int64, device=dev)

    def step_device():
        if sh is not None:
            sh.search(xq_dev, k, out=(D_dev, I_dev))
        else:
            ix.search_tensors_into(xq_dev, k, D_dev, I_dev)

    def step_host():
        if sh is not None:
            sh.search_host(xq_pin, k, D_pin, I_pin)   # each rank uploads its slice of the replicated batch
        else:
            ix.search_into(xq_pin.numpy(), k, D_pin.numpy(), I_pin.numpy())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, nsteps):
        barrier()
        if not flush:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(nsteps):
                fn()
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1) / nsteps
        else:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]
            for a, b in evs:
                flush_buf.zero_()      # 256 MB written: nothing of the database survives in L2 (untimed)
                a.record()
                fn()
                b.record()
            barrier()
            ms = sum(a.elapsed_time(b) for a, b in evs) / nsteps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(warmup):
        step_device()
    st0 = ix.stats()
    ms_step = timed(step_device, steps)
    st1 = ix.stats()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, D_dev.cpu().numpy(), I_dev.cpu().numpy())
    # per-launch time of the dominant kernel: CUDA events recorded by the library around every launch in the timed
    # region (running sums, read once so that the host loop stays tight)
    n_launch = max(st1["prof_main_launches"] - st0["prof_main_launches"], 1)
    n_search = max(st1["prof_searches"] - st0["prof_searches"], 1)
    launches_per_search = n_launch / n_search   # > 1 when a big batch x big k' is processed in query chunks
    kernel_ms = (st1["prof_main_ms_sum"] - st0["prof_main_ms_sum"]) / n_launch
    pipeline_ms = (st1["prof_total_ms_sum"] - st0["prof_total_ms_sum"]) / n_search
    launches = st1["launches"] - st0["launches"] + (steps if world > 1 else 0)   # + the exchange/merge kernel per step
    e2e_ms = None
    if do_e2e:
        for _ in range(3):
            step_host()
        e2e_ms = timed(step_host, steps)

    # ---- parity spot check on the timed configuration (untimed; collective: every rank searches, rank 0 checks) ----
    step_device()
    torch.cuda.synchronize()
    par = None
    if rank == 0 and parity != "off":
        nchk = min(nchk, nq)
        Dg, Ig = D_dev[:nchk].cpu().numpy(), I_dev[:nchk].cpu().numpy()
        if parity == "full" or (parity == "auto" and ctx.rows_total <= 1_000_000 and not wl.get("per_gpu")):
            par = parity_full(wl, xq_host, Dg, Ig, nchk)
        else:
            par = parity_sampled(wl, ix, ctx.hi - ctx.lo, xq_host, Dg, Ig, nchk)
    if world > 1:
        dist.barrier()
    if rank != 0:
        return None

    st = ix.stats()
    used_algo = st["last_algo"]
    rows_local = ctx.hi - ctx.lo
    elem = 2 if (used_algo == b2f.ALGO_TENSOR or ctx.storage == b2f.STORE_BF16) else 4
    dpad = (d + 63) // 64 * 64 if elem == 2 else d
    if used_algo == b2f.ALGO_TENSOR and nq > 128:
        flops = 2.0 * nq * rows_local * d / launches_per_search   # per launch
        ach = flops / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tf"], "unit": "TFLOP/s",
                "frac": round(ach / peaks["tf"], 4), "traffic": None, "frac_of_sustained": round(ach / peaks["tf_sus"], 4)}
    else:
        passes = (nq + 7) // 8 if used_algo == b2f.ALGO_SCAN else 1   # the scan walks the queries in groups of <= 8
        bytes_ = (rows_local * dpad * elem + min(nq, 8 if used_algo == b2f.ALGO_SCAN else nq) * d * 4) * passes
        ach = bytes_ / (kernel_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm"], 4), "traffic": None}
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = f"{wl['key']}|nq{nq}|{'tensor' if used_algo == b2f.ALGO_TENSOR else 'scan'}"
        if key in tr and world == 1:
            roof["traffic"] = tr[key]["bytes"]
            roof["traffic_source"] = tr[key]["capture"]
    except Exception:
        pass
    roof["kernel"] = "tensor_scan_kernel (K2 tcgen05)" if used_algo == b2f.ALGO_TENSOR else "scan_kernel (K1)"
    roof["kernel_ms"] = round(kernel_ms, 4)
    roof["launches_per_search"] = round(launches_per_search, 2)
    roof["peak_source"] = peaks["src"] + (" burst" if roof["bound"] == "tensor" else "")
    roof["pipeline_ms"] = round(pipeline_ms, 4)
    rec = {
        "metric": metric_name(wl), "value": round(nq / (ms_step * 1e-3), 1), "unit": "queries/sec",
        "ms_per_step": round(ms_step, 4), "steps": steps, "warmup": warmup,
        "dtype": "bf16 tensor-core candidates + f32 exact re-rank" if used_algo == b2f.ALGO_TENSOR else "f32",
        "config": cfg,
        "engine": {"algo": {1: "scan", 2: "tensor"}.get(used_algo, "?"), "kprime": st["last_kprime"],
                   "fallback_queries": st["fallback_queries"], "overflow_queries": st["overflow_queries"],
                   "rescued_queries": st["rescued_queries"],
                   "filter_survivors_per_query": round(st["last_list_entries"] / max(nq, 1), 1),
                   "exchange": (os.environ.get("B200FLAT_EXCHANGE", "peer").lower() if world > 1 else None)},
        "roofline": roof, "gpu_launches": int(launches),
    }
    if e2e_ms is not None:
        rec["e2e"] = {"value": round(nq / (e2e_ms * 1e-3), 1), "unit": "queries/sec", "ms_per_step": round(e2e_ms, 4),
                      "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * 12}
    if par is not None:
        rec["parity_check"] = par
    return rec


def brief(rec):
    """A series / c4 entry: the record without the contract's top-level boilerplate."""
    keep = ("value", "unit", "ms_per_step", "steps", "dtype", "engine", "roofline", "parity_check", "e2e", "clocks")
    out = {"workload": rec["config"]["workload"], "nq": rec["config"]["nq"], "k": rec["config"]["k"],
           "rows_total": rec["config"]["rows_total"], "rows_per_gpu": rec["config"]["rows_per_gpu"]}
    out.update({k_: rec[k_] for k_ in keep if k_ in rec})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every measurement (headline, e2e, series, c4)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--algo", default="auto", choices=["auto", "scan", "tensor"])
    ap.add_argument("--slack", type=int, default=0, help="tensor path: extra coarse candidates per query (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-series", action="store_true", help="skip the N = 1 series (other batch sizes, BASELINE configs[2])")
    ap.add_argument("--no-c4", action="store_true", help="skip the BASELINE configs[3] record (12.5M bf16 rows per GPU)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--nq", type=int, default=0, help="diagnostics: another batch size on the workload's rows")
    ap.add_argument("--cpu-baseline-only", action="store_true", help="internal: print the cpu_baseline record for --nq queries and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (distances, labels) of the headline's last timed step as DIR/*.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cpu_baseline_only:
        w0 = WORKLOADS[args.workload]
        print(json.dumps(cpu_baseline(w0, args.nq if args.nq > 0 else w0["nq"], args.cpu_budget)), flush=True)
        return
    wl = dict(WORKLOADS[args.workload])
    if args.nq > 0:
        wl["nq"] = args.nq
        wl["label"] += " [--nq %d]" % args.nq
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import torch
    import torch.distributed as dist

    import rag_faiss_embedding_b200 as b2f

    # before any torch CPU op: torchrun exports OMP_NUM_THREADS=1 and the intra-op pool keeps the size it was first used
    # with, which would cripple rank 0's cpu_baseline leg (N = 2, first run: 149 q/s on 24 cores instead of ~1400)
    torch.set_num_threads(host_threads())
    if args.warmup < 3:
        args.warmup = 3
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env = {"b2f": b2f, "torch": torch, "dist": dist, "rank": rank, "world": world, "local_rank": local_rank, "dev": dev,
           "peaks": load_peaks()}
    headline = args.workload == "c2"
    parity = "off" if args.no_parity else "auto"
    _, _, nq = shard_rows(wl, world)

    # ---- the headline measurement (clocks sampled through warm-up, the timed region and the e2e region) -------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx = Ctx(env, wl, args.algo, args.slack)
    rec = measure(ctx, nq, args.steps, args.warmup, do_e2e=True, parity=parity, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    series, c4 = [], None
    sw = min(args.warmup, 3)
    if headline and world == 1 and not args.no_series:
        # the other batch sizes of configs[1] on the same index
        for nq_s, algo_s in ((1, "auto"), (1, "tensor"), (32, "auto"), (128, "auto"), (4096, "auto")):
            ctx.ix.set_search_params(algo={"auto": b2f.ALGO_AUTO, "tensor": b2f.ALGO_TENSOR}[algo_s])
            r = measure(ctx, nq_s, args.steps, sw, do_e2e=False, parity=parity)
            if r:
                series.append(brief(r))
        ctx.close()
        ctx = None
        # BASELINE configs[2]: 10M x 768 inner product (normalized), k = 100, batch 1 / 32 / 4096
        c3 = Ctx(env, WORKLOADS["c3_nq4096"], "auto", 0)
        for nq_s in (1, 32, 4096):
            s2 = ClockSampler(local_rank)
            s2.start()
            r = measure(c3, nq_s, args.steps, sw, do_e2e=False, parity=parity if nq_s == 4096 else "off")
            ck = s2.stop()
            if r:
                r["clocks"] = ck
                series.append(brief(r))
        c3.close()
    if ctx is not None:
        ctx.close()
        ctx = None
    if headline and not args.no_c4:
        # BASELINE configs[3] at this N: 12.5M bf16 rows on every GPU (100M x 384 over 8), batch 4096, k = 10
        c4ctx = Ctx(env, WORKLOADS["c4shard"], "auto", 0)
        s4 = ClockSampler(local_rank)
        if rank == 0:
            s4.start()
        r = measure(c4ctx, WORKLOADS["c4shard"]["nq"], args.steps, sw, do_e2e=False, parity=parity)
        ck = s4.stop() if rank == 0 else None
        if r:
            r["clocks"] = ck
            c4 = brief(r)
            c4["config"] = r["config"]
        # the north star's small-batch target on this configuration: batch 1 and 32 against the HBM roofline
        small = []
        for nq_s in (1, 32):
            rs = measure(c4ctx, nq_s, args.steps, sw, do_e2e=False, parity="off")
            if rs:
                small.append(brief(rs))
        if c4 is not None and small:
            c4["small_batches"] = small
        c4ctx.close()

    if rank == 0:
        line = {
            "metric": rec["metric"], "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": rec["dtype"], "data": "synthetic", "config": rec["config"], "engine": rec["engine"],
            "roofline": rec["roofline"], "e2e": rec["e2e"], "gpu_launches": rec["gpu_launches"], "clocks": clocks,
        }
        if "parity_check" in rec:
            line["parity_check"] = rec["parity_check"]
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_isolated(args.workload, wl, nq, args.cpu_budget if world == 1 else min(args.cpu_budget, 10.0))
        if series:
            line["series"] = series
        if c4 is not None:
            line["c4"] = c4
        print(json.dumps(line), flush=True)
    if world > 1:
        # The other ranks must SLEEP while rank 0 times the CPU leg: an NCCL barrier spins on the host, and with the
        # container's CPU quota N - 1 spinning ranks starve the sgemm (N = 4: 45 q/s instead of ~1400).  A blocking
        # wait on the rendezvous store does not spin.
        try:
            store = dist.distributed_c10d._get_default_store()
            if rank == 0:
                store.set("b200flat_cpu_leg_done", "1")
            else:
                store.wait(["b200flat_cpu_leg_done"])
        except Exception:
            pass
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
