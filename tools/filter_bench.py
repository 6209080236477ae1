"""Filtered search on one B200: BASELINE config 2 (1M x 384 rows from add_synthetic, L2), fp32 and bf16 storage.

For nq = 1, 32 and 1024 top-k (k = 10) and range search at about 10 hits per query (1024 queries), each selector -- Range
over half the rows, Batch at 50 %, 1 % and 0.01 % of the rows, Not of the 1 % Batch -- is timed against the unfiltered
call on the same queries (CUDA-synchronised host clock, median of --reps calls after warm-up, device queries and device
selector data), with the fallback / overflow / range-pass counts of the filtered searches.  The cost of the bitmap and
masked-bias kernels is taken as the difference between a filtered and an unfiltered search on the scan path at nq = 1
(bitmap only) and on the tensor path at nq = 32 (bitmap and masked bias).  The rows (1.5 GB fp32, 0.8 GB bf16) exceed the 126 MB L2.

usage: python tools/filter_bench.py [--reps 20] [--out filter_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rag_faiss_embedding_b200 as m  # noqa: E402

N, D, SEED, K = 1_000_000, 384, 1234, 10
COUNTERS = ("fallback_queries", "overflow_queries", "range_queries")


def timed(fn, reps, sync):
    fn()
    fn()
    sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card, flush=True)
    sync = torch.cuda.synchronize
    rng = np.random.default_rng(7)
    dev = torch.device("cuda", 0)
    sels = {
        "range_50%": m.IDSelectorRange(0, N // 2),
        "batch_50%": m.IDSelectorBatch(torch.from_numpy(rng.choice(N, N // 2, replace=False)).to(dev)),
        "batch_1%": m.IDSelectorBatch(torch.from_numpy(rng.choice(N, N // 100, replace=False)).to(dev)),
        "batch_0.01%": m.IDSelectorBatch(torch.from_numpy(rng.choice(N, N // 10000, replace=False)).to(dev)),
    }
    sels["not_batch_1%"] = m.IDSelectorNot(sels["batch_1%"])
    result = {"card": card, "config": f"{N} x {D} synthetic (add_synthetic seed {SEED}), L2, k = {K}", "runs": []}
    for storage in (m.STORE_F32, m.STORE_BF16):
        sname = "fp32" if storage == m.STORE_F32 else "bf16"
        ix = m.IndexFlat(D, m.METRIC_L2, storage=storage, device=0)
        ix.add_synthetic(SEED, 0, N)
        base = torch.from_numpy(ix.reconstruct_n(0, 1024)).to(dev)
        xq = base + 0.01 * torch.randn(base.shape, generator=torch.Generator().manual_seed(3)).to(dev)
        radius = float(ix.search(xq, 10)[0][:, -1].median())
        for nq in (1, 32, 1024, "range"):
            q = xq if nq == "range" else xq[:nq]

            def call(sel):
                p = None if sel is None else m.SearchParameters(sel)
                return (lambda: ix.range_search(q, radius, params=p)) if nq == "range" else (lambda: ix.search(q, K, params=p))

            t0 = timed(call(None), a.reps, sync)
            for name, sel in sels.items():
                before = ix.stats()
                t = timed(call(sel), a.reps, sync)
                after = ix.stats()
                row = {"storage": sname, "nq": nq, "selector": name, "unfiltered_ms": t0, "filtered_ms": t, "ratio": t / t0,
                       "last_algo": after["last_algo"]}
                row.update({c: after[c] - before[c] for c in COUNTERS})
                if nq == "range":
                    row["hits"] = ix.last_range_info["hits"]
                result["runs"].append(row)
                print(json.dumps(row), flush=True)
        # the bitmap and masked-bias kernels alone: events around them are not exposed, so time the nq = 1 scan-path
        # search with and without the Not(1 %) filter (same rows read, the filter adds the bitmap build) and the tensor
        # path at nq = 32 (adds the masked bias as well)
        for algo, nq in ((m.ALGO_SCAN, 1), (m.ALGO_TENSOR, 32)):
            ix.set_search_params(algo=algo)
            q = xq[:nq]
            t0 = timed(lambda: ix.search(q, K), a.reps, sync)
            t1 = timed(lambda: ix.search(q, K, params=m.SearchParameters(sels["not_batch_1%"])), a.reps, sync)
            row = {"storage": sname, "filter_overhead": "scan nq=1" if algo == m.ALGO_SCAN else "tensor nq=32",
                   "unfiltered_ms": t0, "filtered_ms": t1, "delta_ms": t1 - t0}
            result["runs"].append(row)
            print(json.dumps(row), flush=True)
        ix.set_search_params(algo=m.ALGO_AUTO)
        del ix
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
