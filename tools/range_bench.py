"""Range search on one B200: BASELINE config 2 (1M x 384 rows from add_synthetic, L2, 1024 queries perturbed from rows), on
fp32 and bf16 storage.  Radii come from a search(k) so that the median hits per query are about 10, 100 and 1000.

Reports, per storage and radius: ms per range search (CUDA-synchronised host clock, after warm-up, median and spread of
--reps calls) next to search(k = 10 / 100) on the same queries; the share of queries served by the exact range scan; host
syncs and kernels per call; the hits per query (median, max); and the exact range scan alone (algo = SCAN) at nq = 1 and
8 as GB/s of algorithmic bytes (both passes counted: 2 x rows x d x 4 B per group of <= 8 queries) against a device copy.
The database (1.5 GB fp32, 0.8 GB bf16) is larger than the 126 MB L2.

usage: python tools/range_bench.py [--reps 20] [--out range_bench.json]
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

N, D, NQ, SEED = 1_000_000, 384, 1024, 1234


def timed(fn, reps, sync):
    fn()
    sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts)}


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
    # the copy peak of this card: a device-to-device copy of 2 GB, read + write bytes
    src = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    cp = timed(lambda: dst.copy_(src), 10, sync)
    copy_gbs = 2 * src.numel() * 4 / (cp["median_ms"] * 1e-3) / 1e9
    del src, dst
    result = {"card": card, "copy_GBps": copy_gbs, "config": f"{N} x {D} synthetic, L2, {NQ} queries perturbed from rows", "runs": []}
    rng = np.random.default_rng(5)
    for storage in (m.STORE_F32, m.STORE_BF16):
        sname = "fp32" if storage == m.STORE_F32 else "bf16"
        ix = m.IndexFlatL2(D, storage=storage)
        ix.add_synthetic(SEED, 0, N)
        rows = ix.reconstruct_n(0, 4096)
        pick = rng.integers(0, 4096, NQ)
        xq = (rows[pick] + 0.05 * rng.standard_normal((NQ, D)) * np.abs(rows[pick]).mean()).astype(np.float32)
        xq_t = torch.from_numpy(xq).cuda()
        for k in (10, 100):
            t = timed(lambda: ix.search(xq_t, k), a.reps, sync)
            result["runs"].append({"storage": sname, "op": f"search k={k}", **t})
            print(sname, f"search k={k}", t, flush=True)
        Dk, _ = ix.search(xq, 1024)
        for target in (10, 100, 1000):
            radius = float(np.median(Dk[:, target - 1]))
            lims, _, _ = ix.range_search(xq_t, radius)
            info = dict(ix.last_range_info)
            hits = np.diff(lims.cpu().numpy())
            s0 = ix.stats()
            t = timed(lambda: ix.range_search(xq_t, radius), a.reps, sync)
            s1 = ix.stats()
            rec = {"storage": sname, "op": f"range_search ~{target}/query", "radius": radius, **t,
                   "median_hits": float(np.median(hits)), "max_hits": int(hits.max()), "hits": info["hits"],
                   "scan_share": info["scan_queries"] / NQ, "host_syncs": info["host_syncs"], "launches": info["launches"],
                   "launches_per_call": (s1["launches"] - s0["launches"]) / (a.reps + 1)}
            result["runs"].append(rec)
            print(rec, flush=True)
        # the exact range scan alone, nq = 1 and 8: algorithmic bytes = 2 passes x the database per group of <= 8 queries
        scan = m.SearchParams()
        scan.algo = m.ALGO_SCAN
        db_bytes = N * D * (4 if storage == m.STORE_F32 else 2)
        radius = float(np.median(Dk[:, 9]))
        for nq in (1, 8):
            t = timed(lambda: ix.range_search(xq_t[:nq], radius, params=scan), a.reps, sync)
            gbs = 2 * db_bytes / (t["median_ms"] * 1e-3) / 1e9
            rec = {"storage": sname, "op": f"exact range scan nq={nq}", **t, "algorithmic_GBps": gbs, "share_of_copy": gbs / copy_gbs}
            result["runs"].append(rec)
            print(rec, flush=True)
        del ix
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        json.dump(result, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
