"""remove_ids on one B200: BASELINE config 2 (1M x 384 from add_synthetic, fp32 and bf16 storage) and config 3 (10M x 768,
fp32), L2.

Patterns: row 0 (every row moves by one), 1 % random ids, the first half as a range, and the last row only (nothing
moves: the stats pass alone).  Per pattern: the median ms of --reps fresh removals (the index is rebuilt between them;
remove_ids is synchronous, timed with a host clock); the bytes the compaction moves, from the shapes (every moved row of
every array read once and written once); that traffic as GB/s next to a 2 GB device-to-device copy measured in the same
run (read + write bytes); and the rebuild workaround on the same rows (reconstruct_n into a device buffer, reset, add).
Parity: 256 sampled survivors reconstruct to the bits of their generated rows (bf16 storage: rounded around the first
add's centre), and a 64-query search after the removal against the rebuilt index: the share of equal ids and the largest
relative distance difference (the rebuild's reset takes a new centre, so its tensor pass certifies differently and a query
may be served by another path; bf16 storage also rounds every row again).

usage: python tools/remove_bench.py [--reps 3] [--configs c2,c3] [--out remove_bench.json]
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
import oracle as orc  # noqa: E402
import rag_faiss_embedding_b200 as m  # noqa: E402

CONFIGS = {"c2": [(1_000_000, 384, m.STORE_F32), (1_000_000, 384, m.STORE_BF16)], "c3": [(10_000_000, 768, m.STORE_F32)]}
SEED = 1234


def patterns(n):
    rng = np.random.default_rng(7)
    return {
        "row0": np.array([0], np.int64),
        "random1pct": np.sort(rng.choice(n, n // 100, replace=False)).astype(np.int64),
        "first_half": m.IDSelectorRange(0, n // 2),
        "last_row": np.array([n - 1], np.int64),
    }


def removed_rows(n, sel):
    if isinstance(sel, m.IDSelectorRange):
        return np.arange(sel.imin, sel.imax)
    return sel


def moved_bytes(n, d, storage, gone):
    """Bytes the compaction reads and writes: the survivors above the first removed row, in all three arrays."""
    moved = (n - int(gone[0])) - len(gone)
    dpad = (d + 63) // 64 * 64
    row = (d * 4 if storage == m.STORE_F32 else 0) + dpad * 2 + 4
    return 2 * moved * row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    assert m.device_count() > 0, "remove_bench needs a B200"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card, flush=True)
    sync = torch.cuda.synchronize
    src = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    sync()
    ts = []
    for _ in range(10):
        t0 = time.perf_counter()
        dst.copy_(src)
        sync()
        ts.append(time.perf_counter() - t0)
    copy_gbs = 2 * src.numel() * 4 / statistics.median(ts) / 1e9
    del src, dst
    print(f"device copy of 2 GB: {copy_gbs:.0f} GB/s (read + write)", flush=True)
    out = {"card": card, "copy_GBps": copy_gbs, "reps": a.reps, "runs": []}
    for cname in a.configs.split(","):
        for n, d, storage in CONFIGS[cname]:
            sname = "fp32" if storage == m.STORE_F32 else "bf16"
            xq = torch.from_numpy(orc.c_synth_rows(SEED + 1, 0, 64, d)).cuda()

            def fresh():
                ix = m.IndexFlat(d, m.METRIC_L2, storage=storage)
                ix.reserve(n)
                ix.add_synthetic(SEED, 0, n)
                return ix

            ix = fresh()
            ix.remove_ids(np.array([n - 1]))   # warm-up: modules, workspace, flags
            mu = orc.np_centre(orc.c_synth_rows(SEED, 0, min(n, 65536), d)) if storage == m.STORE_BF16 else None
            for pname, sel in patterns(n).items():
                gone = removed_rows(n, sel)
                ms = []
                for _ in range(a.reps):
                    del ix
                    ix = fresh()
                    sync()
                    t0 = time.perf_counter()
                    assert ix.remove_ids(sel) == len(gone)
                    ms.append((time.perf_counter() - t0) * 1e3)
                D1, I1 = ix.search(xq, 10)
                kept = np.delete(np.arange(n), gone)
                pos = np.sort(np.random.default_rng(len(gone)).choice(len(kept), 256, replace=False))
                want = np.concatenate([orc.c_synth_rows(SEED, int(kept[p_]), 1, d) for p_ in pos])
                if mu is not None:
                    want = orc.np_bf16_rows(want, mu)
                got = np.stack([ix.reconstruct(int(p_)) for p_ in pos])
                rows_exact = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
                # the rebuild workaround on the same rows (its first run also warms up its allocations: not counted)
                rb = []
                for _ in range(a.reps + 1):
                    del ix
                    ix = fresh()
                    sync()
                    t0 = time.perf_counter()
                    keep = torch.ones(n, dtype=torch.bool, device="cuda")
                    keep[torch.from_numpy(np.asarray(gone)).cuda()] = False
                    rows = torch.empty((n, d), dtype=torch.float32, device="cuda")
                    C = m._capi
                    C.check(ix._lib.b2f_index_reconstruct(ix._h, 0, n, rows.data_ptr(), C.MEM_DEVICE, None))
                    rows = rows[keep]
                    ix.reset()
                    ix.add(rows)
                    sync()
                    rb.append((time.perf_counter() - t0) * 1e3)
                    del rows, keep
                rebuild_ms = statistics.median(rb[1:])
                D2, I2 = ix.search(xq, 10)
                sync()
                I1, I2, D1, D2 = I1.cpu().numpy(), I2.cpu().numpy(), D1.cpu().numpy(), D2.cpu().numpy()
                ids_equal = float(np.mean(I1 == I2))
                rel = float(np.max(np.abs(D1.astype(np.float64) - D2) / np.maximum(np.abs(D2.astype(np.float64)), 1e-30)))
                med = statistics.median(ms)
                mb = moved_bytes(n, d, storage, gone)
                r = {"config": cname, "n": n, "d": d, "storage": sname, "pattern": pname, "removed": int(len(gone)),
                     "remove_ms_median": med, "remove_ms_all": ms, "moved_GB": mb / 1e9,
                     "GBps": mb / (med * 1e-3) / 1e9 if mb else 0.0, "rebuild_ms": rebuild_ms,
                     "rows_exact": rows_exact, "ids_equal": ids_equal, "max_rel_D": rel}
                out["runs"].append(r)
                print(f"{cname} {sname:4s} {pname:11s} removed {len(gone):>8d}: {med:8.2f} ms, moved {mb / 1e9:6.2f} GB "
                      f"({r['GBps']:6.0f} GB/s = {100 * r['GBps'] / copy_gbs:5.1f} % of copy); rebuild {rebuild_ms:8.2f} ms; "
                      f"rows exact {rows_exact}, ids equal {ids_equal:.4f}, max rel D {rel:.1e}", flush=True)
            del ix
            torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
