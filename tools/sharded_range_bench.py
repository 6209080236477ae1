"""Range search over a row-sharded index: BASELINE config 2 (1M x 384 rows from add_synthetic, L2, fp32 storage) split over
the ranks of a torchrun job, 1024 queries perturbed from rows, radii from a search(k) so that the median hits per query are
about 10, 100 and 1000 (as tools/range_bench.py).

Reports per radius: ms per ShardedIndexFlat.range_search (median of --reps calls after warm-up, host clock around a call
that ends in a device synchronise and a barrier); the local range search alone (the slowest rank's median); their
difference (lims all-gather + hit all-gathers + merges); the merge kernel's CUDA-event time in the sharded call and its
rate over the bytes it must move (read: 12 B per hit + the parts' lims; written: 12 B per hit); gathered_bytes; and the
single-GPU IndexFlat.range_search over the same 1M rows.  Also, on one GPU whatever the world size: the merge kernel alone
on the single-GPU result cut into G = 2 and 8 row-range parts (what G shards would send), so its rate is measured even
where only one GPU is available.  The card's name and power limit are read in the same run.

usage: torchrun --nproc_per_node N tools/sharded_range_bench.py [--reps 20] [--out sharded_range_bench.json]
       (N = 1 also runs without torchrun)
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
from rag_faiss_embedding_b200 import sharded  # noqa: E402

N, D, NQ, SEED = 1_000_000, 384, 1024, 1234


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(fn):
        fn()
        sync()
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            fn()
            sync()
            ts.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(ts)

    def slowest(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    card = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    merge_ms = []   # CUDA-event time of every merge launch of the sharded call being measured

    def timed_merge(lims_parts, recv, part_bytes, off_i, Dm, Im):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sharded.merge_range_strided(lims_parts, recv, part_bytes, off_i, Dm, Im)
        e1.record()
        merge_ms.append((e0, e1))

    ix = m.ShardedIndexFlat(D, m.METRIC_L2, storage=m.STORE_F32, device=dev, range_merge_fn=timed_merge)
    ix.add_synthetic(SEED, N)
    one = m.IndexFlatL2(D, storage=m.STORE_F32, device=dev)   # the single-GPU comparison, on every rank's GPU
    one.add_synthetic(SEED, 0, N)
    rng = np.random.default_rng(5)
    rows = orc.c_synth_rows(SEED, 0, 4096, D)
    pick = rng.integers(0, 4096, NQ)
    xq = (rows[pick] + 0.05 * rng.standard_normal((NQ, D)) * np.abs(rows[pick]).mean()).astype(np.float32)
    xq_t = torch.from_numpy(xq).cuda()
    Dk, _ = one.search(xq_t, 1024)
    Dk = Dk.cpu().numpy()
    result = {"card": card, "world": world, "config": f"{N} x {D} synthetic, L2, fp32 storage, {NQ} queries perturbed from rows",
              "reps": a.reps, "runs": []}
    off = ix.segments.single_offset()
    for target in (10, 100, 1000):
        radius = float(np.median(Dk[:, target - 1]))
        lims, _, _ = ix.range_search(xq_t, radius)
        info = dict(ix.last_range_info)
        hits = np.diff(lims.cpu().numpy())
        t_sharded = timed(lambda: ix.range_search(xq_t, radius))
        del merge_ms[:]
        ix.range_search(xq_t, radius)
        sync()
        t_merge = slowest(sum(e0.elapsed_time(e1) for e0, e1 in merge_ms))
        ix.local.set_search_params(id_offset=off)
        t_local = slowest(timed(lambda: ix.local.range_search(xq_t, radius)))
        t_one = timed(lambda: one.range_search(xq_t, radius))
        total = int(lims[-1])
        moved = 12 * total * 2 + 8 * world * (NQ + 1)
        rec = {"op": f"range_search ~{target}/query", "radius": radius, "median_hits": float(np.median(hits)),
               "max_hits": int(hits.max()), "hits": total, "sharded_ms": t_sharded, "local_ms_slowest_rank": t_local,
               "gather_and_merge_ms": t_sharded - t_local, "merge_kernel_ms": t_merge,
               "merge_GBps": moved / (t_merge * 1e-3) / 1e9 if t_merge > 0 else None, "chunks": info["chunks"],
               "gathered_bytes": info["gathered_bytes"], "single_gpu_ms": t_one}
        # the merge kernel alone on this GPU: the single-GPU result cut into G row-range parts, packed as G ranks send them
        lo, Do, Io = one.range_search(xq_t, radius)
        for G in (2, 8):
            bounds = torch.tensor([s for s, _ in sharded.partition_rows(N, G)][1:], device="cuda")
            part_of = torch.bucketize(Io, bounds, right=True)
            qid = torch.repeat_interleave(torch.arange(NQ, device="cuda"), lo.diff(), output_size=total)
            lims_parts = torch.zeros((G, NQ + 1), dtype=torch.int64, device="cuda")
            parts = []
            for g in range(G):
                sel = part_of == g
                lims_parts[g, 1:] = torch.bincount(qid[sel], minlength=NQ).cumsum(0)
                parts.append((Do[sel], Io[sel]))
            nmax = max(int(p[0].numel()) for p in parts)
            off_i, part = sharded._range_layout(nmax)
            recv = torch.zeros(G * part, dtype=torch.uint8, device="cuda")
            for g, (dp, ip) in enumerate(parts):
                recv[g * part: g * part + 4 * dp.numel()].view(torch.float32).copy_(dp)
                recv[g * part + off_i: g * part + off_i + 8 * ip.numel()].view(torch.int64).copy_(ip)
            Dm, Im = torch.empty_like(Do), torch.empty_like(Io)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sharded.merge_range_strided(lims_parts, recv, part, off_i, Dm, Im)
            e0.record()
            for _ in range(a.reps):
                sharded.merge_range_strided(lims_parts, recv, part, off_i, Dm, Im)
            e1.record()
            torch.cuda.synchronize()
            assert torch.equal(Im, Io) and torch.equal(Dm.view(torch.int32), Do.view(torch.int32)), "merge != single GPU"
            ms = e0.elapsed_time(e1) / a.reps
            rec[f"merge_alone_G{G}_ms"] = ms
            rec[f"merge_alone_G{G}_GBps"] = (24 * total + 8 * G * (NQ + 1)) / (ms * 1e-3) / 1e9
        result["runs"].append(rec)
        if rank == 0:
            print(json.dumps(rec), flush=True)
    if rank == 0:
        print("card:", card, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
            json.dump(result, open(a.out, "w"), indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
