"""GPU tier, N > 1: the row-sharded index over NCCL (one process per GPU) against a single-GPU index and
the oracle.  Skipped unless at least 2 GPUs are visible (run under `gpurun --gpus 2`)."""
import os
import socket

import numpy as np
import pytest

import oracle as orc

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import rag_faiss_embedding_b200 as b2f

        d, n, nq, k = 128, 60001, 150, 10
        xq = torch.from_numpy(orc.c_synth_rows(5678, 0, nq, d)).cuda()
        for metric in (1, 0):
            ix = b2f.ShardedIndexFlat(d, metric, device=rank)
            ix.add_synthetic(1234, n)            # every rank generates its own slice on its own GPU
            assert ix.ntotal == n
            D, I = ix.search(xq, k)               # replicated queries -> identical merged result on all ranks
            D1, I1 = ix.search(xq[:1], k)         # nq = 1 goes through the streaming scan on every shard
            # the exchange under stress: back-to-back searches of changing size (double-buffered peer slots), a
            # message larger than the first slots (the exchange is re-created collectively), the NCCL form of the
            # same step, host-resident queries (slice upload + all-gather), an empty batch
            outs = [ix.search(xq[: 10 + 7 * i], k) for i in range(8)]
            Db, Ib = ix.search(xq.repeat(250, 1), k)              # 37500 queries: a 4.5 MB message
            os.environ["B200FLAT_EXCHANGE"] = "nccl"
            Dn, In = ix.search(xq, k)
            del os.environ["B200FLAT_EXCHANGE"]
            Dh, Ih = ix.search_host(xq.cpu().pin_memory(), k)
            De, Ie = ix.search(xq[:0], k)
            Dnp, Inp = ix.search(xq.cpu().numpy(), k)             # host queries: one all-gather, numpy results
            Dct, Ict = ix.search(xq.cpu(), k)
            torch.cuda.synchronize()
            same = all(torch.equal(Io, I[: Io.shape[0]]) and torch.equal(Do, D[: Do.shape[0]]) for Do, Io in outs)
            same = same and torch.equal(Ib[:nq], I) and torch.equal(Ib[-nq:], I) and torch.equal(Db[nq:2 * nq], D)
            same = same and torch.equal(In, I) and torch.equal(Dn, D)
            same = same and torch.equal(Ih.cuda(), I) and torch.equal(Dh.cuda(), D) and tuple(Ie.shape) == (0, k)
            same = same and all(isinstance(Dx, np.ndarray) and np.array_equal(Ix, I.cpu().numpy())
                                and np.array_equal(Dx, D.cpu().numpy()) for Dx, Ix in ((Dnp, Inp), (Dct, Ict)))
            # caller-owned result tensors (nothing allocated per search)
            Do, Io = torch.empty_like(D), torch.empty_like(I)
            ix.search(xq, k, out=(Do, Io))
            torch.cuda.synchronize()
            same = same and torch.equal(Io, I) and torch.equal(Do, D)
            # add, search, add, search: the shard offset of the single-segment search must not leak into the
            # multi-segment remap (rows arrive in two adds, so every shard holds two label ranges)
            ix2 = b2f.ShardedIndexFlat(d, metric, device=rank)
            ix2.add_synthetic(1234, 30000)
            Da, Ia = ix2.search(xq, k)
            ix2.add_synthetic(1234, n - 30000)
            D2, I2 = ix2.search(xq, k)
            torch.cuda.synchronize()
            same = same and ix2.ntotal == n and torch.equal(I2, I) and torch.allclose(D2, D, rtol=1e-6)
            same = same and bool((Ia < 30000).all())
            np.savez(os.path.join(out_dir, f"r{rank}_m{metric}.npz"), D=D.cpu().numpy(), I=I.cpu().numpy(),
                     D1=D1.cpu().numpy(), I1=I1.cpu().numpy(), nlocal=ix.local.ntotal, same=bool(same))
    finally:
        dist.destroy_process_group()


def test_sharded_nccl_matches_oracle(tmp_path):
    import torch
    import torch.multiprocessing as mp

    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(world, 8)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d, n, nq, k = 128, 60001, 150, 10
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, nq, d)
    for metric in (1, 0):
        D_ref, I_ref = orc.np_search_f64(xb, xq, k, metric)
        total = 0
        for r in range(world):
            z = np.load(os.path.join(tmp_path, f"r{r}_m{metric}.npz"))
            res = orc.recall_and_errors(z["D"], z["I"], D_ref, I_ref, metric)
            assert res["recall"] == 1.0 and res["id_mismatch"] == 0 and res["max_rel_err"] <= 1e-5, (r, metric, res)
            res1 = orc.recall_and_errors(z["D1"], z["I1"], D_ref[:1], I_ref[:1], metric)
            assert res1["recall"] == 1.0 and res1["id_mismatch"] == 0, (r, metric, res1)
            assert bool(z["same"]), (r, metric, "exchange variants disagree")
            total += int(z["nlocal"])
        assert total == n


def test_two_devices_in_one_process():
    """One process driving indexes on two GPUs (kernel attributes are configured per device): both answer exactly,
    through both search paths, interleaved."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import rag_faiss_embedding_b200 as b2f

    d, n, k = 128, 30000, 10
    xb = orc.c_synth_rows(1234, 0, n, d)
    xq = orc.c_synth_rows(5678, 0, 200, d)
    D_ref, I_ref = orc.np_search_f64(xb, xq, k, 1)
    idx = [b2f.IndexFlat(d, 1, device=dev) for dev in (0, 1)]
    for ix in idx:
        ix.add(xb)
    for algo in (b2f.ALGO_TENSOR, b2f.ALGO_SCAN, b2f.ALGO_TENSOR):
        for ix in (idx[1], idx[0]):
            nq = 200 if algo == b2f.ALGO_TENSOR else 9
            D, I = ix.set_search_params(algo=algo).search(xq[:nq], k)
            r = orc.recall_and_errors(D, I, D_ref[:nq], I_ref[:nq], 1)
            assert r["recall"] == 1.0 and r["id_mismatch"] == 0 and r["max_rel_err"] <= 1e-5, (ix.device, algo, r)
