"""GPU tier of ShardedIndexFlat.range_search: the merge kernel (b2f_merge_range_strided) bit for bit against its numpy
restatement; per-shard IndexFlats on one GPU merged by it against one IndexFlat over every row; the whole sharded path
with two processes sharing one GPU over gloo; and, on >= 2 GPUs, the NCCL path with one process per GPU.

On fp32 storage a shard holds exactly the rows one index would hold, and a range hit's distance does not depend on the
path or the batch (DESIGN 3.5), so merged results must equal one index's bit for bit."""
import os
import socket

import numpy as np
import pytest

import oracle as orc
from tests import exact_checks as ec
from tests.range_merge_reference import np_merge_range, np_union_range, random_parts

pytestmark = pytest.mark.gpu

L2, IP = orc.METRIC_L2, orc.METRIC_INNER_PRODUCT


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _same(a, b):
    """two (lims, D, I) results are identical: lims, labels and distance bits"""
    la, Da, Ia = (np.asarray(t.cpu() if hasattr(t, "cpu") else t) for t in a)
    lb, Db, Ib = (np.asarray(t.cpu() if hasattr(t, "cpu") else t) for t in b)
    return (np.array_equal(la.astype(np.int64), lb.astype(np.int64)) and np.array_equal(Ia, Ib)
            and np.array_equal(Da.view(np.uint32), Db.view(np.uint32)))


def _radius(ix, xq, metric, j):
    """a radius with about j hits per query: the median over queries of the j-th top-k distance"""
    D, _ = ix.search(xq, j + 1)
    return float(np.median(np.asarray(D.cpu() if hasattr(D, "cpu") else D)[:, j]))


# ---- the kernel ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nparts", [1, 2, 3, 8, 32])
@pytest.mark.parametrize("nq", [0, 1, 1000, 5000])
def test_merge_kernel_equals_restatement(nparts, nq):
    import torch

    from rag_faiss_embedding_b200 import sharded

    rng = np.random.default_rng(nparts * 7919 + nq)
    big = (nq // 2, 1 << 20) if nq == 1000 and nparts in (3, 32) else None
    empty_parts = [nparts - 1] if nparts > 1 else []
    empty_queries = [0, nq - 1] if nq > 2 else []
    lims, D, I = random_parts(rng, nparts, nq, 40, empty_parts=empty_parts, empty_queries=empty_queries, big=big)
    want = np_merge_range(lims, D, I)
    assert _same(want, np_union_range(lims, D, I))
    nmax = max(len(i) for i in I)
    off_i, part = sharded._range_layout(max(nmax, 1))
    buf = np.zeros(nparts * part, np.uint8)
    for g in range(nparts):
        buf[g * part: g * part + 4 * len(D[g])] = D[g].view(np.uint8)
        buf[g * part + off_i: g * part + off_i + 8 * len(I[g])] = I[g].view(np.uint8)
    total = int(want[0][-1])
    Dm = torch.full((max(total, 4),), float("nan"), dtype=torch.float32, device="cuda")
    Im = torch.full((max(total, 4),), -7, dtype=torch.int64, device="cuda")
    lims_d = torch.from_numpy(lims).cuda()
    sharded.merge_range_strided(lims_d, torch.from_numpy(buf).cuda(), part, off_i, Dm, Im)
    torch.cuda.synchronize()
    assert _same(want, (want[0], Dm[:total], Im[:total]))
    assert bool((Im[total:] == -7).all())   # nothing written past the result
    if nparts == 32:
        from rag_faiss_embedding_b200 import _capi

        lims33 = torch.zeros((33, nq + 1), dtype=torch.int64, device="cuda")
        rc = _capi.load().b2f_merge_range_strided(nq, 33, lims33.data_ptr(), Dm.data_ptr(), Im.data_ptr(), 16,
                                                  Dm.data_ptr(), Im.data_ptr(), 0, None)
        assert rc == _capi.EINVAL


# ---- shards on one GPU, merged by merge_range ----------------------------------------------------------------------
def _shards(m, rows, G, metric, storage):
    """G IndexFlats on one GPU; shard g holds blocks g and G + g of 2 G blocks (two label segments each)"""
    from rag_faiss_embedding_b200.sharded import SegmentMap

    blocks = np.array_split(np.arange(len(rows)), 2 * G)
    out = []
    for g in range(G):
        ix = m.IndexFlat(rows.shape[1], metric, storage=storage, device=0)
        seg = SegmentMap()
        for b in (blocks[g], blocks[G + g]):
            ix.add(rows[b])
            seg.append(int(b[0]), len(b))
        assert seg.monotone()
        out.append((ix, seg))
    return out


def _merged(shards, xq, radius, params):
    from rag_faiss_embedding_b200.sharded import merge_range

    parts = []
    for ix, seg in shards:
        lims, D, I = ix.range_search(xq, radius, params=params)
        parts.append((lims, D, seg.to_global_torch(I)))
    return merge_range(parts)


@pytest.mark.parametrize("metric", [L2, IP])
def test_shards_merged_equal_one_index(metric):
    import torch

    import rag_faiss_embedding_b200 as m

    d, n = 128, 20000
    rows = orc.c_synth_rows(31, 0, n, d)
    xq = torch.from_numpy(orc.c_synth_rows(32, 0, 300, d)).cuda()
    xq[5] = torch.from_numpy(rows[77]).cuda()
    one = m.IndexFlat(d, metric, storage=m.STORE_F32, device=0)
    one.add(rows)
    radius = _radius(one, xq, metric, 30)
    for G in (1, 3, 4):
        shards = _shards(m, rows, G, metric, m.STORE_F32)
        for algo in (m.ALGO_TENSOR, m.ALGO_SCAN):
            p = m.SearchParams(algo=algo)
            want = one.range_search(xq, radius, params=p)
            got = _merged(shards, xq, radius, p)
            assert int(want[0][-1]) > 0
            assert _same(got, want), (G, algo)


@pytest.mark.parametrize("metric", [L2, IP])
def test_shards_merged_exact_on_lattice(metric):
    import torch

    import rag_faiss_embedding_b200 as m

    lat = ec.lattice(12000, 64, 4, seed=3)
    xq = lat.near(64)
    lat.verify(xq)
    one = m.IndexFlat(64, metric, storage=m.STORE_F32, device=0)
    one.add(lat.rows)
    radius = _radius(one, xq, metric, 50)
    shards = _shards(m, lat.rows, 3, metric, m.STORE_F32)
    for algo in (m.ALGO_TENSOR, m.ALGO_SCAN):
        lims, D, I = _merged(shards, torch.from_numpy(xq).cuda(), radius, m.SearchParams(algo=algo))
        ec.check_range_exact(lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy(), lat.rows, xq, radius, metric)


# ---- two processes sharing one GPU, gloo ---------------------------------------------------------------------------
# Only range_search, add and remove_ids run on these indexes: the top-k path's peer exchange spin-waits on the other
# rank's flag, and two contexts time-slicing one GPU must not be put in that position.
def _one_gpu_worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import rag_faiss_embedding_b200 as m
        from rag_faiss_embedding_b200 import sharded

        d = 96
        z = np.load(os.path.join(out_dir, "in.npz"))
        xq = torch.from_numpy(z["xq"]).cuda()
        out = {}
        for metric in (L2, IP):
            r = float(z[f"r{metric}"])
            ix = m.ShardedIndexFlat(d, metric, storage=m.STORE_F32, device=0)
            ix.add(z["xb1"])
            res = {"a": ix.range_search(xq, r)}
            ix.add(z["xb2"])
            res["b"] = ix.range_search(xq, r)
            res["b_np"] = ix.range_search(z["xq"], r)
            ix.remove_ids(m.IDSelectorRange(100, 900))
            res["c"] = ix.range_search(xq, r)
            sharded.RANGE_PART_BYTES = 4096
            res["c_chunked"] = ix.range_search(xq, r)
            out[f"chunks{metric}"] = ix.last_range_info["chunks"]
            sharded.RANGE_PART_BYTES = 256 << 20
            res["empty"] = ix.range_search(xq[:0], r)
            for k, (lims, D, I) in res.items():
                for name, t in (("lims", lims), ("D", D), ("I", I)):
                    out[f"{metric}_{k}_{name}"] = t.cpu().numpy() if hasattr(t, "cpu") else t
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **out)
    finally:
        dist.destroy_process_group()


def test_two_processes_on_one_gpu(tmp_path):
    import torch
    import torch.multiprocessing as mp

    import rag_faiss_embedding_b200 as m

    d = 96
    xb1 = orc.c_synth_rows(41, 0, 7001, d)
    xb2 = orc.c_synth_rows(41, 7001, 3000, d)
    xq = orc.c_synth_rows(42, 0, 200, d)
    db = np.concatenate([xb1, xb2])
    radii = {}
    for metric in (L2, IP):
        one = m.IndexFlat(d, metric, storage=m.STORE_F32, device=0)
        one.add(db)
        radii[f"r{metric}"] = _radius(one, xq, metric, 20)
        del one
    np.savez(os.path.join(tmp_path, "in.npz"), xb1=xb1, xb2=xb2, xq=xq, **radii)
    mp.spawn(_one_gpu_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    zs = [np.load(os.path.join(tmp_path, f"r{k}.npz")) for k in range(2)]
    for metric in (L2, IP):
        r = radii[f"r{metric}"]
        dbs = {"a": xb1, "b": db, "c": np.delete(db, np.arange(100, 900), axis=0)}
        for key, rows in dbs.items():
            one = m.IndexFlat(d, metric, storage=m.STORE_F32, device=0)
            one.add(rows)
            want = one.range_search(torch.from_numpy(xq).cuda(), r)
            assert int(want[0][-1]) > 0
            keys = [key] + {"b": ["b_np"], "c": ["c_chunked"]}.get(key, [])
            for z in zs:
                for k in keys:
                    got = tuple(z[f"{metric}_{k}_{name}"] for name in ("lims", "D", "I"))
                    assert _same(got, want), (metric, k)
                assert z[f"{metric}_b_np_lims"].dtype == np.uint64
                assert int(z[f"chunks{metric}"]) > 1
                assert z[f"{metric}_empty_lims"].tolist() == [0] and len(z[f"{metric}_empty_I"]) == 0


# ---- >= 2 GPUs, NCCL -----------------------------------------------------------------------------------------------
def _nccl_worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ok = {}
    try:
        import rag_faiss_embedding_b200 as m
        from rag_faiss_embedding_b200 import sharded

        d, n1, n2, k = 128, 30011, 20000, 10
        xq_np = orc.c_synth_rows(52, 0, 400, d)
        xq = torch.from_numpy(xq_np).cuda()
        for storage in (m.STORE_F32, m.STORE_BF16):
            for metric in (L2, IP):
                tag = f"s{storage}_m{metric}"
                ix = m.ShardedIndexFlat(d, metric, storage=storage, device=rank)
                ix.add_synthetic(51, n1)
                one = m.IndexFlat(d, metric, storage=m.STORE_F32, device=rank)   # every row, on this rank's GPU
                one.add_synthetic(51, 0, n1)
                r = _radius(one, xq, metric, 40)
                part = one.range_search(xq, r)   # the first n1 rows only
                one.add_synthetic(51, n1, n2)   # the rows ix.add_synthetic(51, n2) adds below
                full = one.range_search(xq, r)
                Dk0, Ik0 = ix.search(xq, k)
                results = {"add1": ix.range_search(xq, r)}
                ix.add_synthetic(51, n2)
                Dk1, Ik1 = ix.search(xq, k)
                results["add2"] = ix.range_search(xq, r)
                Dk2, Ik2 = ix.search(xq, k)
                torch.cuda.synchronize()
                ok[tag + "_topk"] = bool(torch.equal(Ik1, Ik2) and torch.equal(Dk1, Dk2) and Ik0.shape == (400, k))
                results["numpy"] = ix.range_search(xq_np, r)
                results["nohit"] = ix.range_search(xq, -1.0 if metric == L2 else 1e30)
                results["empty"] = ix.range_search(xq[:0], r)
                sharded.RANGE_PART_BYTES = 1 << 16
                results["chunked"] = ix.range_search(xq, r)
                ok[tag + "_chunks"] = ix.last_range_info["chunks"] > 1
                sharded.RANGE_PART_BYTES = 256 << 20
                ix.remove_ids(m.IDSelectorRange(1000, 31000))
                one.remove_ids(m.IDSelectorRange(1000, 31000))
                results["removed"] = ix.range_search(xq, r)
                Dk3, Ik3 = ix.search(xq, k)
                Dw, Iw = one.search(xq, k)
                torch.cuda.synchronize()
                if storage == m.STORE_F32:
                    ok[tag + "_add1"] = _same(results["add1"], part)
                    for key in ("add2", "numpy", "chunked"):
                        ok[tag + "_" + key] = _same(results[key], full)
                    ok[tag + "_removed"] = _same(results["removed"], one.range_search(xq, r))
                    ok[tag + "_topk_single"] = bool(torch.equal(Iw, Ik3) and torch.allclose(Dw, Dk3, rtol=1e-5))
                else:
                    # bf16: every shard rounds around its own centre; the result is the union of the shards' own results
                    ix.local.set_search_params(id_offset=0)
                    lims, D, I = ix.local.range_search(xq, r)
                    I = ix.segments.to_global_torch(I)
                    parts = [None] * world
                    dist.all_gather_object(parts, (lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()))
                    want = np_union_range(np.stack([p[0] for p in parts]), [p[1] for p in parts], [p[2] for p in parts])
                    ok[tag + "_removed"] = _same(results["removed"], want)
                ok[tag + "_numpy_type"] = results["numpy"][0].dtype == np.uint64
                ok[tag + "_nohit"] = int(results["nohit"][0][-1]) == 0 and len(results["nohit"][2]) == 0
                ok[tag + "_empty"] = results["empty"][0].tolist() == [0]
                ok[tag + "_chunked_same"] = _same(results["chunked"], results["add2"])
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **ok)
    finally:
        dist.destroy_process_group()


def test_sharded_range_nccl():
    import tempfile

    import torch
    import torch.multiprocessing as mp

    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(world, 8)
    with tempfile.TemporaryDirectory() as out_dir:
        mp.spawn(_nccl_worker, args=(world, _free_port(), out_dir), nprocs=world, join=True)
        for r in range(world):
            z = np.load(os.path.join(out_dir, f"r{r}.npz"))
            bad = [k for k in z.files if not bool(z[k])]
            assert not bad and len(z.files) > 20, (r, bad)
