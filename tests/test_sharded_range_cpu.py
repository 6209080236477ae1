"""CPU tier of ShardedIndexFlat.range_search: the merge's numpy restatement against a sort-based union, the query
chunking, the C-ABI argument checks of b2f_merge_range_strided, and the whole sharded path (lims all-gather, chunked hit
all-gathers, merge) on gloo with world sizes 2 and 3 over oracle-backed shards, against a float64 range search of the
concatenated database.  Integer data keeps every distance exact, so results must be equal, not close."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as orc
from tests.helpers import OracleIndex
from tests.range_merge_reference import np_merge_range, np_range_merge_fn, np_union_range, random_parts
from tests.range_reference import np_range_search_f64

D_DIM = 16


class RangeOracleIndex(OracleIndex):
    """OracleIndex with range_search over the float64 reference and faiss's remove_ids."""

    def range_search(self, x, radius, params=None):
        x = np.ascontiguousarray(x, np.float32)
        if x.ndim != 2 or x.shape[1] != self.d:
            raise AssertionError("dimension mismatch")
        lims, D, I = np_range_search_f64(self.x, x, radius, self.metric_type)
        off = self._offset if params is None else int(params.id_offset)
        self.last_range_info = {"hits": int(lims[-1]), "tensor_queries": 0, "scan_queries": len(x), "launches": 0,
                                "host_syncs": 0}
        return lims.astype(np.uint64), D.astype(np.float32), I + off

    def remove_ids(self, ids):
        ids = np.asarray(ids, np.int64)
        ids = np.unique(ids[(ids >= 0) & (ids < self.ntotal)])
        self.x = np.delete(self.x, ids, axis=0)
        return int(len(ids))


# ---- the merge -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nparts", [1, 2, 3, 7, 32])
@pytest.mark.parametrize("nq", [0, 1, 40])
def test_merge_restatement_equals_sorted_union(nparts, nq):
    rng = np.random.default_rng(nparts * 100 + nq)
    empty_parts = [0] if nparts > 2 else []
    empty_queries = [q for q in (0, 5) if q < nq and nq > 1]
    lims, D, I = random_parts(rng, nparts, nq, 60, empty_parts=empty_parts, empty_queries=empty_queries)
    assert nparts == 1 or lims[:, 0].any(), "bases should not all be 0"
    got = np_merge_range(lims, D, I)
    want = np_union_range(lims, D, I)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))   # distances moved bit for bit
    for q in range(nq):
        assert np.all(np.diff(got[2][got[0][q]:got[0][q + 1]]) > 0)


def test_range_chunks_cap_each_rank_and_isolate_big_queries(monkeypatch):
    from rag_faiss_embedding_b200 import sharded

    monkeypatch.setattr(sharded, "RANGE_PART_BYTES", 32 + 12 * 10)   # 10 hits per rank per gather
    counts = np.array([[3, 3, 3, 30, 0, 4, 4, 4, 0, 0],
                       [1, 1, 1, 1, 11, 1, 1, 1, 0, 0]])
    lims = np.stack([np.concatenate([[0], np.cumsum(c)]) for c in counts]) + np.array([[5], [0]])   # any base
    chunks = sharded.ShardedIndexFlat._range_chunks(lims)
    assert chunks == [(0, 3), (3, 4), (4, 5), (5, 7), (7, 10)]
    for q0, q1 in chunks:
        n = lims[:, q1] - lims[:, q0]
        assert q1 - q0 == 1 or n.max() <= 10
        assert sharded._packed_layout(int(n.max()))[1] <= sharded.RANGE_PART_BYTES or q1 - q0 == 1
    assert sharded.ShardedIndexFlat._range_chunks(np.zeros((3, 1), np.int64)) == []


def test_segment_map_monotone():
    from rag_faiss_embedding_b200.sharded import SegmentMap

    s = SegmentMap()
    assert s.monotone()
    s.append(10, 5)
    s.append(40, 5)
    assert s.monotone()
    s.append(20, 3)
    assert not s.monotone()
    s = SegmentMap()
    s.append(10, 5)
    s.append(12, 5)   # overlaps the first segment's labels: not label order either
    assert not s.monotone()


def test_merge_range_c_abi_arguments():
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    buf = (ctypes.c_int64 * 64)()
    p = ctypes.addressof(buf)
    f = lib.b2f_merge_range_strided
    assert f(1, 0, p, p, p, 16, p, p, 0, None) == _capi.EINVAL          # nparts < 1
    assert f(1, 33, p, p, p, 16, p, p, 0, None) == _capi.EINVAL         # nparts > 32
    assert f(-1, 2, p, p, p, 16, p, p, 0, None) == _capi.EINVAL         # nq < 0
    assert f(1, 2, None, p, p, 16, p, p, 0, None) == _capi.EINVAL       # no lims
    assert f(1, 2, p, None, p, 16, p, p, 0, None) == _capi.EINVAL       # NULL hits with queries present
    assert f(1, 2, p, p, p, 16, p, None, 0, None) == _capi.EINVAL
    assert f(1, 2, p, p, p, 24, p, p, 0, None) == _capi.EINVAL          # stride not a multiple of 16
    assert f(1, 2, p, p, p, 0, p, p, 0, None) == _capi.EINVAL
    assert f(1, 2, p, p, p + 4, 16, p, p, 0, None) == _capi.EINVAL      # misaligned labels
    import rag_faiss_embedding_b200 as m

    if m.device_count() == 0:
        assert f(1, 2, p, p, p, 16, p, p, 0, None) == _capi.ENOGPU
        assert f(0, 1, p, None, None, 16, None, None, 0, None) == _capi.ENOGPU   # nq = 0: no hit pointers needed


# ---- the sharded path on gloo --------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _data():
    rng = np.random.default_rng(7)
    rows = lambda n: rng.integers(-3, 4, (n, D_DIM)).astype(np.float32)   # noqa: E731
    xb1, xb2, xb3, xq = rows(300), rows(157), rows(61), rows(12)
    xq[3] = xb1[17]
    return xb1, xb2, xb3, xq


RADIUS = {orc.METRIC_L2: 90.0, orc.METRIC_INNER_PRODUCT: 20.0}
REMOVE_RANGE = (50, 120)
REMOVE_BATCH = np.array([0, 3, 3, 200, 299, 351, 384, 386, 10 ** 6, -2])


def _edge_cases(metric, xq):
    """(name, queries, radius) run on the final database: no hit, L2 radius <= 0 / IP everything, nq = 0"""
    if metric == orc.METRIC_L2:
        return [("nohit", xq + 0.5, 1.0), ("zero", xq, 0.0), ("negative", xq, -1.0), ("empty", xq[:0], 90.0)]
    return [("nohit", xq, 1e6), ("all", xq, -1e9), ("empty", xq[:0], 20.0)]


def _worker(rank, world, port, metric, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from rag_faiss_embedding_b200 import IDSelectorBatch, IDSelectorRange, sharded
        from rag_faiss_embedding_b200.sharded import ShardedIndexFlat

        xb1, xb2, xb3, xq = _data()
        r = RADIUS[metric]
        out = {}

        def run(name, q=xq, radius=r):
            lims, D, I = ix.range_search(q, radius)
            assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
            out[name + "_lims"], out[name + "_D"], out[name + "_I"] = lims, D, I
            out[name + "_chunks"] = ix.last_range_info["chunks"]

        ix = ShardedIndexFlat(D_DIM, metric, local_index=RangeOracleIndex(D_DIM, metric), range_merge_fn=np_range_merge_fn)
        ix.add(xb1)
        run("add1")
        ix.add(xb2)                       # two segments per shard, labels interleaved across ranks
        run("add2")
        ix.remove_ids(IDSelectorRange(*REMOVE_RANGE))
        ix.remove_ids(IDSelectorBatch(REMOVE_BATCH))
        run("removed")
        # add_local: rank r first takes piece world + r, then the lower-labelled piece r -- a segment below an earlier one
        pieces = np.array_split(np.arange(len(xb3)), 2 * world)
        for piece in (pieces[world + rank], pieces[rank]):
            ix.add_local(xb3[piece], ix.ntotal + int(piece[0]))
        ix.set_total(ix.ntotal + len(xb3))
        assert not ix.segments.monotone()
        run("local")
        for name, q, radius in _edge_cases(metric, xq):
            run(name, q, radius)
        # a cap of a few hits per rank and gather: several chunks, the largest query in one of its own
        per_q = np.diff(out["local_lims"].astype(np.int64))
        budget = max(1, int(per_q.max()) // (2 * world))
        sharded.RANGE_PART_BYTES = 32 + 12 * budget
        run("chunked")
        sharded.RANGE_PART_BYTES = 256 << 20
        with pytest.raises(AssertionError):
            ix.range_search(xq[:, :-1], r)
        with pytest.raises(RuntimeError):
            ix.range_search(xq, float("nan"))
        ix.reset()
        ix.add(xb2)
        run("reset")
        out["nlocal"] = ix.local.ntotal
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **out)
    finally:
        dist.destroy_process_group()


def _check(z, name, rows, q, radius, metric):
    rl, rD, rI = np_range_search_f64(rows, q, radius, metric)
    lims = z[name + "_lims"].astype(np.int64)
    assert np.array_equal(lims, rl), name
    assert np.array_equal(z[name + "_I"], rI), name
    assert np.array_equal(z[name + "_D"], rD.astype(np.float32)), name


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("metric", [orc.METRIC_L2, orc.METRIC_INNER_PRODUCT])
def test_sharded_range_equals_single(tmp_path, world, metric):
    mp.spawn(_worker, args=(world, _free_port(), metric, str(tmp_path)), nprocs=world, join=True)
    xb1, xb2, xb3, xq = _data()
    r = RADIUS[metric]
    db1 = xb1
    db2 = np.concatenate([xb1, xb2])
    db3 = np.delete(db2, np.arange(*REMOVE_RANGE), axis=0)
    ids = np.unique(REMOVE_BATCH[(REMOVE_BATCH >= 0) & (REMOVE_BATCH < len(db3))])
    db3 = np.delete(db3, ids, axis=0)
    db4 = np.concatenate([db3, xb3])
    zs = [np.load(os.path.join(tmp_path, f"r{k}.npz")) for k in range(world)]
    for z in zs:
        _check(z, "add1", db1, xq, r, metric)
        _check(z, "add2", db2, xq, r, metric)
        _check(z, "removed", db3, xq, r, metric)
        _check(z, "local", db4, xq, r, metric)
        _check(z, "chunked", db4, xq, r, metric)
        for name, q, radius in _edge_cases(metric, xq):
            _check(z, name, db4, q, radius, metric)
        _check(z, "reset", xb2, xq, r, metric)
        assert int(z["local_chunks"]) == 1 and int(z["chunked_chunks"]) > 2
        assert int(z["nohit_chunks"]) == 0 and int(z["empty_chunks"]) == 0
    assert sum(int(z["nlocal"]) for z in zs) == len(xb2)
    assert int(zs[0]["local_lims"][-1]) > 0 and int(zs[0]["nohit_lims"][-1]) == 0
