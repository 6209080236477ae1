"""CPU tier of index.remove_ids: the run list and where each row goes (the host build of the function the compaction
kernel uses) against numpy bookkeeping, the compaction's tile waits, the selector surface, the sharded renumbering on
gloo, and FAISSVectorStore.remove_documents -- all without a GPU."""
import ctypes
import os
import pickle
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as orc
from tests.helpers import OracleIndex, np_topk_merge_fn

TILE_BYTES = 32 << 10   # kRemoveTileBytes


class RemovableOracleIndex(OracleIndex):
    """OracleIndex with faiss's remove_ids over np.delete (1-D id arrays)."""

    def remove_ids(self, ids):
        ids = np.asarray(ids, np.int64)
        ids = np.unique(ids[(ids >= 0) & (ids < self.ntotal)])
        self.x = np.delete(self.x, ids, axis=0)
        return int(len(ids))


def _plan(ntotal, ids, row_bytes=4):
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    ids = np.ascontiguousarray(ids, np.int64)
    runs = np.zeros(max(2 * len(ids), 2), np.int64)
    dest = np.zeros(max(ntotal, 1), np.int64)
    nruns, ntiles = ctypes.c_int64(), ctypes.c_int64()
    rc = lib.b2f_remove_plan(ntotal, len(ids), ids.ctypes.data, row_bytes, runs.ctypes.data, ctypes.byref(nruns),
                             dest.ctypes.data, None, 0, ctypes.byref(ntiles))
    assert rc == 0, _capi.last_error()
    tiles = np.zeros(3 * max(ntiles.value, 1), np.int64)
    rc = lib.b2f_remove_plan(ntotal, len(ids), ids.ctypes.data, row_bytes, None, ctypes.byref(nruns), None,
                             tiles.ctypes.data, ntiles.value, ctypes.byref(ntiles))
    assert rc == 0
    return runs[:2 * nruns.value].reshape(-1, 2), dest[:ntotal], tiles[:3 * ntiles.value].reshape(-1, 3)


def _np_runs(ntotal, ids):
    u = np.unique(np.asarray(ids, np.int64))
    u = u[(u >= 0) & (u < ntotal)]
    if not len(u):
        return np.zeros((0, 2), np.int64)
    cut = np.nonzero(np.diff(u) != 1)[0] + 1
    return np.array([[g[0], g[-1] + 1] for g in np.split(u, cut)], np.int64)


def _np_dest(ntotal, ids):
    gone = np.zeros(ntotal, bool)
    u = np.asarray(ids, np.int64)
    gone[u[(u >= 0) & (u < ntotal)]] = True
    dest = np.full(ntotal, -1, np.int64)
    kept = np.delete(np.arange(ntotal), np.nonzero(gone)[0])
    dest[kept] = np.arange(len(kept))
    return dest


def _cases():
    rng = np.random.default_rng(7)
    n = 5000
    yield "first", n, [0]
    yield "last", n, [n - 1]
    yield "all", n, list(range(n))
    yield "alternate", n, list(range(0, n, 2))
    yield "alternate_odd", n, list(range(1, n, 2))
    yield "long_runs", n, list(range(10, 2000)) + list(range(2001, 4000)) + [4999]
    yield "front_range", n, list(range(0, 2500))
    yield "random_1pct", n, rng.choice(n, 50, replace=False).tolist()
    yield "messy", n, [-5, 3, 3, 9999, 2, 4, -1, 4998, 5000, 1 << 40, 2, 17, 16]
    yield "nothing_valid", n, [-1, n, n + 7]
    yield "empty", n, []
    yield "tiny", 1, [0]


@pytest.mark.parametrize("name,n,ids", list(_cases()), ids=[c[0] for c in _cases()])
def test_runs_and_destinations_match_numpy(name, n, ids):
    ids = np.asarray(ids, np.int64)
    perm = np.random.default_rng(1).permutation(len(ids))   # any order
    runs, dest, _ = _plan(n, ids[perm])
    assert np.array_equal(runs, _np_runs(n, ids)), name
    assert np.array_equal(dest, _np_dest(n, ids)), name


@pytest.mark.parametrize("row_bytes", [4, 12, 1536, 768, 3072, 20000, 65536])
@pytest.mark.parametrize("name,n,ids", [c for c in _cases() if c[0] not in ("empty", "nothing_valid")],
                         ids=[c[0] for c in _cases() if c[0] not in ("empty", "nothing_valid")])
def test_tiles_wait_exactly_for_the_lower_tiles_they_overwrite(row_bytes, name, n, ids):
    """For every tile of the compaction: the tiles whose source rows its destination meets, other than itself, are all
    lower, and they are exactly the tiles it waits for."""
    _, dest, tiles = _plan(n, ids, row_bytes)
    first = int(_np_runs(n, ids)[0, 0])
    T = max(1, TILE_BYTES // row_bytes)
    assert len(tiles) == -(-(n - first) // T)
    assert np.array_equal(tiles[:, 0], first + T * np.arange(len(tiles)))
    for t, (s0, w0, w1) in enumerate(tiles):
        d = dest[s0:min(s0 + T, n)]
        d = d[d >= 0]
        assert np.all(np.diff(d) == 1), "a tile's survivors must land on one contiguous range, in order"
        if not len(d):
            assert w0 == w1 == t
            continue
        assert d[0] >= first and d[-1] <= s0 + T - 1, "a row moved up, or below the first removed row"
        meets = set(range((d[0] - first) // T, (d[-1] - first) // T + 1)) - {t}
        assert all(u < t for u in meets)
        assert set(range(w0, w1)) == meets, (t, w0, w1, sorted(meets))


def test_remove_plan_rejects_bad_arguments():
    from rag_faiss_embedding_b200 import _capi

    lib = _capi.load()
    nr, nt = ctypes.c_int64(), ctypes.c_int64()
    assert lib.b2f_remove_plan(-1, 0, None, 4, None, ctypes.byref(nr), None, None, 0, ctypes.byref(nt)) == _capi.EINVAL
    assert lib.b2f_remove_plan(10, 3, None, 4, None, ctypes.byref(nr), None, None, 0, ctypes.byref(nt)) == _capi.EINVAL
    assert lib.b2f_remove_plan(10, 0, None, 0, None, ctypes.byref(nr), None, None, 0, ctypes.byref(nt)) == _capi.EINVAL
    assert lib.b2f_index_remove_ids(None, 0, None, None) == _capi.EINVAL
    assert lib.b2f_index_remove_range(None, 0, 1, None) == _capi.EINVAL


def test_selectors_and_coercion():
    import rag_faiss_embedding_b200 as m
    from rag_faiss_embedding_b200.index import _id_array

    r = m.IDSelectorRange(3, 9)
    assert (r.imin, r.imax) == (3, 9)
    b = m.IDSelectorBatch(np.array([5, 1, 5], np.int32))
    assert b.ids.dtype == np.int64 and b.ids.tolist() == [5, 1, 5]
    b2 = m.IDSelectorBatch(2, [7, 8, 9])
    assert b2.ids.tolist() == [7, 8]
    assert m.IDSelectorBatch(torch.tensor([4, 2])).ids.tolist() == [4, 2]
    with pytest.raises(AssertionError):
        m.IDSelectorBatch(4, [1, 2])
    with pytest.raises(TypeError):
        m.IDSelectorBatch()
    assert _id_array([]).dtype == np.int64 and _id_array([]).shape == (0,)
    assert _id_array(np.array([2.0, 3.0])).tolist() == [2, 3]
    assert _id_array(torch.arange(3, dtype=torch.int32)).tolist() == [0, 1, 2]
    for bad in (np.zeros((2, 2), np.int64), 5, torch.zeros(2, 1)):
        with pytest.raises(AssertionError):
            _id_array(bad)


def test_shim_exports_selectors_and_no_cpu_removal():
    import importlib
    import sys

    import rag_faiss_embedding_b200 as m

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rag-faiss-embedding_b200", "shim")
    sys.path.insert(0, shim)
    try:
        sys.modules.pop("faiss", None)
        faiss = importlib.import_module("faiss")
        assert faiss.IDSelectorRange is m.IDSelectorRange and faiss.IDSelectorBatch is m.IDSelectorBatch
        assert callable(faiss.IndexFlatL2.remove_ids)
        if m.device_count() > 0:
            return
        # no GPU: no index exists to remove from -- creation fails with B2F_ENOGPU, there is no CPU path
        with pytest.raises(m.B200FlatError) as e:
            faiss.IndexFlatL2(8).remove_ids(faiss.IDSelectorRange(0, 1))
        assert e.value.code == m._capi.ENOGPU
    finally:
        sys.path.remove(shim)
        sys.modules.pop("faiss", None)


def test_segment_map_remove():
    from rag_faiss_embedding_b200.sharded import SegmentMap

    seg = SegmentMap()
    seg.append(5, 3)      # local 0..2 -> 5..7
    seg.append(100, 4)    # local 3..6 -> 100..103
    seg.append(200, 2)    # local 7..8 -> 200..201
    local = seg.remove(np.array([1, 6, 100, 101, 102, 103, 150, 200], np.int64))
    assert local.tolist() == [1, 3, 4, 5, 6, 7]
    # labels 1 and 6 below / inside the first segment; the second segment is gone; 150 lies on another shard
    assert seg.nlocal == 3
    assert seg.local_starts == [0, 2] and seg.global_starts == [4, 200 - 8 + 1]
    seg2 = SegmentMap()
    seg2.append(0, 4)
    seg2.append(10, 4)
    seg2.remove(np.arange(4, 10))   # the gap between the segments closes: they merge
    assert seg2.local_starts == [0] and seg2.global_starts == [0] and seg2.nlocal == 8


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


D_, K_ = 16, 9
REMOVE1 = np.array([0, 3, 250, 251, 252, 299, 300, 301, 520, 578, -1, 10 ** 6, 3], np.int64)   # spans shards and segments
REMOVE2 = np.array([5, 400, 401, 402, 403, 404, 640], np.int64)


def _sharded_worker(rank, world, port, metric, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from rag_faiss_embedding_b200 import IDSelectorRange
        from rag_faiss_embedding_b200.sharded import ShardedIndexFlat

        xb1 = orc.np_synth_rows(21, 0, 301, D_)
        xb2 = orc.np_synth_rows(21, 301, 279, D_)
        xb3 = orc.np_synth_rows(21, 580, 90, D_)
        xq = orc.np_synth_rows(22, 0, 7, D_)

        ix = ShardedIndexFlat(D_, metric, local_index=RemovableOracleIndex(D_, metric), merge_fn=np_topk_merge_fn)
        ix.add(xb1)
        ix.add(xb2)
        n1 = ix.remove_ids(REMOVE1)
        D1, I1 = ix.search(xq, K_)
        ix.add(xb3)
        D2, I2 = ix.search(xq, K_)
        n2 = ix.remove_ids(REMOVE2)
        n3 = ix.remove_ids(IDSelectorRange(10, 20))
        D3, I3 = ix.search(xq, K_)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), D1=D1, I1=I1, D2=D2, I2=I2, D3=D3, I3=I3, n=[n1, n2, n3],
                 ntotal=ix.ntotal, nlocal=ix.local.ntotal)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("metric", [orc.METRIC_L2, orc.METRIC_INNER_PRODUCT])
def test_sharded_remove_equals_single(tmp_path, world, metric):
    mp.spawn(_sharded_worker, args=(world, _free_port(), metric, str(tmp_path)), nprocs=world, join=True)
    xb = orc.np_synth_rows(21, 0, 580, D_)
    xq = orc.np_synth_rows(22, 0, 7, D_)
    ref = RemovableOracleIndex(D_, metric)
    ref.add(xb)
    n1 = ref.remove_ids(REMOVE1)
    D1, I1 = orc.c_search(ref.x, xq, K_, metric)
    ref.add(orc.np_synth_rows(21, 580, 90, D_))
    D2, I2 = orc.c_search(ref.x, xq, K_, metric)
    n2 = ref.remove_ids(REMOVE2)
    n3 = ref.remove_ids(np.arange(10, 20))
    D3, I3 = orc.c_search(ref.x, xq, K_, metric)
    assert (n1, n2, n3) == (10, 7, 10)
    total = 0
    for r in range(world):
        z = np.load(os.path.join(tmp_path, f"r{r}.npz"))
        assert z["n"].tolist() == [n1, n2, n3] and int(z["ntotal"]) == ref.ntotal
        for a, b in (("D1", D1), ("I1", I1), ("D2", D2), ("I2", I2), ("D3", D3), ("I3", I3)):
            assert np.array_equal(z[a], b), (r, a)
        total += int(z["nlocal"])
    assert total == ref.ntotal


def test_store_remove_documents(monkeypatch, tmp_path):
    from rag_faiss_embedding_b200 import store as st

    def fake_write(index, path):
        orc.np_write_index(path, index.x, index.metric_type)

    monkeypatch.setattr(st, "IndexFlatL2", RemovableOracleIndex)
    monkeypatch.setattr(st, "write_index", fake_write)
    path = str(tmp_path / "faiss_index.bin")
    s = st.FAISSVectorStore(dimension=8, index_path=path)
    x = orc.np_synth_rows(5, 0, 7, 8)
    s.add_vectors(x, [70, 60, 50, 40, 30, 20, 10])
    assert s.remove_documents([60, 20, 999]) == 2
    assert s.doc_ids == [70, 50, 40, 30, 10] and s.index.ntotal == 5
    assert np.array_equal(s.index.x, x[[0, 2, 3, 4, 6]])
    for row, doc in ((1, 50), (2, 40), (4, 10)):
        _, ids = s.search(x[[0, 2, 3, 4, 6][row]], k=1)
        assert ids == [doc]
    assert s.remove_documents([]) == 0 and s.remove_documents([12345]) == 0
    s.save_index()
    xs, _ = orc.np_read_index(path)
    assert np.array_equal(xs, x[[0, 2, 3, 4, 6]]) and pickle.load(open(path + ".mapping", "rb")) == s.doc_ids
    assert s.remove_documents([70, 50, 40, 30, 10]) == 5
    assert s.doc_ids == [] and s.index.ntotal == 0
