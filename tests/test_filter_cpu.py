"""CPU tier of filtered search: the selector classes and their coercion to the C struct, SearchParameters, the faiss
shim's names, the C ABI's argument checks, ENOGPU without a GPU, the sharded index's global-to-local selector mapping,
and sharded filtered top-k and range search on gloo (world sizes 2 and 3) over oracle-backed shards, against an oracle
search over the allowed rows of the concatenated database."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as orc
import rag_faiss_embedding_b200 as b2f
from rag_faiss_embedding_b200 import _capi as C
from tests.helpers import OracleIndex, np_topk_merge_fn
from tests.range_merge_reference import np_range_merge_fn
from tests.range_reference import np_range_search_f64


def np_member(sel, labels):
    """numpy restatement of faiss's is_member (Not chains folded)."""
    neg = False
    while isinstance(sel, b2f.IDSelectorNot):
        sel, neg = sel.sel, not neg
    labels = np.asarray(labels, np.int64)
    if isinstance(sel, b2f.IDSelectorRange):
        mem = (labels >= sel.imin) & (labels < sel.imax)
    elif isinstance(sel, b2f.IDSelectorBatch):
        ids = set(np.asarray(sel.ids).tolist())
        mem = np.array([int(x) in ids for x in labels], bool)
    else:
        bits = np.unpackbits(np.asarray(sel.bitmap), bitorder="little").astype(bool)
        mem = np.array([0 <= x < len(bits) and bits[x] for x in labels], bool)
    return mem != neg


def _selectors(n):
    rng = np.random.default_rng(n)
    ids = np.concatenate([rng.choice(n, n // 4, replace=False), [0, 0, -3, n, n + 9]]).astype(np.int64)
    bm = rng.integers(0, 256, (n * 2 // 3) // 8, dtype=np.uint8)
    out = [b2f.IDSelectorRange(n // 5, n // 2), b2f.IDSelectorBatch(ids), b2f.IDSelectorBitmap(bm),
           b2f.IDSelectorRange(7, 7), b2f.IDSelectorBatch(np.zeros(0, np.int64))]
    return out + [b2f.IDSelectorNot(s) for s in out[:3]] + [b2f.IDSelectorNot(b2f.IDSelectorNot(out[1]))]


# ---- selectors -----------------------------------------------------------------------------------------------------------
def test_selector_classes_and_coercion():
    from rag_faiss_embedding_b200.index import _c_selector, selector_contains

    bm = np.array([0b00000101, 0xff, 0x80], np.uint8)
    s = b2f.IDSelectorBitmap(2, bm)          # n counts BYTES: 16 labels
    assert s.bitmap.shape == (2,)
    assert list(np.nonzero(selector_contains(s, np.arange(-2, 30)))[0] - 2) == [0, 2] + list(range(8, 16))
    c, keep = _c_selector(s)
    assert (c.kind, c.negate, c.n) == (C.SEL_BITMAP, 0, 2) and c.data == keep.ctypes.data
    n3 = b2f.IDSelectorNot(b2f.IDSelectorNot(b2f.IDSelectorNot(b2f.IDSelectorRange(3, 9))))
    c, _ = _c_selector(n3)
    assert (c.kind, c.negate, c.imin, c.imax) == (C.SEL_RANGE, 1, 3, 9)
    c, keep = _c_selector(b2f.IDSelectorBatch([5, 5, 2]))
    assert (c.kind, c.n) == (C.SEL_BATCH, 3) and keep.dtype == np.int64
    c, _ = _c_selector(b2f.IDSelectorBatch(np.zeros(0)))
    assert c.n == 0 and not c.data
    assert b2f.IDSelectorBatch(2, [4, 5, 6]).ids.tolist() == [4, 5]
    for n in (1, 100, 1000):
        for sel in _selectors(n):
            labels = np.arange(-5, n + 20)
            assert np.array_equal(selector_contains(sel, labels), np_member(sel, labels))
    for cls in (b2f.IDSelectorAnd, b2f.IDSelectorOr, b2f.IDSelectorXor, b2f.IDSelectorArray):
        with pytest.raises(TypeError, match="not supported"):
            cls(b2f.IDSelectorRange(0, 1), b2f.IDSelectorRange(0, 2))
    with pytest.raises(TypeError, match="unsupported selector"):
        b2f.IDSelectorNot(object())
    with pytest.raises(TypeError):
        _c_selector([1, 2, 3])
    with pytest.raises(AssertionError):
        b2f.IDSelectorBitmap(5, np.zeros(2, np.uint8))


def test_search_parameters_and_shim():
    p = b2f.SearchParameters()
    assert p.sel is None
    p.sel = b2f.IDSelectorRange(0, 4)
    assert b2f.SearchParameters(sel=p.sel).sel is p.sel
    import importlib
    import sys

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rag-faiss-embedding_b200", "shim")
    sys.path.insert(0, shim)
    try:
        sys.modules.pop("faiss", None)
        faiss = importlib.import_module("faiss")
    finally:
        sys.path.remove(shim)
        sys.modules.pop("faiss", None)
    for name in ("SearchParameters", "IDSelectorRange", "IDSelectorBatch", "IDSelectorBitmap", "IDSelectorNot",
                 "IDSelectorAnd", "IDSelectorOr"):
        assert getattr(faiss, name) is getattr(b2f, name), name


def test_capi_argument_checks_and_no_gpu():
    lib = C.load()
    q = np.zeros((1, 4), np.float32)
    D = np.zeros((1, 1), np.float32)
    I = np.zeros((1, 1), np.int64)
    h = ctypes.c_void_p()
    for kind, n, data in ((0, 0, None), (4, 0, None), (C.SEL_BATCH, -1, None), (C.SEL_BATCH, 3, None),
                          (C.SEL_BITMAP, 2, None)):
        s = C.Selector(kind=kind, n=n, data=data)
        assert lib.b2f_index_search_filtered(None, 1, q.ctypes.data, 1, D.ctypes.data, I.ctypes.data, C.MEM_HOST, None,
                                             None, ctypes.byref(s)) == C.EINVAL
        assert "selector" in C.last_error()
        assert lib.b2f_index_range_search_filtered(None, 1, q.ctypes.data, 1.0, C.MEM_HOST, None, None, ctypes.byref(s),
                                                   ctypes.byref(h)) == C.EINVAL
        assert "selector" in C.last_error()
    ok = C.Selector(kind=C.SEL_RANGE, imin=0, imax=3)
    assert lib.b2f_index_search_filtered(None, 1, q.ctypes.data, 1, D.ctypes.data, I.ctypes.data, C.MEM_HOST, None, None,
                                         ctypes.byref(ok)) == C.EINVAL
    assert "index is NULL" in C.last_error()
    if b2f.device_count() == 0:
        with pytest.raises(b2f.B200FlatError) as e:
            b2f.IndexFlat(4)
        assert e.value.code == C.ENOGPU


# ---- sharded: the global-to-local mapping ------------------------------------------------------------------------------------
class FilterOracleIndex(OracleIndex):
    """OracleIndex with range search and filtered search (SearchParameters: membership of label = row + offset)."""

    def _allowed(self, params):
        if params is None or params.sel is None:
            return np.ones(self.ntotal, bool)
        return np_member(params.sel, np.arange(self.ntotal) + self._offset)

    def search(self, q, k, params=None):
        allowed = self._allowed(params)
        idx = np.nonzero(allowed)[0]
        q = np.ascontiguousarray(q, np.float32)
        if len(idx) == 0:
            fill = np.finfo(np.float32).max * (1 if self.metric_type == orc.METRIC_L2 else -1)
            return np.full((len(q), k), fill, np.float32), np.full((len(q), k), -1, np.int64)
        D, I = orc.c_search(self.x[idx], q, k, self.metric_type)
        return D, np.where(I >= 0, idx[np.maximum(I, 0)] + self._offset, -1)

    def range_search(self, x, radius, params=None):
        lims, D, I = np_range_search_f64(self.x, np.ascontiguousarray(x, np.float32), radius, self.metric_type)
        keep = self._allowed(params)[I]
        nl = np.concatenate([[0], np.cumsum([keep[lims[q]:lims[q + 1]].sum() for q in range(len(x))])]).astype(np.int64)
        self.last_range_info = {"hits": int(nl[-1])}
        return nl.astype(np.uint64), D[keep].astype(np.float32), I[keep] + self._offset


def test_sharded_local_params_mapping():
    from rag_faiss_embedding_b200.sharded import ShardedIndexFlat

    ix = ShardedIndexFlat(8, local_index=FilterOracleIndex(8))
    ix.add_local(np.zeros((30, 8), np.float32), 100)
    sel = b2f.IDSelectorBatch([101, 105, 129, 130, 3])
    off = ix._local_offset()
    assert off == 100 and ix._local_params(b2f.SearchParameters(sel), off).sel is sel   # passed through
    assert ix._local_params(None, off) is None and ix._local_params(b2f.SearchParameters(), off) is None
    ix.add_local(np.zeros((20, 8), np.float32), 7)     # a second segment, below the first
    ix.add_local(np.zeros((5, 8), np.float32), 1000)
    off = ix._local_offset()
    assert off is None
    labels = ix.segments.to_global_numpy(np.arange(55))
    for s in _selectors(1100) + [sel]:
        lp = ix._local_params(b2f.SearchParameters(s), off)
        assert isinstance(lp.sel, b2f.IDSelectorBitmap)
        assert np.array_equal(np_member(lp.sel, np.arange(55)), np_member(s, labels))


# ---- sharded on gloo ---------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


D_DIM, K, NQ = 16, 7, 9


def _data():
    xb = np.rint(orc.np_synth_rows(31, 0, 700, D_DIM) * 8).astype(np.float32)
    xq = np.rint(orc.np_synth_rows(32, 0, NQ, D_DIM) * 8).astype(np.float32)
    return xb, xq


def _radius(metric):
    return 60.0 if metric == orc.METRIC_L2 else 3.0


def _worker(rank, world, port, metric, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from rag_faiss_embedding_b200.sharded import ShardedIndexFlat

        xb, xq = _data()
        ix = ShardedIndexFlat(D_DIM, metric, local_index=FilterOracleIndex(D_DIM, metric), merge_fn=np_topk_merge_fn,
                              range_merge_fn=np_range_merge_fn)
        res = {}
        ix.add(xb[:500])
        for stage in ("one", "two"):
            if stage == "two":
                ix.add(xb[500:])   # two segments per shard: the host-side bitmap mapping
            for i, sel in enumerate(_selectors(ix.ntotal)):
                sp = b2f.SearchParameters(sel)
                D, I = ix.search(xq, K, params=sp)
                lims, Dr, Ir = ix.range_search(xq, _radius(metric), params=sp)
                res.update({f"{stage}{i}_D": D, f"{stage}{i}_I": I, f"{stage}{i}_l": lims.astype(np.int64),
                            f"{stage}{i}_Dr": Dr, f"{stage}{i}_Ir": Ir})
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("metric", [orc.METRIC_L2, orc.METRIC_INNER_PRODUCT])
def test_sharded_filtered_gloo(tmp_path, world, metric):
    mp.spawn(_worker, args=(world, _free_port(), metric, str(tmp_path)), nprocs=world, join=True)
    xb, xq = _data()
    for stage, n in (("one", 500), ("two", 700)):
        ref = FilterOracleIndex(D_DIM, metric)
        ref.add(xb[:n])
        for i, sel in enumerate(_selectors(n)):
            sp = b2f.SearchParameters(sel)
            D, I = ref.search(xq, K, params=sp)
            lims, Dr, Ir = ref.range_search(xq, _radius(metric), params=sp)
            assert np.all(np_member(sel, I[I >= 0])) and np.all(np_member(sel, Ir))
            for r in range(world):
                z = np.load(os.path.join(tmp_path, f"r{r}.npz"))
                key = f"{stage}{i}"
                assert np.array_equal(z[f"{key}_I"], I), (r, key)
                assert np.array_equal(z[f"{key}_D"], D), (r, key)
                assert np.array_equal(z[f"{key}_l"], lims.astype(np.int64)), (r, key)
                assert np.array_equal(z[f"{key}_Ir"], Ir) and np.array_equal(z[f"{key}_Dr"], Dr), (r, key)
