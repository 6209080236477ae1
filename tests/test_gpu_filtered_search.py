"""GPU tier (-m gpu): filtered search (faiss ID selectors) on every search path.

A filtered search must return what the unfiltered search of an index holding only the allowed rows returns, with the
labels mapped back: on integer lattice data (tests/exact_checks.py) the float64 brute force over the allowed rows, bit for
bit and in tie order.  Each case asserts from the index's counters that the path it names served it.  The selectors'
membership is restated here in numpy (np_member), independently of the library's own host-side evaluation."""
import os
import socket

import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import IP, L2, check_structure, lattice
from tests.range_reference import np_range_search_f64
from tests.test_gpu_exact_ties import R, MU, _level_rows, _planted, _queries

pytestmark = pytest.mark.gpu

METRICS = (L2, IP)
STORAGES = (0, 1)
FMAX = np.finfo(np.float32).max


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


# ---- selectors and the reference ---------------------------------------------------------------------------------------
def np_member(m, sel, labels):
    """numpy restatement of faiss's is_member for the supported selectors (Not chains folded)."""
    neg = False
    while isinstance(sel, m.IDSelectorNot):
        sel, neg = sel.sel, not neg
    labels = np.asarray(labels, np.int64)
    if isinstance(sel, m.IDSelectorRange):
        mem = (labels >= sel.imin) & (labels < sel.imax)
    elif isinstance(sel, m.IDSelectorBatch):
        ids = sel.ids.cpu().numpy() if hasattr(sel.ids, "cpu") else np.asarray(sel.ids)
        mem = np.array([int(x) in set(ids.tolist()) for x in labels], bool) if len(labels) < 64 else np.isin(labels, ids)
    else:
        bm = sel.bitmap.cpu().numpy() if hasattr(sel.bitmap, "cpu") else np.asarray(sel.bitmap)
        bits = np.unpackbits(bm, bitorder="little").astype(bool)
        mem = np.zeros(labels.shape, bool)
        ok = (labels >= 0) & (labels < len(bits))
        mem[ok] = bits[labels[ok]]
    return mem != neg


def selectors(m, n, off, rng):
    """(name, selector) covering Range, Batch with duplicates and ids with no row, a Bitmap shorter than the index, and
    each under Not; labels are rows + off."""
    ids = rng.choice(n, n // 3, replace=False) + off
    batch = np.concatenate([ids, ids[:50], [-5, -1, off - 1, off + n, off + n + 1000]]).astype(np.int64)
    nbytes = (n * 3 // 4 + off) // 8   # ends before the last quarter of the rows
    bm = rng.integers(0, 256, nbytes, dtype=np.uint8)
    out = [("range", m.IDSelectorRange(off + n // 5, off + 3 * n // 5)),
           ("batch", m.IDSelectorBatch(batch)),
           ("bitmap", m.IDSelectorBitmap(nbytes, np.concatenate([bm, [255, 255]]).astype(np.uint8)))]
    return out + [("not_" + name, m.IDSelectorNot(s)) for name, s in out]


def ref_topk(rows, xq, k, metric, allowed, off=0):
    """float64 brute force over the allowed rows, labels mapped back (ties: lower label first, as the engine)."""
    idx = np.nonzero(allowed)[0]
    if len(idx) == 0:
        return (np.full((len(xq), k), FMAX if metric == L2 else -FMAX, np.float32), np.full((len(xq), k), -1, np.int64))
    D, I = orc.np_search_f64(rows[idx], xq, k, metric)
    return D, np.where(I >= 0, idx[np.maximum(I, 0)] + off, -1)


def assert_topk(D, I, rows, xq, k, metric, allowed, off=0):
    D, I = np.asarray(D), np.asarray(I)
    check_structure(D, I, metric, len(rows), off)
    Dr, Ir = ref_topk(rows, xq, k, metric, allowed, off)
    got = I[I >= 0] - off
    assert np.all(allowed[got]), "an excluded row was returned"
    if not (np.array_equal(I, Ir) and np.array_equal(D, Dr)):
        bad = np.nonzero((I != Ir) | (D != Dr))
        q, j = int(bad[0][0]), int(bad[1][0])
        raise AssertionError(f"{len(bad[0])} positions differ; first query {q} pos {j}: got ({D[q, j]!r}, {I[q, j]}), "
                             f"want ({Dr[q, j]!r}, {Ir[q, j]})")


def ref_range(rows, xq, radius, metric, allowed, off=0):
    lims, D, I = np_range_search_f64(rows, xq, radius, metric)
    keep = allowed[I]
    nl = np.zeros_like(lims)
    for q in range(len(xq)):
        nl[q + 1] = nl[q] + int(keep[lims[q]:lims[q + 1]].sum())
    return nl, D[keep], I[keep] + off


def assert_range(res, rows, xq, radius, metric, allowed, off=0):
    lims, D, I = (np.asarray(a.cpu() if hasattr(a, "cpu") else a) for a in res)
    rl, rD, rI = ref_range(rows, xq, radius, metric, allowed, off)
    assert np.array_equal(lims.astype(np.int64), rl), "hit counts differ"
    assert np.array_equal(I, rI), "hit ids differ"
    assert np.array_equal(D.astype(np.float64), rD), "hit distances differ"


def _fsearch(m, ix, xq, k, sel, algo, off=0):
    ix.set_search_params(algo=algo, id_offset=off)
    before = ix.stats()
    D, I = ix.search(xq, k, params=m.SearchParameters(sel=sel))
    after = ix.stats()
    st = {c: after[c] - before[c] for c in ("fallback_queries", "range_queries", "searches")}
    st.update(last_algo=after["last_algo"], last_kprime=after["last_kprime"])
    return D, I, st


def _index(m, lat, metric, storage):
    ix = m.IndexFlat(lat.d, metric, storage=storage)
    ix.add(lat.rows)
    return ix


# ---- 1. lattice data, bit for bit, every path --------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_scan_paths(m, metric, storage):
    """K1 at nq = 1 and nq = 8, every selector, id_offset 0 and 1000."""
    k = 10
    lat, xq, _ = _planted(6000, 128, 8, k, metric, seed=101 + metric)
    ix = _index(m, lat, metric, storage)
    rng = np.random.default_rng(5)
    for off in (0, 1000):
        for name, sel in selectors(m, len(lat.rows), off, rng):
            allowed = np_member(m, sel, np.arange(len(lat.rows)) + off)
            for nq in (1, 8):
                D, I, st = _fsearch(m, ix, xq[:nq], k, sel, m.ALGO_SCAN, off)
                assert st["last_algo"] == m.ALGO_SCAN and st["searches"] == 1, st
                assert_topk(D, I, lat.rows, xq[:nq], k, metric, allowed, off)


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("shape", [(30000, 385, 129, 10), (200, 128, 64, 10), (30000, 384, 833, 10)],
                         ids=["list", "heap", "pairs"])
def test_tensor_paths(m, metric, storage, shape):
    """K2 LIST, HEAP (a few-row index) and CTA pairs (nq >= 256), every selector, id_offset 0 and 7."""
    import ctypes

    n, d, nq, k = shape
    out = (ctypes.c_int32 * 12)()
    assert m._capi.load().b2f_plan_describe(nq, n, d, k, 0, out) == 0
    want = {"list": (1, 0), "heap": (0, 0), "pairs": (1, 1)}[{129: "list", 64: "heap", 833: "pairs"}[nq]]
    assert (out[3], out[4]) == want, list(out)
    lat, xq, _ = _planted(n, d, nq, k, metric, seed=111 + metric + nq)
    ix = _index(m, lat, metric, storage)
    rng = np.random.default_rng(nq)
    for off in (0, 7):
        for name, sel in selectors(m, n, off, rng):
            allowed = np_member(m, sel, np.arange(n) + off)
            D, I, st = _fsearch(m, ix, xq, k, sel, m.ALGO_TENSOR, off)
            assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] > 0, (name, st)
            assert_topk(D, I, lat.rows, xq, k, metric, allowed, off)


@pytest.mark.parametrize("metric", METRICS)
def test_heap_mode_after_list_overflows(m, metric):
    """The contiguous-ties data of test_gpu_exact_ties switches the index to per-thread heaps plus the range pass; filtered
    searches before and after the switch are exact."""
    k, nq = 10, 256
    lat = lattice(60000, 128, R, MU, seed=21 + metric)
    centres = _queries(lat, metric, 300)
    for c in centres:
        lat.plant(np.repeat(c[None], 80, 0), contiguous=True)
    pick = lat.rng.integers(0, 300, nq)
    xq = (centres[pick] + np.eye(128, dtype=np.float32)[lat.rng.integers(0, 128, nq)]) if metric == L2 else centres[pick].copy()
    xq = xq.astype(np.float32)
    lat.verify(xq)
    ix = _index(m, lat, metric, 0)
    sel = m.IDSelectorNot(m.IDSelectorRange(10000, 30000))
    allowed = np_member(m, sel, np.arange(len(lat.rows)))
    seen = []
    for it in range(4):
        D, I, st = _fsearch(m, ix, xq, k, sel, m.ALGO_TENSOR)
        assert_topk(D, I, lat.rows, xq, k, metric, allowed)
        seen.append(st)
    assert seen[3]["range_queries"] > 0, seen


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_range_pass_and_fewer_than_k_allowed(m, metric, storage):
    """Uncertifiable ties (the groups of test_gpu_exact_ties.test_tensor_uncertifiable_ties) put the index in range-pass
    mode; filtered searches then run the range pass over their failed queries, among them the 5000-copy group, whose
    lists overflow and hand the range pass tau = FLT_MAX (an +inf threshold).  Queries with fewer than k allowed rows
    (and none at all) are answered exactly too: their candidates are every allowed row."""
    k = 10
    lat = lattice(40000, 128, R, MU, seed=11 + metric)
    sizes = [40] * 4 + [100] * 4 + [400] * 4 + [1500] * 2 + [5000]
    xq = _queries(lat, metric, 48)
    for q, size in enumerate(sizes):
        ys = _level_rows(lat, metric, xq[q], 1, size if size <= 100 else 1)
        lat.plant(ys if size <= 100 else np.repeat(ys, size, 0))
    lat.verify(xq)
    ix = _index(m, lat, metric, storage)
    for it in range(2):   # unfiltered: the first batch's failures switch the range pass on
        ix.set_search_params(algo=m.ALGO_TENSOR)
        ix.search(xq, k)
    n = len(lat.rows)
    rng = np.random.default_rng(3)
    few = np.sort(rng.choice(n, 6, replace=False)).astype(np.int64)
    cases = [("few", m.IDSelectorBatch(few)), ("none", m.IDSelectorBatch(np.zeros(0, np.int64))),
             ("half", m.IDSelectorRange(0, n // 2)), ("empty_range", m.IDSelectorRange(50, 50)),
             ("all_but_few", m.IDSelectorNot(m.IDSelectorBatch(few)))]
    ranged = {}
    for name, sel in cases:
        allowed = np_member(m, sel, np.arange(n))
        ranged[name] = 0
        for it in range(2):
            D, I, st = _fsearch(m, ix, xq, k, sel, m.ALGO_TENSOR)
            assert_topk(D, I, lat.rows, xq, k, metric, allowed)
            ranged[name] += st["range_queries"]
            if not allowed.any():
                assert np.all(I == -1) and np.all(D == (FMAX if metric == L2 else -FMAX))
    print(f"metric {metric} storage {storage}: range-pass queries per selector {ranged}")
    assert ranged["all_but_few"] > 0, ranged


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_range_search_paths(m, metric, storage):
    """Range search on the tensor pass and with algo = SCAN, 1100 queries (across the 1024-query chunk boundary), every
    selector; radii FLT_MAX and 1e38 (thresholds that overflow to +inf) never return an excluded label."""
    lat, xq, _ = _planted(20000, 128, 1100, 10, metric, seed=131 + metric)
    ix = _index(m, lat, metric, storage)
    n = len(lat.rows)
    keys = orc.np_search_f64(lat.rows, xq[:64], 20, metric)[0]
    radius = float(np.median(keys[:, -1])) + (0.5 if metric == L2 else -0.5)
    rng = np.random.default_rng(9)
    for off in (0, 3):
        for name, sel in selectors(m, n, off, rng):
            allowed = np_member(m, sel, np.arange(n) + off)
            for algo in (m.ALGO_TENSOR, m.ALGO_SCAN):
                ix.set_search_params(algo=algo, id_offset=off)
                res = ix.range_search(xq, radius, params=m.SearchParameters(sel=sel))
                info = ix.last_range_info
                if algo == m.ALGO_SCAN:
                    assert info["scan_queries"] == len(xq), info
                else:
                    assert info["tensor_queries"] > 0, info
                assert_range(res, lat.rows, xq, radius, metric, allowed, off)
    ix.set_search_params(algo=m.ALGO_AUTO, id_offset=0)
    sel = m.IDSelectorRange(100, 300)
    allowed = np_member(m, sel, np.arange(n))
    for big in (float(FMAX), 1e38):
        r = big if metric == L2 else -big
        lims, D, I = ix.range_search(xq[:8], r, params=m.SearchParameters(sel=sel))
        assert np.all((I >= 100) & (I < 300)) and int(lims[-1]) == 8 * 200
        assert_range((lims, D, I), lat.rows, xq[:8], r, metric, allowed)


# ---- 2. edge cases ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_edges(m, metric):
    lat, xq, _ = _planted(5000, 64, 300, 10, metric, seed=141 + metric)
    n = len(lat.rows)
    ix = _index(m, lat, metric, 0)
    pad = FMAX if metric == L2 else -FMAX
    radius = 1e9 if metric == L2 else -1e9
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        ix.set_search_params(algo=algo)
        # nothing allowed
        for sel in (m.IDSelectorBatch(np.zeros(0, np.int64)), m.IDSelectorRange(10, 10), m.IDSelectorRange(20, 5),
                    m.IDSelectorNot(m.IDSelectorRange(-1, n + 1)), m.IDSelectorBitmap(np.zeros(0, np.uint8))):
            D, I = ix.search(xq, 10, params=m.SearchParameters(sel))
            assert np.all(I == -1) and np.all(D == pad)
            lims, Dr, Ir = ix.range_search(xq, radius, params=m.SearchParameters(sel))
            assert np.all(lims == 0) and len(Ir) == 0
        # everything allowed: bit-identical to the unfiltered call
        D0, I0 = ix.search(xq, 10)
        r0 = ix.range_search(xq, radius)
        for sel in (m.IDSelectorRange(-5, n + 5), m.IDSelectorNot(m.IDSelectorBatch(np.array([n + 3], np.int64))),
                    m.IDSelectorBitmap(np.full((n + 7) // 8, 255, np.uint8))):
            D, I = ix.search(xq, 10, params=m.SearchParameters(sel))
            assert np.array_equal(I, I0) and np.array_equal(D.view(np.uint32), D0.view(np.uint32))
            r = ix.range_search(xq, radius, params=m.SearchParameters(sel))
            assert all(np.array_equal(a, b) for a, b in zip(r, r0))
        # fewer than k allowed
        sel = m.IDSelectorBatch(np.array([3, 3, 4000, 17], np.int64))
        D, I = ix.search(xq, 10, params=m.SearchParameters(sel))
        assert_topk(D, I, lat.rows, xq, 10, metric, np_member(m, sel, np.arange(n)))
        assert np.all(I[:, 3:] == -1)
    # empty index
    e = m.IndexFlat(64, metric)
    D, I = e.search(xq[:3], 5, params=m.SearchParameters(m.IDSelectorRange(0, 10)))
    assert np.all(I == -1)
    lims, Dr, Ir = e.range_search(xq[:3], radius, params=m.SearchParameters(m.IDSelectorRange(0, 10)))
    assert np.all(lims == 0)


@pytest.mark.parametrize("metric", METRICS)
def test_excluded_non_finite_row(m, metric):
    """A row of infinities that the selector excludes: every path returns the exact result over the other rows."""
    lat, xq, _ = _planted(4000, 64, 200, 10, metric, seed=151 + metric)
    rows = lat.rows.copy()
    rows[1234] = np.inf
    ix = m.IndexFlat(64, metric)
    ix.add(rows)
    sel = m.IDSelectorNot(m.IDSelectorBatch(np.array([1234], np.int64)))
    allowed = np.ones(len(rows), bool)
    allowed[1234] = False
    for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
        ix.set_search_params(algo=algo)
        for nq in (1, 200):
            D, I = ix.search(xq[:nq], 10, params=m.SearchParameters(sel))
            assert_topk(D, I, lat.rows, xq[:nq], 10, metric, allowed)
        radius = 40.0 if metric == L2 else 10.0
        assert_range(ix.range_search(xq, radius, params=m.SearchParameters(sel)), lat.rows, xq, radius, metric, allowed)


# ---- 3. real-valued data ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_real_valued_equals_subset_index(m, metric):
    n, d, k = 30000, 384, 10
    xb = orc.c_synth_rows(77, 0, n, d)
    xq = orc.c_synth_rows(78, 0, 300, d)
    ix = m.IndexFlat(d, metric, storage=0)
    ix.add(xb)
    rng = np.random.default_rng(1)
    for name, sel in selectors(m, n, 0, rng):
        allowed = np_member(m, sel, np.arange(n))
        idx = np.nonzero(allowed)[0]
        sub = m.IndexFlat(d, metric, storage=0)
        sub.add(xb[idx])
        for nq in (1, 300):
            D, I = ix.search(xq[:nq], k, params=m.SearchParameters(sel))
            Ds, Is = sub.search(xq[:nq], k)
            Is = idx[Is]
            assert np.allclose(D, Ds, rtol=1e-5, atol=1e-6), name
            diff = I != Is
            if diff.any():   # only where the two distances tie
                assert np.allclose(D[diff], Ds[diff], rtol=1e-6), name
        radius = float(np.median(ix.search(xq[:32], 20)[0][:, -1]))
        r_all = ix.range_search(xq, radius)
        lims, Dr, Ir = ix.range_search(xq, radius, params=m.SearchParameters(sel))
        keep = allowed[r_all[2]]
        assert np.array_equal(Ir, r_all[2][keep]) and np.array_equal(Dr.view(np.uint32), r_all[1][keep].view(np.uint32))


# ---- 4. call forms and state ---------------------------------------------------------------------------------------------------
def test_call_forms_and_state(m):
    import torch

    metric, k = L2, 10
    lat, xq, _ = _planted(20000, 128, 64, k, metric, seed=161)
    ix = _index(m, lat, metric, 1)
    n = len(lat.rows)
    ids = np.random.default_rng(2).choice(n, 3000, replace=False).astype(np.int64)
    bm = np.packbits(np.arange(n) % 3 == 0, bitorder="little")
    D0, I0 = ix.search(xq, k)
    xd = torch.from_numpy(xq).cuda()
    for sel in (m.IDSelectorBatch(ids), m.IDSelectorBatch(torch.from_numpy(ids).cuda()), m.IDSelectorBitmap(bm),
                m.IDSelectorNot(m.IDSelectorBitmap(torch.from_numpy(bm).cuda()))):
        allowed = np_member(m, sel, np.arange(n))
        sp = m.SearchParameters()
        sp.sel = sel
        for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
            ix.set_search_params(algo=algo)
            Dh, Ih = ix.search(xq, k, params=sp)
            assert_topk(Dh, Ih, lat.rows, xq, k, metric, allowed)
            Dd, Id = ix.search(xd, k, params=sp)
            assert Dd.is_cuda and np.array_equal(Id.cpu().numpy(), Ih) and np.array_equal(Dd.cpu().numpy(), Dh)
            Dt = torch.empty((len(xq), k), dtype=torch.float32, device="cuda")
            It = torch.empty((len(xq), k), dtype=torch.int64, device="cuda")
            ix.search_tensors_into(xd, k, Dt, It, params=sp)
            assert np.array_equal(It.cpu().numpy(), Ih) and np.array_equal(Dt.cpu().numpy(), Dh)
            lims, Dr, Ir = ix.range_search(xd, 60.0, params=sp)
            assert lims.is_cuda
            assert_range((lims, Dr, Ir), lat.rows, xq, 60.0, metric, allowed)
    ix.set_search_params(algo=m.ALGO_AUTO)
    D1, I1 = ix.search(xq, k)
    assert np.array_equal(I1, I0) and np.array_equal(D1.view(np.uint32), D0.view(np.uint32))


# ---- 5. store and shards -------------------------------------------------------------------------------------------------------
def test_store_doc_ids(m, tmp_path):
    d = 32
    xb = orc.c_synth_rows(5, 0, 500, d)
    store = m.FAISSVectorStore(dimension=d, index_path=str(tmp_path / "none.bin"))
    store.add_vectors(xb, list(range(1000, 1500)))
    want = {1003, 1100, 1250, 1499}
    dist, ids = store.search(xb[0], k=10, doc_ids=sorted(want))
    assert set(ids) == want and len(ids) == 4
    D, many = store.search_many(xb[:5], k=3, doc_ids=[1001, 1002])
    assert all(set(r) <= {1001, 1002} and len(r) == 2 for r in many)
    assert store.search(xb[0], k=3)[1][0] == 1000


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _shard_cases(m, n):
    rng = np.random.default_rng(4)
    return selectors(m, n, 0, rng)


def _sharded_worker(rank, world, port, out_dir, backend):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = 0 if backend == "gloo" else rank
    torch.cuda.set_device(dev)
    if backend == "gloo":
        os.environ["B200FLAT_EXCHANGE"] = "nccl"   # two processes on one GPU: the all-gather form, not the peer exchange
        dist.init_process_group("gloo", rank=rank, world_size=world)
    else:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import rag_faiss_embedding_b200 as mm

        d, k = 64, 10
        xb1 = orc.c_synth_rows(21, 0, 3001, d)
        xb2 = orc.c_synth_rows(21, 3001, 999, d)
        xq = orc.c_synth_rows(22, 0, 40, d)
        out = {}
        for metric in (L2, IP):
            ix = mm.ShardedIndexFlat(d, metric, device=dev)
            ix.add(xb1)
            for stage in ("one", "two"):
                if stage == "two":
                    ix.add(xb2)   # each shard now holds two segments
                n = ix.ntotal
                radius = 9.0 if metric == L2 else 2.0
                for name, sel in _shard_cases(mm, n):
                    sp = mm.SearchParameters(sel=sel)
                    D, I = ix.search(xq, k, params=sp)
                    Dd, Id = ix.search(torch.from_numpy(xq).cuda(dev), k, params=sp)
                    lims, Dr, Ir = ix.range_search(xq, radius, params=sp)
                    out[f"{metric}_{stage}_{name}"] = (D, I, Dd.cpu().numpy(), Id.cpu().numpy(), lims.astype(np.int64), Dr, Ir)
        if rank == 0:
            np.savez(os.path.join(out_dir, "r0.npz"), **{f"{key}_{i}": v for key, t in out.items() for i, v in enumerate(t)})
    finally:
        dist.destroy_process_group()


def _check_sharded(m, out_dir):
    z = np.load(os.path.join(out_dir, "r0.npz"))
    d, k = 64, 10
    xb = orc.c_synth_rows(21, 0, 4000, d)
    xq = orc.c_synth_rows(22, 0, 40, d)
    for metric in (L2, IP):
        for stage, n in (("one", 3001), ("two", 4000)):
            one = m.IndexFlat(d, metric, storage=0)
            one.add(xb[:n])
            radius = 9.0 if metric == L2 else 2.0
            for name, sel in _shard_cases(m, n):
                key = f"{metric}_{stage}_{name}"
                sp = m.SearchParameters(sel=sel)
                D1, I1 = one.search(xq, k, params=sp)
                l1, Dr1, Ir1 = one.range_search(xq, radius, params=sp)
                # top-k: a shard may be served by another path than the whole index (the exact scan instead of the
                # tensor pass's re-rank), whose fp32 sums run in another order -- ids equal, distances to the last bits
                for di, ii in ((0, 1), (2, 3)):
                    assert np.array_equal(z[f"{key}_{ii}"], I1), key
                    assert np.allclose(z[f"{key}_{di}"], D1, rtol=1e-5, atol=1e-6), key
                # range search: every path computes a hit's distance with the same code, so the bits agree
                assert np.array_equal(z[f"{key}_4"], l1.astype(np.int64)) and np.array_equal(z[f"{key}_6"], Ir1), key
                assert np.array_equal(z[f"{key}_5"], Dr1), key


def test_sharded_two_processes_one_gpu_gloo(m, tmp_path):
    import torch.multiprocessing as mp

    mp.spawn(_sharded_worker, args=(2, _free_port(), str(tmp_path), "gloo"), nprocs=2, join=True)
    _check_sharded(m, str(tmp_path))


def test_sharded_nccl(m, tmp_path):
    import torch
    import torch.multiprocessing as mp

    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    mp.spawn(_sharded_worker, args=(world, _free_port(), str(tmp_path), "nccl"), nprocs=world, join=True)
    _check_sharded(m, str(tmp_path))
