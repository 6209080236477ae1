"""GPU tier (-m gpu): index.remove_ids.

A removal must leave exactly the index one add of the survivors would have built, as long as the centre is the same (the
removed rows are all at or above 65536, past the rows the centre comes from): the same stored bits, the same search and
range-search bits, the same search counters, the same file.  Where the removal takes rows the centre came from, the
survivors keep their bits and the centre stays.  A removed non-finite row gives the tensor pass back.  The compaction is
checked over many tiles per CTA, and against searches still in flight on another stream."""
import os
import socket

import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import IP, L2, check_exact, check_range_exact, lattice

pytestmark = pytest.mark.gpu

METRICS = (L2, IP)
STORAGES = (0, 1)   # fp32, bf16
COUNTERS = ("fallback_queries", "overflow_queries", "rescued_queries", "range_queries", "last_kprime")


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


def _survivors(n, ids):
    ids = np.asarray(ids, np.int64)
    return np.delete(np.arange(n), np.unique(ids[(ids >= 0) & (ids < n)]))


def _stored(x, storage, mu_rows=None):
    """What the index stores for rows x: x itself, or on bf16 storage fl32(mu + bf16(x - mu)), mu from mu_rows (the first
    rows of the first add)."""
    if storage == 0:
        return x
    mu = orc.np_centre((x if mu_rows is None else mu_rows)[:65536])
    return orc.np_bf16_rows(x, mu)


def _file(m, ix, path):
    m.write_index(ix, path)
    with open(path, "rb") as f:
        return f.read()


def _counters(ix):
    s = ix.stats()
    return {c: s[c] for c in COUNTERS}, s["last_list_entries"]


# ---- 1. equivalence to a rebuild -----------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_equals_rebuild(m, metric, storage, tmp_path):
    n, d = 70001, 96
    x = orc.c_synth_rows(31, 0, n, d)
    rng = np.random.default_rng(3)
    ids = np.concatenate([rng.choice(np.arange(65536, n - 1), 300, replace=False),   # singletons
                          np.arange(66000, 66517), np.arange(69000, 69100),            # runs
                          [n - 1, 66000, 66001, 67777, 67777],                          # the last row, duplicates
                          [-1, -70000, n, n + 5, 1 << 40]])                             # out of range
    rng.shuffle(ids)
    keep = _survivors(n, ids)
    a = m.IndexFlat(d, metric, storage=storage)
    a.add(x)
    launches = a.stats()["launches"]
    assert a.remove_ids(ids) == n - len(keep)
    assert a.ntotal == len(keep) and a.stats()["launches"] > launches
    b = m.IndexFlat(d, metric, storage=storage)
    b.add(x[keep])
    assert np.array_equal(a.reconstruct_n().view(np.uint32), b.reconstruct_n().view(np.uint32))
    assert np.array_equal(a.reconstruct_n().view(np.uint32), _stored(x[keep], storage, x).view(np.uint32))
    q = (x[rng.integers(0, n, 1024)] + np.float32(0.01) * rng.standard_normal((1024, d)).astype(np.float32)).astype(np.float32)
    runs = [(m.ALGO_SCAN, 1, 10), (m.ALGO_SCAN, 1, 100)] + [(m.ALGO_TENSOR, nq, k) for nq in (64, 1024) for k in (10, 100)]
    for algo, nq, k in runs:
        Da, Ia = a.set_search_params(algo=algo).search(q[:nq], k)
        Db, Ib = b.set_search_params(algo=algo).search(q[:nq], k)
        assert np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32)), (algo, nq, k)
        (ca, la), (cb, lb) = _counters(a), _counters(b)
        assert ca == cb, (algo, nq, k, ca, cb)
        if la != lb:   # the list-entry count follows the order CTAs tighten thresholds in: equal only if b repeats itself
            a.search(q[:nq], k)
            b.search(q[:nq], k)
            assert _counters(b)[1] != lb, f"last_list_entries {la} vs {lb} on a repeatable search"
    Dk, _ = b.set_search_params(algo=m.ALGO_SCAN).search(q[:64], 10)
    radius = float(np.median(Dk[:, -1]))
    for algo in (m.ALGO_AUTO, m.ALGO_SCAN):
        p = m.SearchParams()
        p.algo = algo
        la, Da, Ia = a.range_search(q[:64], radius, params=p)
        lb, Db, Ib = b.range_search(q[:64], radius, params=p)
        assert np.array_equal(la, lb) and np.array_equal(Ia, Ib) and np.array_equal(Da.view(np.uint32), Db.view(np.uint32))
    fa = _file(m, a, str(tmp_path / "a.bin"))
    if storage == 0:
        orc.c_write_index(str(tmp_path / "ref.bin"), x[keep], metric)
        assert fa == open(tmp_path / "ref.bin", "rb").read()
    else:
        assert fa == _file(m, b, str(tmp_path / "b.bin"))


# ---- 2. removals that take the centre's rows ------------------------------------------------------------------------
def _queries(lat, metric, nq):
    if metric == L2:
        return lat.near(nq)
    sigma = lat.rng.choice(np.array([-1.0, 1.0], np.float32), (nq, lat.d))
    return (lat.R * sigma).astype(np.float32)


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_front_removals_keep_bits_and_centre(m, metric, storage):
    n, d, k = 3001, 64, 10
    lat = lattice(n, d, 8, 3, seed=5)
    rows = lat.rows.copy()
    xq = _queries(lat, metric, 48)
    ix = m.IndexFlat(d, metric, storage=storage)
    ix.add(rows)
    model = rows
    radius = float(np.median(orc.np_search_f64(rows, xq, k, metric)[0][:, -1]))
    # row 0; the front 100 (3000 -> 2900 rows); all but the first and the last 99; all but one
    for sel in (np.array([0]), m.IDSelectorRange(0, 100), m.IDSelectorBatch(np.arange(1, 2801)), np.arange(0, 99)):
        if isinstance(sel, m.IDSelectorRange):
            gone = np.arange(sel.imin, sel.imax)
        else:
            gone = sel.ids if isinstance(sel, m.IDSelectorBatch) else sel
        assert ix.remove_ids(sel) == len(gone)
        model = np.delete(model, gone, axis=0)
        assert ix.ntotal == len(model)
        assert np.array_equal(ix.reconstruct_n().view(np.uint32), model.view(np.uint32))
        for algo in (m.ALGO_SCAN, m.ALGO_TENSOR):
            D, I = ix.set_search_params(algo=algo).search(xq, k)
            check_exact(D, I, model, xq, k, metric)
        for algo in (m.ALGO_AUTO, m.ALGO_SCAN):
            p = m.SearchParams()
            p.algo = algo
            lims, D, I = ix.range_search(xq, radius, params=p)
            check_range_exact(lims, D, I, model, xq, radius, metric)
    assert ix.ntotal == 1
    assert ix.remove_ids(m.IDSelectorRange(-5, 10)) == 1 and ix.ntotal == 0
    D, I = ix.search(xq, k)
    assert (I == -1).all()
    # not a reset: the next add is stored around the first add's centre
    y = orc.c_synth_rows(9, 0, 500, d) * np.float32(4) + np.float32(3)
    ix.add(y)
    assert np.array_equal(ix.reconstruct_n().view(np.uint32), _stored(y, storage, rows).view(np.uint32))
    D, I = ix.set_search_params(algo=m.ALGO_TENSOR).search(y[:64], k)
    D_ref, I_ref = orc.np_search_f64(_stored(y, storage, rows), y[:64], k, metric)
    assert orc.recall_and_errors(D, I, D_ref, I_ref, metric)["recall"] == 1.0


# ---- 3. a removed infinite row gives the tensor pass back ----------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_removing_inf_row_restores_tensor_pass(m, metric, storage):
    n, d, nq, k = 20000, 64, 64, 10
    x = orc.c_synth_rows(41, 0, n, d)
    bad = 12345
    x[bad, 7] = np.inf
    clean = np.delete(x, bad, axis=0)
    rng = np.random.default_rng(8)
    q = (clean[rng.integers(0, n - 1, nq)] + np.float32(0.01)).astype(np.float32)
    D_ref, _ = orc.np_search_f64(clean, q, 10, metric)
    radius = float(np.median(D_ref[:, -1]))
    ix = m.IndexFlat(d, metric, storage=storage)
    ix.add(x)
    ix.range_search(q, radius)
    assert ix.last_range_info["scan_queries"] == nq
    assert ix.remove_ids([bad]) == 1
    lims, D, I = ix.range_search(q, radius)
    assert ix.last_range_info["scan_queries"] == 0 and ix.last_range_info["tensor_queries"] == nq
    # (bf16 storage took its centre without the infinite row's block, so an index of the clean rows is another index: the
    # reference is this index's own exact scan, whose results have the same bits as the tensor pass's)
    p = m.SearchParams()
    p.algo = m.ALGO_SCAN
    lr, Dr, Ir = ix.range_search(q, radius, params=p)
    assert np.array_equal(lims, lr) and np.array_equal(I, Ir) and np.array_equal(D.view(np.uint32), Dr.view(np.uint32))
    f0 = ix.stats()["fallback_queries"]
    D, I = ix.set_search_params(algo=m.ALGO_TENSOR).search(q, k)
    assert ix.stats()["fallback_queries"] == f0 and ix.stats()["last_algo"] == m.ALGO_TENSOR
    Dr, Ir = ix.set_search_params(algo=m.ALGO_SCAN).search(q, k)
    r = orc.recall_and_errors(D, I, Dr, Ir, metric)
    assert r["recall"] == 1.0 and r["id_mismatch"] == 0, r


# ---- 4. many windows ----------------------------------------------------------------------------------------------
def _assert_rows(ix, expect, chunk=1 << 18):
    for r0 in range(0, len(expect), chunk):
        got = ix.reconstruct_n(r0, min(chunk, len(expect) - r0))
        assert np.array_equal(got.view(np.uint32), expect[r0:r0 + chunk].view(np.uint32)), f"rows from {r0}"


@pytest.mark.parametrize("metric,storage", [(L2, 0), (IP, 1)])
def test_many_windows(m, metric, storage):
    n, d = 2_000_000, 384
    x = orc.c_synth_rows(51, 0, n, d)
    stored = _stored(x, storage)
    ix = m.IndexFlat(d, metric, storage=storage)
    ix.add(x)
    assert ix.remove_ids(m.IDSelectorRange(0, 1)) == 1          # every row moves by one
    model = stored[1:]
    _assert_rows(ix, model)
    ids = np.random.default_rng(4).choice(len(model), len(model) // 100, replace=False)
    assert ix.remove_ids(ids) == len(ids)
    keep = _survivors(len(model), ids)
    model = model[keep]
    _assert_rows(ix, model)
    # the moved scan copy and biases: the tensor path (which reads them) agrees with the exact scan (which does not)
    q = model[np.random.default_rng(5).integers(0, len(model), 64)]
    D, I = ix.set_search_params(algo=m.ALGO_TENSOR).search(q, 10)
    assert ix.stats()["last_algo"] == m.ALGO_TENSOR
    D_ref, I_ref = ix.set_search_params(algo=m.ALGO_SCAN).search(q, 10)
    r = orc.recall_and_errors(D, I, D_ref, I_ref, metric)
    assert r["recall"] == 1.0 and r["max_rel_err"] <= 1e-5, r


# ---- 5. ordering without synchronising ------------------------------------------------------------------------------
def test_searches_in_flight_see_the_old_rows(m):
    import torch

    n, d, nq, k = 1_000_000, 128, 1024, 10
    x = orc.c_synth_rows(61, 0, n, d)
    ids = np.arange(0, n, 3)
    keep = _survivors(n, ids)
    ix = m.IndexFlat(d, L2)
    ix.add(x)
    old = m.IndexFlat(d, L2)
    old.add(x)
    new = m.IndexFlat(d, L2)
    new.add(x[keep])
    q = torch.from_numpy(x[np.random.default_rng(6).integers(0, n, nq)] + np.float32(0.01)).cuda()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        before = [ix.search(q, k) for _ in range(4)]        # enqueued, not waited for
    assert ix.remove_ids(ids) == len(ids)
    with torch.cuda.stream(side):
        after = ix.search(q, k)
    side.synchronize()
    Do, Io = old.search(q.cpu().numpy(), k)
    Dn, In = new.search(q.cpu().numpy(), k)
    for D, I in before:
        assert np.array_equal(I.cpu().numpy(), Io) and np.allclose(D.cpu().numpy(), Do, rtol=1e-6)
    assert np.array_equal(after[1].cpu().numpy(), In) and np.allclose(after[0].cpu().numpy(), Dn, rtol=1e-6)


def test_interleaved_add_remove(m):
    d, k = 40, 5
    ix = m.IndexFlat(d, L2)
    model = np.zeros((0, d), np.float32)
    rng = np.random.default_rng(9)
    for step in range(6):
        y = orc.c_synth_rows(70 + step, 0, 3000 + 700 * step, d)
        ix.add(y)
        model = np.concatenate([model, y])
        ids = rng.integers(-10, len(model) + 10, 900)
        assert ix.remove_ids(ids) == len(model) - len(_survivors(len(model), ids))
        model = model[_survivors(len(model), ids)]
        assert ix.ntotal == len(model)
        q = model[rng.integers(0, len(model), 16)]
        D, I = ix.set_search_params(algo=m.ALGO_SCAN).search(q, k)
        D_ref, I_ref = orc.c_search(model, q, k, L2)
        r = orc.recall_and_errors(D, I, D_ref, I_ref, L2)
        assert r["recall"] == 1.0 and r["id_mismatch"] == 0, (step, r)
    assert np.array_equal(ix.reconstruct_n(), model)


# ---- 6. through the faiss shim --------------------------------------------------------------------------------------
def test_faiss_shim(m):
    import importlib
    import sys

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rag-faiss-embedding_b200", "shim")
    sys.path.insert(0, shim)
    try:
        sys.modules.pop("faiss", None)
        faiss = importlib.import_module("faiss")
        d = 32
        x = orc.c_synth_rows(81, 0, 1000, d)
        ix = faiss.IndexFlatL2(d)
        ix.add(x)
        assert ix.remove_ids(faiss.IDSelectorRange(100, 200)) == 100
        assert ix.remove_ids(np.array([0, 5, 5, 899, 900, -1])) == 3
        assert ix.remove_ids(faiss.IDSelectorBatch(2, np.array([1, 2, 3]))) == 2
        model = np.delete(np.delete(np.delete(x, np.arange(100, 200), 0), [0, 5, 899], 0), [1, 2], 0)
        launches, before = ix.stats()["launches"], ix.reconstruct_n()
        assert ix.remove_ids([]) == 0 and ix.remove_ids(faiss.IDSelectorRange(5, 5)) == 0
        assert ix.remove_ids(np.array([len(model), -3])) == 0
        assert ix.stats()["launches"] == launches and ix.ntotal == len(model)
        assert np.array_equal(ix.reconstruct_n(), before) and np.array_equal(before, model)
        with pytest.raises(AssertionError):
            ix.remove_ids(np.zeros((2, 2), np.int64))
    finally:
        sys.path.remove(shim)
        sys.modules.pop("faiss", None)


# ---- 7. sharded, on GPUs --------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import rag_faiss_embedding_b200 as b2f

        d, k = 64, 10
        x = orc.c_synth_rows(91, 0, 50000, d)
        ix = b2f.ShardedIndexFlat(d, L2, device=rank)
        ix.add(x[:30000])
        ix.add(x[30000:])
        ix.remove_ids(np.arange(1000, 2000))
        ix.remove_ids(np.array([0, 29000, 30000, 49999]))
        xq = torch.from_numpy(x[::997].copy()).cuda()
        D, I = ix.search(xq, k)
        torch.cuda.synchronize()
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), D=D.cpu().numpy(), I=I.cpu().numpy(), ntotal=ix.ntotal)
    finally:
        dist.destroy_process_group()


def test_sharded_remove(m, tmp_path):
    import torch
    import torch.multiprocessing as mp

    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    mp.spawn(_sharded_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    x = orc.c_synth_rows(91, 0, 50000, 64)
    keep = _survivors(50000, np.concatenate([np.arange(1000, 2000), [0, 29000, 30000, 49999]]))
    single = m.IndexFlat(64, L2)
    single.add(x[keep])
    D_ref, I_ref = single.search(x[::997].copy(), 10)
    for r in range(world):
        z = np.load(os.path.join(tmp_path, f"r{r}.npz"))
        assert int(z["ntotal"]) == len(keep)
        assert np.array_equal(z["I"], I_ref) and np.allclose(z["D"], D_ref, rtol=1e-6)
