"""GPU tier (-m gpu): IndexFlat.range_search against float64 brute force on the authoritative rows, path independence
(tensor-pass lists vs the exact range scan, bit for bit), agreement with top-k search, list overflow, edge inputs, the
numpy / torch / faiss-shim interfaces, and that a range search leaves top-k search state alone."""
import os
import sys

import numpy as np
import pytest

import oracle as orc
from tests.range_reference import np_range_search_f64

pytestmark = pytest.mark.gpu

REL, ABS = 1e-5, 1e-4
L2, IP = orc.METRIC_L2, orc.METRIC_INNER_PRODUCT


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    if mod.device_count() == 0:
        pytest.skip("no B200")
    return mod


def _params(m, algo, id_offset=0):
    p = m.SearchParams()
    p.algo = algo
    p.id_offset = id_offset
    return p


def _rows(n, d, seed, nc=64):
    """Clustered rows (embedding-like), so that radii select anything from 1 to 1000s of neighbours."""
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((nc, d)).astype(np.float32)
    return (c[rng.integers(0, nc, n)] + 0.5 * rng.standard_normal((n, d))).astype(np.float32)


def _queries(xb, nq, seed):
    rng = np.random.default_rng(seed)
    return (xb[rng.integers(0, len(xb), nq)] + 0.3 * rng.standard_normal((nq, xb.shape[1]))).astype(np.float32)


_cache = {}


def _index(m, metric, storage, d, n=4000, seed=11):
    key = (metric, storage, d, n, seed)
    if key not in _cache:
        xb = _rows(n, d, seed)
        ix = m.IndexFlat(d, metric, storage=storage)
        ix.add(xb)
        _cache[key] = (ix, ix.reconstruct_n().astype(np.float64), xb)
    return _cache[key]


def _keys64(rows, q, metric):
    return ((rows - q.astype(np.float64)) ** 2).sum(1) if metric == L2 else -(rows @ q.astype(np.float64))


def _radius(rows, q, metric, m_):
    """Midway between the m-th and (m+1)-th float64 key of query q, in a gap wider than 1e-4 relative."""
    s = np.sort(_keys64(rows, q, metric))
    while m_ < len(s) - 1 and s[m_] - s[m_ - 1] <= 1e-4 * max(abs(s[m_]), 1e-30):
        m_ += 1
    r = 0.5 * (s[m_ - 1] + s[m_])
    return float(r if metric == L2 else -r)


def _check(rows, xq, radius, metric, lims, D, I, id_offset=0, exact_q=None):
    """lims / id sets equal the float64 reference wherever a row is not within 1e-5 relative of the radius (a query whose
    radius was chosen in a gap -- exact_q -- must match exactly); distances to 1e-5 relative; the strict inequality on
    every returned distance; ids ascending."""
    lims = np.asarray(lims, np.int64)
    D = np.asarray(D)
    I = np.asarray(I) - id_offset
    assert lims[0] == 0 and np.all(np.diff(lims) >= 0) and lims[-1] == len(D) == len(I)
    rl, rD, rI = np_range_search_f64(rows, xq, radius, metric)
    if metric == L2:
        assert np.all(D < np.float32(radius))
    else:
        assert np.all(D > np.float32(radius))
    for q in range(len(xq)):
        gi, gd = I[lims[q]:lims[q + 1]], D[lims[q]:lims[q + 1]]
        wi, wd = rI[rl[q]:rl[q + 1]], rD[rl[q]:rl[q + 1]]
        assert np.all(np.diff(gi) > 0)
        diff = set(gi.tolist()) ^ set(wi.tolist())
        if diff:
            assert q != exact_q, (q, sorted(diff)[:10])
            k = _keys64(rows[sorted(diff)], xq[q], metric)
            dist = k if metric == L2 else -k
            assert np.all(np.abs(dist - radius) <= REL * abs(radius) + ABS), (q, dist, radius)
        common, a, b = np.intersect1d(gi, wi, return_indices=True)
        with np.errstate(invalid="ignore"):   # (+-inf distances to rows with infinite entries compare equal)
            assert np.all((gd[a] == wd[b]) | (np.abs(gd[a] - wd[b]) <= REL * np.abs(wd[b]) + ABS))


def _rs(ix, xq, radius, params):
    lims, D, I = ix.range_search(xq, radius, params=params)
    return lims.astype(np.int64), D, I, dict(ix.last_range_info)


# ---- 1. exact sets -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [L2, IP])
@pytest.mark.parametrize("storage", [0, 1])
def test_exact_sets_algos_and_radii(m, metric, storage):
    ix, rows, xb = _index(m, metric, storage, 384)
    xq = _queries(xb, 37, 3)
    for m_ in (1, 10, 100, 1000):
        radius = _radius(rows, xq[0], metric, m_)
        res = {}
        for algo in (m.ALGO_AUTO, m.ALGO_TENSOR, m.ALGO_SCAN):
            lims, D, I, info = _rs(ix, xq, radius, _params(m, algo))
            _check(rows, xq, radius, metric, lims, D, I, exact_q=0)
            assert info["hits"] == lims[-1] and info["tensor_queries"] + info["scan_queries"] == len(xq)
            if algo == m.ALGO_SCAN:
                assert info["scan_queries"] == len(xq)
            res[algo] = (lims, D, I)
        # 3. path independence: the lists and the exact range scan give the same bits
        for algo in (m.ALGO_AUTO, m.ALGO_TENSOR):
            for a, b in zip(res[algo], res[m.ALGO_SCAN]):
                assert np.array_equal(a, b)


@pytest.mark.parametrize("nq", [1, 37, 1024, 2500])
def test_exact_sets_batch_sizes(m, nq):
    ix, rows, xb = _index(m, L2, 0, 384)
    xq = _queries(xb, nq, 4)
    radius = _radius(rows, xq[0], L2, 10)
    lims, D, I, info = _rs(ix, xq, radius, _params(m, m.ALGO_TENSOR))
    _check(rows, xq, radius, L2, lims, D, I, exact_q=0)
    assert info["tensor_queries"] == nq and info["host_syncs"] <= (nq + 1023) // 1024 + 2
    # 3. one query at a time gives the same bits
    if nq in (37, 1024):
        sub = range(0, nq, max(1, nq // 16))
        for q in sub:
            l1, d1, i1, _ = _rs(ix, xq[q:q + 1], radius, _params(m, m.ALGO_TENSOR))
            assert np.array_equal(d1, D[lims[q]:lims[q + 1]]) and np.array_equal(i1, I[lims[q]:lims[q + 1]])
        again = _rs(ix, xq, radius, _params(m, m.ALGO_TENSOR))
        for a, b in zip(again[:3], (lims, D, I)):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("d", [1, 100, 384, 385, 1536, 4096])
@pytest.mark.parametrize("metric", [L2, IP])
def test_exact_sets_widths(m, d, metric):
    for storage in (0, 1):
        ix, rows, xb = _index(m, metric, storage, d, n=3000)
        xq = _queries(xb, 9, 5)
        radius = _radius(rows, xq[0], metric, 100)
        lims, D, I, _ = _rs(ix, xq, radius, _params(m, m.ALGO_TENSOR))
        _check(rows, xq, radius, metric, lims, D, I, exact_q=0)
        ls, Ds, Is, _ = _rs(ix, xq, radius, _params(m, m.ALGO_SCAN))
        assert np.array_equal(lims, ls) and np.array_equal(D, Ds) and np.array_equal(I, Is)


# ---- 2. invariants for arbitrary radii -----------------------------------------------------------------------------
def test_invariants_arbitrary_radii(m):
    rng = np.random.default_rng(8)
    for metric in (L2, IP):
        ix, rows, xb = _index(m, metric, 0, 384)
        xq = _queries(xb, 64, 6)
        k = _keys64(rows, xq[0], metric)
        for r in rng.uniform(np.percentile(k, 0.1), np.percentile(k, 20), 4):
            radius = float(r if metric == L2 else -r)
            lims, D, I, _ = _rs(ix, xq, radius, _params(m, m.ALGO_AUTO))
            _check(rows, xq, radius, metric, lims, D, I)


# ---- 4. agreement with top-k ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [L2, IP])
def test_agrees_with_topk(m, metric):
    ix, rows, xb = _index(m, metric, 0, 384)
    xq = _queries(xb, 24, 7)
    p = _params(m, m.ALGO_TENSOR)
    for k in (1, 10, 50):
        Dk, Ik = ix.search(xq, k + 1, params=p)
        for q in range(len(xq)):
            if Dk[q, k - 1] == Dk[q, k]:
                continue
            radius = float(Dk[q, k])   # strict: exactly the k best are inside
            lims, D, I, _ = _rs(ix, xq[q:q + 1], radius, p)
            order = np.argsort(Ik[q, :k])
            assert np.array_equal(I, Ik[q, :k][order]) and np.array_equal(D, Dk[q, :k][order])


# ---- 5. overflow and the exact range scan ------------------------------------------------------------------------------
def test_everything_inside(m):
    ix, rows, xb = _index(m, L2, 0, 128, n=20000)
    xq = _queries(xb, 8, 9)
    lims, D, I, info = _rs(ix, xq, 1e30, _params(m, m.ALGO_TENSOR))
    assert lims.tolist() == [20000 * i for i in range(9)] and info["scan_queries"] == 8
    assert np.array_equal(I.reshape(8, 20000), np.tile(np.arange(20000), (8, 1)))
    ref = ((rows[None, :, :] - xq[:, None, :].astype(np.float64)) ** 2).sum(-1)
    assert np.allclose(D.reshape(8, 20000), ref, rtol=REL, atol=ABS)


def _dense(layout, d=128, nc=60, dup=400, nq=64):
    rng = np.random.default_rng(9)
    centres = rng.standard_normal((nc, d)).astype(np.float32)
    xb = (np.repeat(centres, dup, axis=0) + rng.standard_normal((nc * dup, d)).astype(np.float32) * 1e-3).astype(np.float32)
    if layout == "shuffled":
        xb = xb[rng.permutation(len(xb))]
    xq = (centres[rng.integers(0, nc, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 1e-3).astype(np.float32)
    return xb, xq


@pytest.mark.parametrize("layout", ["shuffled", "contiguous"])
def test_dense_near_duplicates(m, layout):
    xb, xq = _dense(layout)
    ix = m.IndexFlatL2(xb.shape[1], storage=0)
    ix.add(xb)
    rows = ix.reconstruct_n().astype(np.float64)
    lims, D, I, info = _rs(ix, xq, 1.0, _params(m, m.ALGO_TENSOR))   # one cluster: intra ~2.6e-4, inter ~256
    _check(rows, xq, 1.0, L2, lims, D, I)
    assert np.all(np.diff(lims) == 400)
    print(f"\n[range dense {layout}] tensor-path queries {info['tensor_queries']}, exact range scan {info['scan_queries']}")
    if layout == "shuffled":
        assert info["scan_queries"] == 0


# ---- 6. edges --------------------------------------------------------------------------------------------------------
def test_edges(m, tmp_path):
    ix, rows, xb = _index(m, L2, 0, 64, n=3000)
    xq = _queries(xb, 5, 10)
    radius = _radius(rows, xq[0], L2, 20)
    base = _rs(ix, xq, radius, _params(m, m.ALGO_TENSOR))
    xn = xq.copy()
    xn[2, 7] = np.nan
    lims, D, I, _ = _rs(ix, xn, radius, _params(m, m.ALGO_TENSOR))
    assert lims[3] == lims[2]
    for q in (0, 1, 3, 4):
        assert np.array_equal(I[lims[q]:lims[q + 1]], base[2][base[0][q]:base[0][q + 1]])
        assert np.array_equal(D[lims[q]:lims[q + 1]], base[1][base[0][q]:base[0][q + 1]])
    # id_offset
    lo, Do, Io, _ = _rs(ix, xq, radius, _params(m, m.ALGO_TENSOR, id_offset=1000))
    assert np.array_equal(lo, base[0]) and np.array_equal(Do, base[1]) and np.array_equal(Io, base[2] + 1000)
    # empty index, nq = 0, L2 radius <= 0, NaN radius
    empty = m.IndexFlatL2(64)
    assert _rs(empty, xq, 10.0, None)[0].tolist() == [0] * 6
    assert ix.range_search(xq[:0], radius)[0].tolist() == [0]
    assert _rs(ix, xq, 0.0, None)[0].tolist() == [0] * 6
    with pytest.raises(m.B200FlatError):
        ix.range_search(xq, float("nan"))
    # a row with +-inf entries
    for metric in (L2, IP):
        xi = xb.copy()
        xi[17, 3], xi[40, 5] = np.inf, -np.inf
        inf_ix = m.IndexFlat(64, metric, storage=0)
        inf_ix.add(xi)
        r_inf = inf_ix.reconstruct_n().astype(np.float64)
        rad = _radius(r_inf[np.isfinite(r_inf).all(1)], xq[0], metric, 20)
        for algo in (m.ALGO_TENSOR, m.ALGO_SCAN):
            lims, D, I, _ = _rs(inf_ix, xq, rad, _params(m, algo))
            _check(r_inf, xq, rad, metric, lims, D, I)
    # a bf16 index read back from a file
    bix, brows, _ = _index(m, IP, 1, 64, n=3000)
    path = str(tmp_path / "bf16.index")
    m.write_index(bix, path)
    rix = m.read_index(path, storage=1)
    rrows = rix.reconstruct_n().astype(np.float64)
    rad = _radius(rrows, xq[0], IP, 30)
    lims, D, I, _ = _rs(rix, xq, rad, _params(m, m.ALGO_TENSOR))
    _check(rrows, xq, rad, IP, lims, D, I, exact_q=0)


# ---- 7. interfaces ---------------------------------------------------------------------------------------------------
def test_torch_numpy_and_streams(m):
    import torch

    ix, rows, xb = _index(m, L2, 0, 384)
    xq = _queries(xb, 100, 12)
    radius = _radius(rows, xq[0], L2, 50)
    ln, Dn, In, _ = _rs(ix, xq, radius, None)
    lt, Dt, It = ix.range_search(torch.from_numpy(xq).cuda(), radius)
    assert lt.dtype == torch.int64 and lt.is_cuda and Dt.is_cuda and It.dtype == torch.int64
    assert np.array_equal(lt.cpu().numpy(), ln) and np.array_equal(Dt.cpu().numpy(), Dn) and np.array_equal(It.cpu().numpy(), In)
    # on a non-default stream, between an add and a search on the same index
    extra = _rows(500, 384, 99)
    tix = m.IndexFlatL2(384, storage=0)
    tix.add(xb)
    ref = m.IndexFlatL2(384, storage=0)
    ref.add(np.concatenate([xb, extra]))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tix.add(torch.from_numpy(extra).cuda())
        lt, Dt, It = tix.range_search(torch.from_numpy(xq).cuda(), radius)
        Ds, Is = tix.search(torch.from_numpy(xq).cuda(), 10)
        lt, Dt, It, Ds, Is = (t.cpu().numpy() for t in (lt, Dt, It, Ds, Is))
    lr, Dr, Ir, _ = _rs(ref, xq, radius, None)
    Dsr, Isr = ref.search(xq, 10)
    assert np.array_equal(lt, lr) and np.array_equal(Dt, Dr) and np.array_equal(It, Ir)
    assert np.array_equal(Is, Isr) and np.array_equal(Ds, Dsr)


def test_faiss_shim(m):
    import importlib

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rag-faiss-embedding_b200", "shim")
    sys.path.insert(0, shim)
    try:
        sys.modules.pop("faiss", None)
        faiss = importlib.import_module("faiss")
        ix, rows, xb = _index(m, L2, 0, 384)
        xq = _queries(xb, 7, 13)
        for cls, metric in ((faiss.IndexFlatL2, L2), (faiss.IndexFlatIP, IP)):
            f = cls(384)
            f.add(xb)
            r = f.reconstruct_n().astype(np.float64)
            radius = _radius(r, xq[0], metric, 10)
            lims, D, I = f.range_search(xq, radius)
            assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
            _check(r, xq, radius, metric, lims, D, I, exact_q=0)
    finally:
        sys.path.remove(shim)
        sys.modules.pop("faiss", None)


# ---- 8. no side effects on top-k search ------------------------------------------------------------------------------
def test_no_side_effects_on_topk(m):
    """Near-duplicates stored contiguously switch an index into per-thread heaps + the range pass: two twins run the
    same searches, one of them with range searches in between; everything search reports must stay identical."""
    xb, xq = _dense("contiguous", nc=300, dup=80, nq=512)
    a, b = m.IndexFlatL2(128, storage=0), m.IndexFlatL2(128, storage=0)
    a.add(xb)
    b.add(xb)
    p = _params(m, m.ALGO_TENSOR)
    keys = ("fallback_queries", "overflow_queries", "range_queries", "rescued_queries", "last_kprime", "last_algo", "searches")
    for i in range(6):
        Da, Ia = a.search(xq, 10, params=p)
        Db, Ib = b.search(xq, 10, params=p)
        sa, sb = a.stats(), b.stats()
        assert np.array_equal(Da, Db) and np.array_equal(Ia, Ib)
        assert {k: sa[k] for k in keys} == {k: sb[k] for k in keys}, i
        launches = sb["launches"]
        b.range_search(xq[:64], 1.0, params=p)
        b.range_search(xq, 1e-3, params=_params(m, m.ALGO_SCAN))
        sb2 = b.stats()
        assert {k: sb2[k] for k in keys} == {k: sb[k] for k in keys} and sb2["launches"] > launches
        assert sb2["last_launches"] == sb["last_launches"] and sb2["last_list_entries"] == sb["last_list_entries"]
    assert sa["range_queries"] + sa["fallback_queries"] > 0   # the data did engage the order-robust machinery
