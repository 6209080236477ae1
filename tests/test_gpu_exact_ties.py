"""GPU tier (-m gpu): tie order, radius strictness and result self-consistency, bit for bit on every search path.

The engine orders candidates by (key, id): among equal distances the lower label wins (DESIGN §3), and range search is
strict (L2 dist < radius, IP ip > radius; §3.5).  On general data neither can be checked bit for bit.  On integer lattice
data (tests/exact_checks.py) every fp32 sum is exact, so the float64 brute force is the one right answer, tie order
included, and bf16 storage and the tensor pass's coarse keys are exact too.  Every result below must equal it bit for
bit (check_exact), and every case asserts from the index's counters that the path it names really served it.

Planted tie groups: around a query q, group l holds rows whose key is the l-th best level -- L2: q + e_j (distance 1),
q + e_i + e_j (distance 2); IP (queries c * sigma, sigma a sign vector): b - sum of l signed unit vectors, b = mu + R sigma
(inner product c (sigma . b) - c l).  Bigger groups are copies of one row."""
import ctypes

import numpy as np
import pytest

from oracle import np_centre as orc_centre
from tests.exact_checks import (IP, L2, check_consistent, check_exact, check_range_exact, check_structure, lattice)

pytestmark = pytest.mark.gpu

METRICS = (L2, IP)
STORAGES = (0, 1)   # fp32, bf16
COUNTERS = ("fallback_queries", "overflow_queries", "rescued_queries", "range_queries")

# (n, d, nq, k) for the certifiable K2 ties, taken from test_gpu_edges.TENSOR_SHAPES: the streamed LIST kernel (k' = 32 and
# 192), the pair kernel, the Q-resident LIST kernel, HEAP with k' = 32 and 64, and a k' = 192 batch cut into several passes.
# (tests/test_exact_checks_cpu.py checks with the planner that they still reach each of them.)
TIE_SHAPES = [
    (30000, 385, 129, 10),
    (20000, 1536, 129, 100),
    (30000, 384, 833, 10),
    (30000, 384, 300, 10),
    (200, 128, 64, 10),
    (200, 128, 64, 20),
    (8000, 449, 4096, 100),
]
R, MU = 8, 3


@pytest.fixture(scope="module")
def m():
    import rag_faiss_embedding_b200 as mod

    assert mod.device_count() > 0, "no B200 visible"
    return mod


def _plan(m, nq, n, d, k):
    out = (ctypes.c_int32 * 12)()
    assert m._capi.load().b2f_plan_describe(nq, n, d, k, 0, out) == 0
    return dict(zip(["kp", "chunk", "passes", "list", "pair"], list(out)[:5]))


# ---- data --------------------------------------------------------------------------------------------------------------
def _queries(lat, metric, nq):
    if metric == L2:
        return lat.near(nq)
    sigma = lat.rng.choice(np.array([-1.0, 1.0], np.float32), (nq, lat.d))
    return (R * sigma).astype(np.float32)


def _level_rows(lat, metric, q, level, count):
    """count distinct rows (copies once the distinct ones run out) at tie level `level` (1 or 2) of query q."""
    d = lat.d
    rng = lat.rng
    out = []
    if metric == L2:
        for t in range(count):
            y = q.copy()
            js = rng.choice(d, level, replace=False)
            y[js] += rng.choice(np.array([-1.0, 1.0], np.float32), level)
            out.append(y)
    else:
        sigma = np.sign(q)
        b = lat.mu + R * sigma
        for t in range(count):
            y = b.copy()
            js = rng.choice(d, level, replace=False)
            y[js] -= sigma[js]
            out.append(y)
    ys = np.unique(np.array(out, np.float32), axis=0)
    if len(ys) < count:   # (collisions of the random picks: fill up with copies)
        ys = np.concatenate([ys, np.repeat(ys[:1], count - len(ys), 0)])
    return ys[rng.permutation(count)]


def _planted(n, d, nq, k, metric, seed, groups=None, max_planted=64):
    """A lattice of n rows and nq queries; a spread-out subset of the queries gets tie groups of sizes (0.6 k, 0.8 k) at
    levels 1 and 2, so that the k-th neighbour lies inside the level-2 group and both groups lie within k'."""
    lat = lattice(n, d, R, MU, seed)
    xq = _queries(lat, metric, nq)
    g = groups or (max(1, 6 * k // 10), max(1, 8 * k // 10))
    per = sum(g)
    P = max(1, min(nq, max_planted, (n // 2) // (3 * per)))
    which = np.unique(np.linspace(0, nq - 1, P).astype(np.int64))
    for q in which:
        for level, size in enumerate(g, 1):
            lat.plant(_level_rows(lat, metric, xq[q], level, size))
    lat.verify(xq)
    return lat, xq, which


def _index(m, lat, metric, storage):
    ix = m.IndexFlat(lat.d, metric, storage=storage)
    ix.add(lat.rows)
    assert np.array_equal(ix.reconstruct_n(), lat.rows)   # bf16 storage keeps lattice rows exactly
    return ix


def _search(m, ix, xq, k, algo, id_offset=0):
    """(D, I, counter deltas and the last_* fields of this search)."""
    before = ix.stats()
    p = m.SearchParams()
    p.algo = algo
    p.id_offset = id_offset
    D, I = ix.search(xq, k, params=p)
    after = ix.stats()
    st = {c: after[c] - before[c] for c in COUNTERS}
    st.update(last_algo=after["last_algo"], last_kprime=after["last_kprime"], last_launches=after["last_launches"])
    return D, I, st


def _exact(D, I, rows, xq, k, metric, id_offset=0):
    check_structure(D, I, metric, len(rows), id_offset)
    check_exact(D, I, rows, xq, k, metric, id_offset)


# ---- K1: the exact scan --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_scan_tie_order(m, metric, storage):
    """K1 at nq = 1, 2, 3, 5, 8, 9 (the NQ = 1 / 2 / 4 / 8 instantiations, more than one query group) and k = 1, 10, 100,
    1024: the planted level-2 group straddles k = 10; the integer background ties at k = 100 and 1024; query 0 also has
    1100 copies of one row at its best key, more rows at or below the cross-CTA bound than the gather holds
    (kGatherCap = 1024), which forces the two-level merge."""
    lat, xq, _ = _planted(6000, 128, 9, 10, metric, seed=1 + metric, max_planted=9)
    lat.plant(np.repeat(_level_rows(lat, metric, xq[0], 1, 1), 1100, 0))
    lat.verify(xq)
    ix = _index(m, lat, metric, storage)
    for k in (1, 10, 100, 1024):
        for nq in (1, 2, 3, 5, 8, 9):
            D, I, st = _search(m, ix, xq[:nq], k, m.ALGO_SCAN)
            _exact(D, I, lat.rows, xq[:nq], k, metric)
            assert st["last_algo"] == m.ALGO_SCAN and st["last_launches"] == 1 and st["fallback_queries"] == 0, (k, nq, st)


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_scan_shard_smaller_than_k(m, metric, storage):
    """A shard of 50 rows searched with k = 100 and a label offset: every row, in (distance, label) order, then padding."""
    lat = lattice(50, 64, R, MU, seed=7)
    xq = _queries(lat, metric, 3)
    ys = _level_rows(lat, metric, xq[0], 1, 4)
    lat.plant(np.concatenate([ys, ys]))   # duplicated rows: equal keys on different labels
    lat.verify(xq)
    ix = _index(m, lat, metric, storage)
    for nq in (1, 3):
        D, I, st = _search(m, ix, xq[:nq], 100, m.ALGO_SCAN, id_offset=5000)
        _exact(D, I, lat.rows, xq[:nq], 100, metric, id_offset=5000)
        assert (I[:, 50:] == -1).all() and st["last_algo"] == m.ALGO_SCAN


# ---- K2: ties the certification can prove ------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("n,d,nq,k", TIE_SHAPES)
def test_tensor_certified_ties(m, n, d, nq, k, metric):
    """Tie groups wholly inside k' with a wide gap to the background (keys 1 and 2 against ~d R^2): the boundary falls
    inside the level-2 group, so the result is the level-1 group plus the lowest ids of the level-2 group -- and the query
    certifies: no exact scan, no range pass."""
    lat, xq, which = _planted(n, d, nq, k, metric, seed=n + d + nq)
    plan = _plan(m, nq, n, d, k)
    for storage in STORAGES:
        ix = _index(m, lat, metric, storage)
        D, I, st = _search(m, ix, xq, k, m.ALGO_TENSOR)
        _exact(D, I, lat.rows, xq, k, metric)
        assert st["last_algo"] == m.ALGO_TENSOR and st["last_kprime"] == plan["kp"], st
        assert st["fallback_queries"] == 0 and st["range_queries"] == 0 and st["overflow_queries"] == 0, (storage, st)


def _rows_of_norm(T, count, d, rng):
    """count distinct integer vectors with squared norm exactly T and every |coordinate| <= 256: d - 16 coordinates
    near sqrt((T - 5e5) / (d - 16)), the remainder (~5e5) taken greedily by the last 16."""
    body = d - 16
    a = int(np.sqrt((T - 500000) / body)) - 2
    out = []
    while len(out) < count:
        v = np.zeros(d, np.int64)
        v[:body] = (a + rng.integers(0, 5, body)) * rng.choice((-1, 1), body)
        rem = T - int((v * v).sum())
        for j in range(body, d):
            if rem <= 0:
                break
            t = min(int(np.sqrt(rem)), 256)
            v[j] = t * rng.choice((-1, 1))
            rem -= t * t
        if rem == 0:
            out.append(v)
    return np.array(out, np.float32)


def _certify_boundary(B, Bmax, d):
    """rerank_certified (L2) restated in fp32 for a query at the centre (q' = 0, e_q = 0) of rows stored exactly
    (max_row_err = 0), the k'-th coarse key B and max |x'|^2 = Bmax: the largest k-th key it may NOT certify is
    fl(L * L * (1 - 4e-7)), L = sqrt(B - nu).  With perfect-square Bmax and B, every step is exact or rounded once."""
    f = np.float32
    gam = f(f(4) * f(d + 16)) * f(5.9604645e-8)
    m = np.sqrt(f(Bmax))
    nu = gam * (f(f(f(2) * f(0)) * m + f(0)) + m * m)
    L = np.sqrt(max((f(B) + f(0)) - nu, f(0)))
    return (L * L) * (f(1) - f(4e-7))


@pytest.mark.parametrize("inside", [False, True])
def test_tensor_certification_boundary_is_strict(m, inside):
    """A query at the centre, 10 rows at squared distance A, 30 at B = 3000^2 (the k'-th candidate lies among them) and
    the rest farther out up to Bmax = 4000^2.  Every key, the coarse ones included, is exact, so the certification test
    of the first re-rank sees exactly L = sqrt(B - nu): a k-th key A equal to fl(L^2 (1 - 4e-7)) must NOT certify there
    (the extended stage or the exact scan answers), one less must.  The answer is the 10 rows at A in id order either way."""
    d, k, nq = 256, 10, 4
    B, Bmax = 3000 ** 2, 3600 ** 2
    P = _certify_boundary(B, Bmax, d)
    assert float(P).is_integer() and B // 2 < P < B
    A = int(P) - (1 if inside else 0)
    rng = np.random.default_rng(71)
    far = rng.integers(B + 20000, Bmax, 2000 - 21)
    half = np.concatenate([_rows_of_norm(A, 5, d, rng), _rows_of_norm(B, 15, d, rng), _rows_of_norm(Bmax, 1, d, rng)]
                          + [_rows_of_norm(int(t), 1, d, rng) for t in far])
    rows = np.empty((2 * len(half), d), np.float32)
    rows[0::2], rows[1::2] = half, -half            # pairs +-x': the centre is 0
    rows = rows[rng.permutation(len(rows))]
    assert np.array_equal(orc_centre(rows), np.zeros(d, np.float32)) and np.abs(rows).max() <= 256
    assert ((rows.astype(np.float64) ** 2).sum(1) <= Bmax).all()
    xq = np.zeros((nq, d), np.float32)
    for storage in STORAGES:
        ix = m.IndexFlat(d, L2, storage=storage)
        ix.add(rows)
        assert np.array_equal(ix.reconstruct_n(), rows)
        D, I, st = _search(m, ix, xq, k, m.ALGO_TENSOR)
        _exact(D, I, rows, xq, k, L2)
        assert (D == A).all()
        first_failed = st["rescued_queries"] + st["fallback_queries"]
        assert st["last_algo"] == m.ALGO_TENSOR and first_failed == (0 if inside else nq), (A, P, st)


# ---- K2: ties it cannot certify --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_tensor_uncertifiable_ties(m, metric, storage):
    """Groups larger than k' at the k-th key: 40 and 100 distinct rows (the extended certification over every list entry
    can rescue them), 400 and 1500 copies (neither the k' best nor the lists certify: the closing exact scan answers, and
    from the second search on the range pass), and 5000 copies (more equal keys than the merge holds: it gives up, counted
    as an overflow, and the exact scan answers).  Whichever path served a query, the result is exact."""
    k = 10
    lat = lattice(40000, 128, R, MU, seed=11 + metric)
    sizes = [40] * 4 + [100] * 4 + [400] * 4 + [1500] * 2 + [5000]
    xq = _queries(lat, metric, 48)
    for q, size in enumerate(sizes):
        ys = _level_rows(lat, metric, xq[q], 1, size if size <= 100 else 1)
        lat.plant(ys if size <= 100 else np.repeat(ys, size, 0))
    lat.verify(xq)
    ix = _index(m, lat, metric, storage)
    seen = []
    for it in range(3):
        D, I, st = _search(m, ix, xq, k, m.ALGO_TENSOR)
        _exact(D, I, lat.rows, xq, k, metric)
        assert st["last_algo"] == m.ALGO_TENSOR, st
        seen.append(st)
    print(f"metric {metric} storage {storage}: " + "; ".join(str({c: s[c] for c in COUNTERS}) for s in seen))
    assert seen[0]["fallback_queries"] >= 3 and seen[0]["overflow_queries"] >= 1, seen[0]
    assert sum(s["rescued_queries"] for s in seen) > 0, seen
    assert seen[1]["range_queries"] > 0 and seen[2]["range_queries"] > 0, seen
    assert seen[2]["fallback_queries"] < seen[0]["fallback_queries"], seen


@pytest.mark.parametrize("metric", METRICS)
def test_tensor_contiguous_ties_heap_mode(m, metric):
    """300 groups of 80 copies stored side by side: a query's best rows sit in one or two lists, the shared thresholds never
    tighten and the lists overflow, which switches the index to per-thread heaps plus the range pass.  Exact throughout."""
    k, nq = 10, 256
    lat = lattice(60000, 128, R, MU, seed=21 + metric)
    centres = _queries(lat, metric, 300)
    for c in centres:
        lat.plant(np.repeat(c[None], 80, 0), contiguous=True)
    pick = lat.rng.integers(0, 300, nq)
    if metric == L2:   # at distance 1 from the 80 copies of their group
        xq = centres[pick] + np.eye(128, dtype=np.float32)[lat.rng.integers(0, 128, nq)]
    else:              # the group's row is the best inner product (c sigma . (R sigma) against |v| <= R elsewhere)
        xq = centres[pick].copy()
    xq = xq.astype(np.float32)
    lat.verify(xq)
    ix = _index(m, lat, metric, 0)
    seen = []
    for it in range(4):
        D, I, st = _search(m, ix, xq, k, m.ALGO_TENSOR)
        _exact(D, I, lat.rows, xq, k, metric)
        seen.append(st)
    print(f"metric {metric}: " + "; ".join(str({c: s[c] for c in COUNTERS}) for s in seen))
    assert seen[0]["overflow_queries"] > nq // 8, seen[0]
    assert seen[3]["overflow_queries"] == 0 and seen[3]["range_queries"] > 0 and seen[3]["fallback_queries"] <= 4, seen


# ---- batch composition ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_batch_composition_invariance(m, metric):
    """The same lattice queries searched alone (AUTO: the exact scan on fp32 storage), in batches of 7, 129 and 1024, and
    inside a batch of 8192 (the warp-per-query merge) give the same D and I bits -- the float64 brute force's."""
    k = 10
    lat, xq, _ = _planted(20000, 128, 8192, k, metric, seed=31 + metric)
    ix = _index(m, lat, metric, 0)
    D, I, st = _search(m, ix, xq, k, m.ALGO_AUTO)
    assert st["last_algo"] == m.ALGO_TENSOR and st["fallback_queries"] == 0, st
    _exact(D, I, lat.rows, xq, k, metric)
    for q in (0, 1, 4095, 8191):
        D1, I1, st = _search(m, ix, xq[q:q + 1], k, m.ALGO_AUTO)
        assert st["last_algo"] == m.ALGO_SCAN, st
        assert np.array_equal(I1[0], I[q]) and np.array_equal(D1[0].view(np.uint32), D[q].view(np.uint32)), q
    for b in (7, 129, 1024):
        for q0 in (0, 8192 - b, 3000):
            Db, Ib, st = _search(m, ix, xq[q0:q0 + b], k, m.ALGO_AUTO)
            assert st["last_algo"] == m.ALGO_TENSOR, (b, st)
            assert np.array_equal(Ib, I[q0:q0 + b]) and np.array_equal(Db.view(np.uint32), D[q0:q0 + b].view(np.uint32)), (b, q0)


# ---- range search ---------------------------------------------------------------------------------------------------------
def _range(m, ix, xq, radius, algo):
    p = m.SearchParams()
    p.algo = algo
    lims, D, I = ix.range_search(xq, radius, params=p)
    return lims, D, I, dict(ix.last_range_info)


def _radii(r):
    """An attained key r and one fp32 ulp to either side."""
    r = np.float32(r)
    return [float(np.nextafter(r, np.float32(-np.inf))), float(r), float(np.nextafter(r, np.float32(np.inf)))]


@pytest.mark.parametrize("storage", STORAGES)
@pytest.mark.parametrize("metric", METRICS)
def test_range_radius_on_attained_keys(m, metric, storage):
    """The radius set at attained integer keys (the planted level-1 / level-2 keys and a background key with many rows on
    it) and one ulp to either side, under SCAN, TENSOR and AUTO: rows exactly on the radius are never hits (L2 dist < r,
    IP ip > r), and one ulp past it they all are -- the tensor pass's inverted bound must list a row one ulp inside."""
    lat, xq, which = _planted(6000, 64, 40, 10, metric, seed=41 + metric)
    ix = _index(m, lat, metric, storage)
    from oracle import np_search_f64

    Dk, _ = np_search_f64(lat.rows, xq[:1], 200, metric)
    for r in (Dk[0, 0], Dk[0, 9], Dk[0, 150]):
        on_counts = []
        for radius in _radii(r):
            res = {}
            for algo in (m.ALGO_SCAN, m.ALGO_TENSOR, m.ALGO_AUTO):
                lims, D, I, info = _range(m, ix, xq, radius, algo)
                check_range_exact(lims, D, I, lat.rows, xq, radius, metric)
                assert info["tensor_queries"] + info["scan_queries"] == len(xq)
                if algo == m.ALGO_SCAN:
                    assert info["scan_queries"] == len(xq), info
                else:
                    assert info["tensor_queries"] > 0, (algo, info)
                res[algo] = (lims, D, I)
            for a, b in zip(res[m.ALGO_TENSOR], res[m.ALGO_SCAN]):
                assert np.array_equal(a, b)
            on_counts.append(int(np.sum(res[m.ALGO_SCAN][1] == np.float32(r))))
        # below / at / past the radius: rows on r enter only one ulp past it (L2: above r, IP: below r)
        inside = on_counts[2] if metric == L2 else on_counts[0]
        assert on_counts[1] == 0 and inside > 0 and on_counts[0 if metric == L2 else 2] == 0, (r, on_counts)


def test_range_ip_radius_zero_on_orthogonal_rows(m):
    """IP radius 0 against rows orthogonal to the query: ip == 0 exactly, never a hit; at -1 ulp (a subnormal) they all are."""
    lat = lattice(4000, 64, R, 0, seed=51)
    xq = lat.near(8)
    ortho = []
    for q in xq[:4]:
        for i, j in zip(range(0, 64, 2), range(1, 64, 2)):
            y = np.zeros(64, np.float32)
            y[i], y[j] = q[j], -q[i]
            ortho.append(y)
    ids = lat.plant(np.array(ortho, np.float32))
    lat.verify(xq)
    for storage in STORAGES:
        ix = _index(m, lat, IP, storage)
        for radius in (0.0, float(np.nextafter(np.float32(0), np.float32(-np.inf)))):
            for algo in (m.ALGO_SCAN, m.ALGO_TENSOR, m.ALGO_AUTO):
                lims, D, I, info = _range(m, ix, xq, radius, algo)
                check_range_exact(lims, D, I, lat.rows, xq, radius, IP)
                hit_ortho = np.isin(I[lims[0]:lims[1]], ids[:32])
                assert hit_ortho.sum() == (0 if radius == 0.0 else 32), (radius, algo, int(hit_ortho.sum()))


@pytest.mark.parametrize("metric", METRICS)
def test_range_chunk_boundary_and_big_tie_group(m, metric):
    """1025 queries (two chunks of the range pass) and a query with 4200 hits at one key, more than the list filter stages
    (4096), which must go to the exact range scan -- both exact on both storages."""
    lat, xq, _ = _planted(12000, 64, 1025, 10, metric, seed=61 + metric)
    lat.plant(np.repeat(_level_rows(lat, metric, xq[5], 1, 1), 4200, 0))
    lat.verify(xq)
    from oracle import np_search_f64

    Dk, _ = np_search_f64(lat.rows, xq[5:6], 4300, metric)
    r = Dk[0, 4250]   # past the 4200 copies
    for storage in STORAGES:
        ix = _index(m, lat, metric, storage)
        for radius in _radii(r)[1:]:
            lims, D, I, info = _range(m, ix, xq, radius, m.ALGO_TENSOR)
            check_range_exact(lims, D, I, lat.rows, xq, radius, metric)
            assert info["scan_queries"] >= 1 and info["tensor_queries"] > 0, info
            assert lims[6] - lims[5] >= 4200


# ---- non-lattice data: a D must still belong to its I ---------------------------------------------------------------------
def test_near_duplicate_ip_results_are_consistent(m):
    """The normalised near-duplicate inner-product data that test_gpu_parity.py and test_gpu_edges.py check with
    min_recall = 0 (fp32 inner products tie there, so the exact answer is not defined bit for bit): every returned distance
    must still be the fp32 inner product of the row beside it, within the rigorous rounding bound, and no row left out may
    beat the last one returned by more than that bound."""
    from tests.test_gpu_parity import _near_duplicates

    k = 10
    xb, xq = _near_duplicates(60, 400, 512, 0)
    ix = m.IndexFlat(xb.shape[1], IP)
    ix.add(xb)
    for it in range(2):   # the second search runs the range pass
        D, I, st = _search(m, ix, xq, k, m.ALGO_TENSOR)
        check_structure(D, I, IP, len(xb))
        check_consistent(D, I, xb, xq, IP)
    assert st["range_queries"] > 0, st
    # the warp-per-query merge's near-duplicate batch (test_big_batch_warp_merge)
    d, nq = 128, 8192
    rng = np.random.default_rng(5)
    centres = rng.standard_normal((600, d)).astype(np.float32)
    xb2 = (np.repeat(centres, 40, axis=0) + rng.standard_normal((24000, d)).astype(np.float32) * 2e-3).astype(np.float32)
    xq2 = (centres[rng.integers(0, 600, nq)] + rng.standard_normal((nq, d)).astype(np.float32) * 2e-3).astype(np.float32)
    xb2 /= np.linalg.norm(xb2, axis=1, keepdims=True)
    xq2 /= np.linalg.norm(xq2, axis=1, keepdims=True)
    ix2 = m.IndexFlat(d, IP)
    ix2.add(xb2)
    D2, I2, _ = _search(m, ix2, xq2, k, m.ALGO_TENSOR)
    check_structure(D2, I2, IP, len(xb2))
    check_consistent(D2, I2, xb2, xq2, IP)
