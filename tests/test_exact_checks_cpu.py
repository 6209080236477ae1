"""CPU tier: the lattice generator and the strict checkers of tests/exact_checks.py, checked without a GPU.

The generator's premise (exact centre, exact bf16 rows, keys below 2^24) holds over a grid of widths, radii and
centres; on such data the C restatement and the float64 brute force agree bit for bit, ids included; and every checker
rejects a result corrupted in the way it exists to catch."""
import numpy as np
import pytest

import oracle as orc
from tests.exact_checks import (FLT_MAX, IP, L2, assert_exact_premise, check_consistent, check_exact, check_range_exact,
                                check_structure, lattice)
from tests.range_reference import np_range_search_f64


@pytest.mark.parametrize("n,d,R,mu", [
    (1000, 128, 8, 0), (1001, 7, 20, 3), (4000, 1536, 8, -5), (70001, 16, 100, 17), (66000, 384, 40, 0), (3000, 4096, 8, 2),
])
def test_lattice_premise(n, d, R, mu):
    lat = lattice(n, d, R, mu, seed=n + d)
    assert lat.rows.shape == (n, d) and lat.rows.dtype == np.float32
    assert np.array_equal(orc.np_centre(lat.rows), np.full(d, mu, np.float32))
    assert np.array_equal(orc.np_bf16_rows(lat.rows, lat.mu), lat.rows)
    # planting keeps the premise: duplicates and unit offsets around a query, at shuffled ids
    q = lat.near(1)[0]
    ids = lat.plant(np.concatenate([np.repeat(q[None], 5, 0), q + np.eye(d, dtype=np.float32)[:3]]))
    assert len(set(ids.tolist())) == 8 and np.array_equal(lat.rows[ids[:5]], np.repeat(q[None], 5, 0))
    run = lat.plant(np.repeat(q[None] + 1, 4, 0), contiguous=True)
    assert np.array_equal(np.diff(run), [2, 2, 2])
    lat.verify(lat.near(16))
    # a random perturbation of one row breaks the centre: the generator's assertion must notice
    bad = lat.rows.copy()
    bad[0, 0] += 1
    with pytest.raises(AssertionError):
        assert_exact_premise(bad, lat.near(2), lat.mu)


def test_lattice_rejects_keys_beyond_exact_range():
    with pytest.raises(AssertionError):
        lattice(100, 4096, 60, 0, seed=1)   # 4096 * (2 * 60)^2 * 2 > 2^24


@pytest.mark.parametrize("metric", [L2, IP])
@pytest.mark.parametrize("nq", [5, 19, 20, 64])
def test_c_oracle_equals_float64_on_lattice(metric, nq):
    """c_search switches from its sequential to its blas form at nq = 20; on lattice data both are exact, so they must
    equal the float64 brute force bit for bit, tie order included (duplicated rows and planted equal-key groups)."""
    lat = lattice(6000, 128, 8, 2, seed=nq)
    xq = lat.near(nq)
    for q in xq[:3]:
        lat.plant(np.repeat(q[None] + np.eye(128, dtype=np.float32)[0], 12, 0))   # 12 rows at L2 distance 1
    lat.verify(xq)
    for k in (1, 10, 100):
        D, I = orc.c_search(lat.rows, xq, k, metric)
        D_ref, I_ref = orc.np_search_f64(lat.rows, xq, k, metric)
        assert np.array_equal(I, I_ref) and np.array_equal(D, D_ref), (k, metric)
        check_structure(D, I, metric, len(lat.rows))
        check_exact(D, I, lat.rows, xq, k, metric)
        check_consistent(D, I, lat.rows, xq, metric)


@pytest.fixture(scope="module")
def tied():
    """A lattice with a tie group of 12 rows at L2 distance 1 around query 0, and the exact top-20 of 3 queries."""
    lat = lattice(3000, 32, 6, 0, seed=5)
    xq = lat.near(3)
    ids = np.sort(lat.plant(np.repeat(xq[:1] + np.eye(32, dtype=np.float32)[3], 12, 0)))
    D, I = orc.np_search_f64(lat.rows, xq, 20, L2)
    assert np.array_equal(I[0, :12], ids) and (D[0, :12] == 1).all()
    return lat, xq, D, I


def _rejects(fn, *args):
    with pytest.raises(AssertionError):
        fn(*args)


def test_checkers_accept_the_exact_answer(tied):
    lat, xq, D, I = tied
    check_structure(D, I, L2, len(lat.rows))
    check_consistent(D, I, lat.rows, xq, L2)
    check_exact(D, I, lat.rows, xq, 20, L2)


def test_checkers_reject_corrupted_results(tied):
    lat, xq, D, I = tied
    # two tied ids swapped
    I2 = I.copy()
    I2[0, [2, 5]] = I2[0, [5, 2]]
    _rejects(check_structure, D, I2, L2, len(lat.rows))
    _rejects(check_exact, D, I2, lat.rows, xq, 20, L2)
    # a duplicated id (two equal rows of a tie group reported as one row twice)
    I3 = I.copy()
    I3[0, 3] = I3[0, 2]
    _rejects(check_structure, D, I3, L2, len(lat.rows))
    # a D taken from another row
    D4 = D.copy()
    D4[1, 4] = D[1, 7]
    _rejects(check_consistent, D4, I, lat.rows, xq, L2)
    # the lowest-id member at the k boundary replaced by a row beyond the cut with a near-equal distance
    k = 8
    I5 = I[:, :k].copy()
    I5[0, k - 1] = I[0, k]           # the next member of the same tie group: equal distance, higher id
    check_structure(D[:, :k], I5, L2, len(lat.rows))   # (structure alone cannot tell)
    _rejects(check_exact, D[:, :k], I5, lat.rows, xq, k, L2)
    # padding in the middle of a row
    D6, I6 = D.copy(), I.copy()
    D6[2, 4], I6[2, 4] = FLT_MAX, -1
    _rejects(check_structure, D6, I6, L2, len(lat.rows))
    # padding although rows remain, and a row that beats the last returned one
    _rejects(check_consistent, D6[:, :5], I6[:, :5], lat.rows, xq, L2)
    D40, I40 = orc.np_search_f64(lat.rows, xq, 40, L2)
    assert D40[1, 35] > D40[1, 19]
    D7, I7 = D.copy(), I.copy()
    D7[1, 19], I7[1, 19] = D40[1, 35], I40[1, 35]   # a consistent, sorted row that skipped the true 20th neighbour
    check_structure(D7, I7, L2, len(lat.rows))
    _rejects(check_consistent, D7, I7, lat.rows, xq, L2)
    # ids out of range, wrong dtypes
    _rejects(check_structure, D, I + len(lat.rows), L2, len(lat.rows))
    _rejects(check_structure, D.astype(np.float64), I, L2, len(lat.rows))


def test_range_checker_rejects_a_hit_on_the_radius(tied):
    lat, xq, D, I = tied
    for metric in (L2, IP):
        keys = orc.np_search_f64(lat.rows, xq, 40, metric)[0]
        r = float(keys[0, 15])                 # an attained key
        lims, Dr, Ir = np_range_search_f64(lat.rows, xq, r, metric)
        lims, Dr = lims.astype(np.uint64), Dr.astype(np.float32)
        check_range_exact(lims, Dr, Ir, lat.rows, xq, r, metric)
        # the rows exactly on the radius, added to query 0's hits (as a non-strict comparison would)
        ref = orc.np_search_f64(lat.rows, xq[:1], len(lat.rows), metric)
        on = np.sort(ref[1][0][ref[0][0] == r])
        assert len(on) > 0
        hi, hd = Ir[lims[0]:lims[1]], Dr[lims[0]:lims[1]]
        allI = np.concatenate([hi, on])
        order = np.argsort(allI)
        allD = np.concatenate([hd, np.full(len(on), r, np.float32)])[order]
        I_bad = np.concatenate([allI[order], Ir[lims[1]:]])
        D_bad = np.concatenate([allD, Dr[lims[1]:]])
        lims_bad = lims.astype(np.int64).copy()
        lims_bad[1:] += len(on)
        _rejects(check_range_exact, lims_bad, D_bad, I_bad, lat.rows, xq, r, metric)
        # and one hit dropped
        _rejects(check_range_exact, np.concatenate([[0], lims[1:].astype(np.int64) - 1]), Dr[1:], Ir[1:], lat.rows, xq, r,
                 metric)


def test_gpu_tie_shapes_reach_every_tensor_kernel():
    """The certifiable-tie shapes of tests/test_gpu_exact_ties.py still reach each K2 variant (checked with the planner,
    no GPU needed)."""
    from rag_faiss_embedding_b200 import _capi
    from tests import test_gpu_exact_ties as ties
    from tests.test_edges_plan_cpu import _variants

    lib = _capi.load()
    reached = set()
    for n, d, nq, k in ties.TIE_SHAPES:
        reached |= _variants(lib, nq, n, d, k, 0)
    required = {"pair", "Q-resident list", "streamed list", "heap k'=32", "heap k'=64", "multi-pass", "k'=192"}
    assert required <= reached, sorted(required - reached)
