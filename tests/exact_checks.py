"""Integer lattice data and strict result checkers for the exactness tests (CPU and GPU tiers).  TEST INFRASTRUCTURE ONLY.

On general data a search result can only be checked within a tolerance: fp32 and float64 disagree in the last bits, and
`oracle.recall_and_errors` excuses any position whose distance is within 1e-5 of the reference's.  That hides a kernel
that returns the wrong member of a tie group, the same id twice, or a distance that does not belong to the id beside it.

On lattice data it cannot hide.  When every coordinate is a small integer and every partial sum stays below 2^24, every
fp32 sum is exact in any order, so the float64 brute force (`oracle.np_search_f64`) is THE answer, tie order included,
and every search path must reproduce it bit for bit.  When in addition the centre mu is an integer vector and every
|x - mu| <= 256, bf16(x - mu) is exact as well: bf16 storage keeps the rows unchanged and the tensor pass's coarse keys
equal the exact keys (e_q = 0, max_row_err = 0), so certification has no rounding to hide behind.

`lattice` builds such rows in pairs (mu + v, mu - v), so the first min(n, 65536) rows -- the rows the index takes its
centre from -- have the exact mean mu.  Rows planted around a query keep the pairs: every planted row y has its mirror
2 mu - y in the partner slot."""
from __future__ import annotations

import numpy as np

import oracle as orc
from tests.range_reference import np_range_search_f64

L2, IP = orc.METRIC_L2, orc.METRIC_INNER_PRODUCT
FLT_MAX = np.finfo(np.float32).max
U = 2.0 ** -24            # fp32 unit roundoff
EXACT_SUM = 2.0 ** 24     # integer sums below this are exact in fp32
BF16_EXACT = 256          # integers with |v| <= 256 are exact in bf16


class Lattice:
    """n integer rows around the integer centre mu, in pairs (mu + v, mu - v) with |v| <= R per coordinate (an odd n ends
    with the row mu itself).  `plant` overwrites pairs at shuffled ids with chosen rows and their mirrors."""

    def __init__(self, n, d, R, mu, seed):
        self.n, self.d, self.R = n, d, R
        self.mu = np.asarray(mu, np.float32).reshape(d)
        assert np.array_equal(self.mu, np.rint(self.mu)), "mu must be an integer vector"
        self.rng = np.random.default_rng(seed)
        npairs = n // 2
        v = self.rng.integers(-R, R + 1, (npairs, d)).astype(np.float32)
        rows = np.empty((n, d), np.float32)
        rows[0:2 * npairs:2] = self.mu + v
        rows[1:2 * npairs:2] = self.mu - v
        if n % 2:
            rows[-1] = self.mu
        self.rows = rows
        # pair slots still free for planting, in random order (only pairs inside the centre's rows need their mirror
        # there, but every planted row gets one: the layout is the same on both sides of 65536 rows)
        self._order = self.rng.permutation(npairs)
        self._taken = np.zeros(npairs, bool)

    def mirror(self, y):
        return (2 * self.mu - np.asarray(y, np.float32)).astype(np.float32)

    def plant(self, ys, contiguous=False):
        """Write the rows ys [m, d] into m free pairs (ys at the even or odd slot at random, the mirror at the other);
        contiguous: m consecutive pairs with ys at the even slots, i.e. a run of rows a query finds side by side.
        Returns the row ids of ys."""
        ys = np.asarray(ys, np.float32).reshape(-1, self.d)
        m = len(ys)
        if contiguous:
            run = np.convolve(~self._taken, np.ones(m, np.int64), "valid")   # free pairs in each window of m
            starts = np.nonzero(run == m)[0]
            assert len(starts), "no run of free pairs long enough"
            pairs = np.arange(starts[0], starts[0] + m)
            side = np.zeros(m, np.int64)
        else:
            free = self._order[~self._taken[self._order]]
            assert len(free) >= m, "not enough free pairs to plant into"
            pairs = free[:m]
            side = self.rng.integers(0, 2, m)
        self._taken[pairs] = True
        ids = 2 * pairs + side
        self.rows[ids] = ys
        self.rows[2 * pairs + 1 - side] = self.mirror(ys)
        return ids

    def near(self, nq, spread=None):
        """nq lattice queries around mu (coordinates mu + w, |w| <= spread, default R)."""
        s = self.R if spread is None else spread
        return (self.mu + self.rng.integers(-s, s + 1, (nq, self.d))).astype(np.float32)

    def verify(self, xq):
        """The premise of the exact checks, asserted for these rows and queries."""
        assert_exact_premise(self.rows, xq, self.mu)


def lattice(n, d, R, mu=0, seed=0):
    """Lattice rows (see Lattice); mu: an integer vector, or an integer broadcast to every coordinate."""
    mu = np.broadcast_to(np.asarray(mu, np.float32), (d,)).copy()
    lat = Lattice(n, d, R, mu, seed)
    assert_exact_premise(lat.rows, lat.near(4), lat.mu)
    return lat


def assert_exact_premise(rows, xq, mu):
    """Everything the exact checks rely on: integer rows and queries; the centre of the first rows is mu, exactly;
    bf16 storage keeps the rows (and the queries' bf16 copies are exact); every L2 and IP key, and so every partial
    sum of one in any order, is an integer below 2^24 in magnitude."""
    rows = np.asarray(rows, np.float32)
    xq = np.asarray(xq, np.float32)
    assert np.array_equal(rows, np.rint(rows)) and np.array_equal(xq, np.rint(xq)), "rows and queries must be integers"
    assert np.array_equal(orc.np_centre(rows), mu), "the first rows' centre is not mu"
    assert np.array_equal(orc.np_bf16_rows(rows, mu), rows), "bf16 storage would round these rows"
    assert np.abs(rows - mu).max() <= BF16_EXACT and np.abs(xq - mu).max() <= BF16_EXACT
    # L2: sum_i (x_i - q_i)^2 <= d * (max |x - mu| + max |q - mu|)^2; the tensor pass's |x'|^2, |q'|^2 and 2 q'.x' are
    # bounded by the same; IP: sum_i |x_i q_i|
    a = np.abs(rows - mu).max(0).astype(np.float64)
    b = np.abs(xq - mu).max(0).astype(np.float64)
    assert float(((a + b) ** 2).sum()) * 2 < EXACT_SUM, "L2 keys could reach 2^24"
    assert float((np.abs(rows).max(0).astype(np.float64) * np.abs(xq).max(0)).sum()) < EXACT_SUM, "IP keys could reach 2^24"


# ---- checkers ------------------------------------------------------------------------------------------------------------
def _pad(metric):
    return FLT_MAX if metric == L2 else -FLT_MAX


def check_structure(D, I, metric, ntotal=None, id_offset=0):
    """What every top-k result must satisfy, whatever the data: float32 / int64 [nq, k]; padding (-1, +-FLT_MAX) only as a
    trailing run; ids in [id_offset, id_offset + ntotal) and unique within a row; each row sorted by the returned fp32
    values in the metric's direction, equal values in ascending id order."""
    D, I = np.asarray(D), np.asarray(I)
    assert D.dtype == np.float32 and I.dtype == np.int64, (D.dtype, I.dtype)
    assert D.ndim == 2 and D.shape == I.shape, (D.shape, I.shape)
    nq, k = I.shape
    if nq == 0:
        return
    pad = I == -1
    assert np.array_equal(D[pad], np.full(int(pad.sum()), _pad(metric), np.float32)), "padding ids with non-padding distances"
    # trailing: once padded, padded to the end
    assert not np.any(pad[:, :-1] & ~pad[:, 1:]), f"padding in the middle of a row: {np.nonzero(pad[:, :-1] & ~pad[:, 1:])[0][:5]}"
    valid = ~pad
    assert np.all(I[valid] >= id_offset), "negative or foreign id"
    if ntotal is not None:
        assert np.all(I[valid] < id_offset + ntotal), "id beyond the index"
    assert not np.any(np.isnan(D[valid])), "NaN distance returned"
    key = D.astype(np.float64) if metric == L2 else -D.astype(np.float64)
    both = valid[:, :-1] & valid[:, 1:]
    up = key[:, 1:] > key[:, :-1]
    tie = key[:, 1:] == key[:, :-1]
    ordered = up | (tie & (I[:, 1:] > I[:, :-1]))
    bad = both & ~ordered
    assert not bad.any(), f"rows not ordered by (distance, id): query {np.nonzero(bad)[0][0]}, position {np.nonzero(bad)[1][0]}"
    srt = np.sort(np.where(valid, I, -2 - np.arange(k)[None, :]), axis=1)   # (padding made distinct)
    assert not np.any(srt[:, 1:] == srt[:, :-1]), "an id returned twice in one row"


def _keys64(rows, xq, metric):
    """float64 keys [nq, n] (smaller is better) and the fp32 error bound of each, for the exact-difference / dot forms."""
    rows = np.asarray(rows, np.float64)
    xq = np.asarray(xq, np.float64)
    d = rows.shape[1]
    if metric == L2:
        k = (xq * xq).sum(1)[:, None] + (rows * rows).sum(1)[None, :] - 2.0 * (xq @ rows.T)
        small = k < 1e-6 * ((xq * xq).sum(1)[:, None] + 1e-300)
        if small.any():
            qi, xi = np.nonzero(small)
            k[qi, xi] = ((xq[qi] - rows[xi]) ** 2).sum(1)
        k = np.maximum(k, 0.0)
        return k, (d + 4) * U * k
    ip = xq @ rows.T
    return -ip, (d + 2) * U * (np.abs(xq) @ np.abs(rows).T)


def check_consistent(D, I, rows, xq, metric):
    """Against the authoritative rows: every returned D[q, j] is within the fp32 rounding bound of the float64 distance of
    row I[q, j] (L2 (d + 4) u delta, IP (d + 2) u sum |x_i q_i|), and no row outside a query's result has a float64 key
    below its last returned row's by more than both bounds (completeness)."""
    D, I = np.asarray(D), np.asarray(I)
    for q0 in range(0, I.shape[0], 256):   # (a [256, n] float64 block of keys at a time)
        _check_consistent_block(D[q0:q0 + 256], I[q0:q0 + 256], rows, xq[q0:q0 + 256], metric, q0)


def _check_consistent_block(D, I, rows, xq, metric, q0):
    keys, err = _keys64(rows, xq, metric)
    n = keys.shape[1]
    for q in range(I.shape[0]):
        sel = I[q][I[q] >= 0]
        assert np.all(sel < n)
        got = D[q, :len(sel)].astype(np.float64)
        got_key = got if metric == L2 else -got
        dev = np.abs(got_key - keys[q, sel])
        tol = err[q, sel] + 1e-300
        assert np.all(dev <= tol), \
            f"query {q0 + q}: D is not the distance of its id (position {int(np.argmax(dev / tol))}, off by {dev.max():.3g})"
        finite = np.isfinite(keys[q])
        rest = np.ones(n, bool)
        rest[sel] = False
        rest &= finite
        if len(sel) < I.shape[1]:   # padded: every row with a finite key must be in the result
            assert not rest.any(), f"query {q0 + q}: padded although rows {np.nonzero(rest)[0][:5]} exist"
            continue
        if not rest.any() or not len(sel):
            continue
        last = sel[-1]
        beat = rest & (keys[q] < keys[q, last] - err[q, last] - err[q])
        assert not beat.any(), f"query {q0 + q}: row {np.nonzero(beat)[0][0]} beats the last returned row {last}"


def check_exact(D, I, rows, xq, k, metric, id_offset=0):
    """Lattice data: (D, I) equals the float64 brute force exactly -- every id in its place, tie order included, every
    distance equal (np.array_equal, no tolerance)."""
    D_ref, I_ref = orc.np_search_f64(rows, xq, k, metric)
    I = np.asarray(I)
    got_I = np.where(I >= 0, I - id_offset, -1)
    if not (np.array_equal(got_I, I_ref) and np.array_equal(np.asarray(D), D_ref)):
        bad = np.nonzero((got_I != I_ref) | (np.asarray(D) != D_ref))
        q, j = int(bad[0][0]), int(bad[1][0])
        raise AssertionError(f"{len(bad[0])} positions differ from the float64 brute force; first: query {q} position {j}: "
                             f"got ({D[q, j]!r}, {got_I[q, j]}), want ({D_ref[q, j]!r}, {I_ref[q, j]})")


def check_range_exact(lims, D, I, rows, xq, radius, metric, id_offset=0):
    """Lattice data: a range search result equals the float64 reference (tests/range_reference.py) exactly -- the same
    hits per query (strict: L2 dist < radius, IP ip > radius), ids ascending, identical distance values."""
    lims = np.asarray(lims).astype(np.int64)
    D, I = np.asarray(D), np.asarray(I) - id_offset
    rl, rD, rI = np_range_search_f64(rows, xq, radius, metric)
    assert lims[0] == 0 and np.all(np.diff(lims) >= 0) and lims[-1] == len(D) == len(I)
    for q in range(len(xq)):
        gi = I[lims[q]:lims[q + 1]]
        assert np.all(np.diff(gi) > 0), f"query {q}: ids not strictly ascending"
    if not np.array_equal(lims, rl):
        q = int(np.nonzero(lims != rl)[0][0]) - 1
        wi, gi = set(rI[rl[q]:rl[q + 1]].tolist()), set(I[lims[q]:lims[q + 1]].tolist())
        raise AssertionError(f"query {q}: {lims[q + 1] - lims[q]} hits, want {rl[q + 1] - rl[q]}; "
                             f"extra {sorted(gi - wi)[:5]}, missing {sorted(wi - gi)[:5]} (radius {radius!r})")
    assert np.array_equal(I, rI), "hit ids differ from the float64 reference"
    assert np.array_equal(D.astype(np.float64), rD), "hit distances differ from the float64 reference"
