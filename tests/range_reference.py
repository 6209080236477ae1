"""float64 reference for range search, used by the range-search tests (CPU and GPU tiers).  TEST INFRASTRUCTURE ONLY."""
import numpy as np

from oracle import METRIC_L2


def np_range_search_f64(xb, xq, radius, metric=METRIC_L2, block=2048):
    """float64 brute-force range search with faiss's IndexFlat semantics: L2 hits have squared distance < radius, IP hits
    inner product > radius (strict; NaN is never a hit).  Returns (lims int64 [nq + 1], D float64, I int64), ids ascending
    within each query."""
    xb = np.asarray(xb, np.float64)
    xq = np.asarray(xq, np.float64)
    nq = xq.shape[0]
    Ds = [[] for _ in range(nq)]
    Is = [[] for _ in range(nq)]
    with np.errstate(all="ignore"):
        for j0 in range(0, xb.shape[0], block):
            xs = xb[j0:j0 + block]
            if metric == METRIC_L2:
                dist = (xq * xq).sum(1)[:, None] + (xs * xs).sum(1)[None, :] - 2.0 * (xq @ xs.T)
                # exact difference where the expansion cancels or is not finite
                redo = ~np.isfinite(dist) | (dist < 1e-6 * ((xq * xq).sum(1)[:, None] + 1e-300))
                if redo.any():
                    qi, xi = np.nonzero(redo)
                    dist[qi, xi] = ((xq[qi] - xs[xi]) ** 2).sum(1)
                hit = dist < radius
            else:
                dist = xq @ xs.T
                hit = dist > radius
            for q in range(nq):
                sel = np.nonzero(hit[q])[0]
                Ds[q].append(dist[q, sel])
                Is[q].append(sel.astype(np.int64) + j0)
    lims = np.zeros(nq + 1, np.int64)
    for q in range(nq):
        lims[q + 1] = lims[q] + sum(len(a) for a in Is[q])
    D = np.concatenate([np.concatenate(a) if a else np.empty(0) for a in Ds]) if nq else np.empty(0)
    I = np.concatenate([np.concatenate(a) if a else np.empty(0, np.int64) for a in Is]) if nq else np.empty(0, np.int64)
    return lims, D.astype(np.float64), I.astype(np.int64)
