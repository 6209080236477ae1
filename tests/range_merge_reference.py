"""numpy restatement of b2f_merge_range_strided and a sort-based union to check it against (CPU and GPU tiers).
TEST INFRASTRUCTURE ONLY."""
import numpy as np

LABEL_BITS = 40   # the restatement's composite (query, label) keys hold labels below 2^40


def _query_of(rel_p):
    """query of every element of one part, from its lims rebased to 0"""
    return np.searchsorted(rel_p, np.arange(rel_p[-1]), side="right") - 1


def np_merge_range(lims_parts, D_parts, I_parts):
    """What the kernel computes: lims_parts [G, nq + 1] int64 (any base), D_parts / I_parts: each part's hits.  Every hit
    goes to its query's output base + its index in its own list + the labels below it in every other part's list of
    that query (a lower_bound per part).  Returns (lims [nq + 1] from 0, D, I)."""
    lims = np.asarray(lims_parts, np.int64)
    rel = lims - lims[:, :1]
    out_base = rel.sum(0)
    total = int(out_base[-1])
    D = np.full(total, np.nan, np.float32)
    I = np.full(total, -1, np.int64)
    qs = [_query_of(r) for r in rel]
    keys = [(q << LABEL_BITS) | np.asarray(i, np.int64) for q, i in zip(qs, I_parts)]   # sorted: query, then label
    for p in range(len(rel)):
        e = np.arange(rel[p, -1])
        if not len(e):
            continue
        q = qs[p]
        pos = out_base[q] + e - rel[p, q]
        for r in range(len(rel)):
            if r != p:
                pos += np.searchsorted(keys[r], keys[p], side="left") - rel[r, q]
        D[pos] = D_parts[p]
        I[pos] = I_parts[p]
    return out_base, D, I


def np_union_range(lims_parts, D_parts, I_parts):
    """The same result by sorting: every part's hits tagged with their query, ordered by (query, label)."""
    lims = np.asarray(lims_parts, np.int64)
    rel = lims - lims[:, :1]
    q = np.concatenate([_query_of(r) for r in rel])
    D = np.concatenate([np.asarray(d, np.float32) for d in D_parts])
    I = np.concatenate([np.asarray(i, np.int64) for i in I_parts])
    order = np.lexsort((I, q))
    return rel.sum(0), D[order], I[order]


def split_packed(lims_parts, buf, part_bytes, off_i):
    """The parts of a packed all-gather buffer (uint8 [G * part_bytes], part g = [D fp32 | pad | I int64 at off_i])."""
    lims = np.asarray(lims_parts, np.int64)
    n = lims[:, -1] - lims[:, 0]
    D = [buf[g * part_bytes: g * part_bytes + 4 * n[g]].view(np.float32) for g in range(len(n))]
    I = [buf[g * part_bytes + off_i: g * part_bytes + off_i + 8 * n[g]].view(np.int64) for g in range(len(n))]
    return D, I


def np_range_merge_fn(lims_parts, recv, part_bytes, off_i, D, I):
    """ShardedIndexFlat(range_merge_fn=...) stand-in for the CUDA merge: the restatement over host tensors."""
    lims = lims_parts.numpy()
    Dp, Ip = split_packed(lims, recv.numpy(), part_bytes, off_i)
    _, Dm, Im = np_merge_range(lims, Dp, Ip)
    D.numpy()[:] = Dm
    I.numpy()[:] = Im


def random_parts(rng, nparts, nq, max_hits, empty_parts=(), empty_queries=(), big=None, base_max=1000):
    """nparts label-disjoint range results over nq queries: per query a random set of labels dealt to random parts,
    ascending within each part and query.  Parts in empty_parts and queries in empty_queries get no hits; big = (query,
    hits) gives one query that many hits.  Every part's lims start at a random base.  Returns (lims [G, nq + 1], D, I)."""
    counts = rng.integers(0, max_hits + 1, nq)
    if big is not None:
        counts[big[0]] = big[1]
    counts[list(empty_queries)] = 0
    owners = [[] for _ in range(nparts)]
    live = np.array([p for p in range(nparts) if p not in set(empty_parts)], np.int64)
    for q in range(nq):
        labels = np.sort(rng.choice(1 << 30, counts[q], replace=False)) if counts[q] else np.zeros(0, np.int64)
        own = rng.choice(live, counts[q]) if len(live) else np.zeros(0, np.int64)
        for p in range(nparts):
            owners[p].append(labels[own == p])
    lims = np.zeros((nparts, nq + 1), np.int64)
    D, I = [], []
    for p in range(nparts):
        sizes = np.array([len(a) for a in owners[p]], np.int64)
        lims[p] = int(rng.integers(0, base_max + 1)) + np.concatenate([[0], np.cumsum(sizes)])
        I.append(np.concatenate(owners[p]).astype(np.int64) if nq else np.zeros(0, np.int64))
        D.append(rng.standard_normal(len(I[-1])).astype(np.float32))
    return lims, D, I
