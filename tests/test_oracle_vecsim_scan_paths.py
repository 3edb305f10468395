"""Pins oracle/vecsim_oracle.c to the reference on the queries that do not go through the fused top-k scan: range queries,
batch iterators drained to the end, top-k with k > 128, and every query of a multi-value index (best score per label), for all
5 vector types x 3 metrics.  The reference's answers are recorded under tests/golden/reference/ (the `ref` fixture).  CPU only.

Where the reference leaves an order unspecified, both sides are put in (score, label) order before they are compared:
  * BY_SCORE replies of range queries and select-based batches are std::sort by score alone (vec_utils.cpp:105-109), so the
    order of equal scores is whatever introsort leaves;
  * a batch whose last place falls inside a group of equal scores takes an arbitrary part of that group (std::nth_element,
    bf_batch_iterator.h:143-166), so a label tied with a batch's first or last score may come one batch earlier or later.
The top-k heap is order-dependent at the k-th boundary (strict `<` admission, brute_force.h:271-279; a multi-value index
keeps one entry per label, updatable_heap.h:92-111).  The tie groups below are laid out in ascending label order at the front
of the index and are never moved by a swap-delete, which makes the heap's choice the (score, label) one the oracle makes.
"""
import os

import numpy as np
import pytest

import oracle_lib as ol
from oracle_lib import BF16, COS, F16, F32, I8, IP, L2, TIER_AVX512, U8

TYPES = [F32, F16, BF16, I8, U8]
METRICS = [L2, IP, COS]
CASES = [(t, m) for t in TYPES for m in METRICS]
DIMS = [7, 17, 33]


def _exact(vtype):
    return vtype in (F32, I8, U8)


def _tol(s):
    """fp16 / bf16: the port accumulates in fp32 in another order than the reference's fp32-accumulating tiers"""
    return 2e-4 * np.maximum(np.abs(s), 1.0)


class _HalfTier:
    """fp16 distances by the reference's fp32-accumulating tiers (the AVX512-FP16 tier accumulates in fp16, SURVEY.md §0)"""

    def __init__(self, vtype):
        self.on = vtype in (F16, BF16)

    def __enter__(self):
        if self.on:
            os.environ["REF_CPU_MASK"] = "avx512_fp16"

    def __exit__(self, *a):
        os.environ.pop("REF_CPU_MASK", None)


def _canon(ids, scores):
    """(score, label) order"""
    ids, scores = np.asarray(ids, dtype=np.int64), np.asarray(scores, dtype=np.float64)
    o = np.lexsort((ids, scores))
    return ids[o], scores[o]


def _stored_query(p, q):
    """the query as the index stores it (normalised for cosine; int8/uint8 with the norm slot) for distance_from"""
    size = p.L.orc_stored_size(p.vtype, p.dim, p.metric)
    buf = np.zeros(size, dtype=np.uint8)
    buf[: q.nbytes] = np.ascontiguousarray(q).view(np.uint8)
    if p.metric == COS:
        p.L.orc_normalize(ol._p(buf), p.dim, p.vtype)
    return buf


def assert_same_list(vtype, ref, port, complete, what=""):
    """Two score-ordered replies.  Exact types: the same (score, label) sequence, score bits equal.  fp16 / bf16: scores within
    the tolerance position by position, and every label on one side only lies within the tolerance of the last score (or, with
    `complete`, the label sets are equal)."""
    ri, rs = _canon(*ref)
    pi, ps = _canon(*port)
    assert len(ri) == len(pi), (what, len(ri), len(pi))
    if _exact(vtype):
        assert ri.tolist() == pi.tolist(), what
        assert rs.astype(np.float32).tobytes() == ps.astype(np.float32).tobytes(), what
        return
    assert np.all(np.abs(rs - ps) <= _tol(rs)), (what, np.max(np.abs(rs - ps)))
    rmap, pmap = dict(zip(ri.tolist(), rs.tolist())), dict(zip(pi.tolist(), ps.tolist()))
    for lab in set(rmap) & set(pmap):
        assert abs(rmap[lab] - pmap[lab]) <= _tol(rmap[lab]), (what, lab)
    only = set(rmap) ^ set(pmap)
    assert not (complete and only), (what, sorted(only)[:10])
    if only:
        cut = max(rs[-1], ps[-1])
        for lab in only:
            s = rmap.get(lab, pmap.get(lab))
            assert abs(s - cut) <= 2 * _tol(cut), (what, lab, s, cut)


def check_range(vtype, r, p, q, radius, order, all_dist):
    ri, rs = r.range(q, radius, order)
    pi, ps = p.range(q, radius, order)
    if order == 1:
        assert pi.tolist() == sorted(pi.tolist())
        assert ri.tolist() == sorted(ri.tolist())
    if _exact(vtype):
        assert_same_list(vtype, (ri, rs), (pi, ps), True, ("range", radius, order))
        return
    # fp16 / bf16: only labels farther than the tolerance from the radius must agree
    rmap, pmap = dict(zip(ri.tolist(), rs.tolist())), dict(zip(pi.tolist(), ps.tolist()))
    for lab in set(rmap) ^ set(pmap):
        assert abs(all_dist[lab] - radius) <= 2 * _tol(radius), ("range", radius, lab, all_dist[lab])
    for lab in set(rmap) & set(pmap):
        assert abs(rmap[lab] - pmap[lab]) <= _tol(rmap[lab])


def check_batches(vtype, r, p, q, size, order):
    """Drain the reference's batch iterator `size` at a time against the oracle's all-labels order cut into batches."""
    got = r.batches(q, size, order)
    ai, as_ = p.all_sorted(q)
    want = [(ai[i:i + size], as_[i:i + size]) for i in range(0, len(ai), size)]
    assert [len(b[0]) for b in got] == [len(b[0]) for b in want], ("batch sizes", size)
    seen = []
    for bi, ((gi, gs), (wi, ws)) in enumerate(zip(got, want)):
        if order == 1:
            assert gi.tolist() == sorted(gi.tolist())
        gi, gs = _canon(gi, gs)
        if _exact(vtype):
            assert gs.astype(np.float32).tobytes() == ws.astype(np.float32).tobytes(), ("batch", size, bi)
            inner = (ws > ws[0]) & (ws < ws[-1])  # a label tied with the batch's first or last score may change batch
            assert set(gi[(gs > gs[0]) & (gs < gs[-1])].tolist()) == set(wi[inner].tolist()), ("batch", size, bi)
        else:
            assert np.all(np.abs(gs - ws) <= _tol(ws)), ("batch", size, bi)
        seen += gi.tolist()
    assert len(seen) == len(set(seen)) == len(ai)
    assert set(seen) == set(ai.tolist())


def _rows(rng, vtype, n, dim, scale=1.0):
    return ol.to_type(rng.uniform(-scale, scale, (n, dim)).astype(np.float32), vtype)


def _radii(ds):
    """from the oracle's sorted distances: 0, an observed distance exactly (included: the test is `<=`), the float just below it
    (excluded), a double that rounds to it (both sides cast the radius to float), one far inside the set, 1e9"""
    d = np.float32(ds[len(ds) // 3])
    below = float(np.nextafter(d, np.float32(-np.inf)))
    near = float(d) + float(np.spacing(d)) * 0.25
    assert np.float32(near) == d
    return [0.0, float(d), below, near, float(np.float32(ds[(2 * len(ds)) // 3])), 1e9]


# ------------------------------------------------------------------ single-value
@pytest.mark.parametrize("vtype,metric", CASES)
def test_single_value_scan_paths_match_reference(oracle, ref, vtype, metric):
    """range at several radii in both orders, batch iterators drained at several sizes and in both orders, top-k with
    k in {129, 300, n, n+1}, on a single-value index with a group of 40 identical rows and a few swap-deletes."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(500 + ci)
    n, dim = 600, DIMS[ci % 3]
    x = _rows(rng, vtype, n, dim, 1.0 if metric != IP else 1.7)
    x[200:240] = x[37]  # identical rows, labels ascending in row order: score ties
    with _HalfTier(vtype):
        r = ol.RefIndex(vtype, dim, metric)
        p = ol.PortIndex(vtype, dim, metric, tier=TIER_AVX512)
        r.add_many(x, 1)
        p.add_many(x, 1)
        for lab in (590, 300, 451):  # swap-deletes outside the tie group
            assert r.delete(lab) == p.delete(lab) == 1
        assert r.size() == p.size() == n - 3
        for qi in range(2):
            q = _rows(rng, vtype, 1, dim)[0] if qi == 0 else x[37].copy()
            ai, as_ = p.all_sorted(q)
            all_dist = dict(zip(ai.tolist(), as_.tolist()))
            for radius in _radii(as_):
                for order in (0, 1):
                    check_range(vtype, r, p, q, radius, order, all_dist)
            for size, order in ((1, 0), (7, 1), (128, 0), (129, 0), (500, 0)):
                if size == 1 and qi == 1:
                    continue
                check_batches(vtype, r, p, q, size, order)
            for k in (129, 300, n - 3, n - 2):
                assert_same_list(vtype, r.topk(q, k), p.topk(q, k), k >= n - 3, ("topk", k))
            ri, _ = r.topk(q, 300, 1)
            pi, _ = p.topk(q, 300, 1)
            assert ri.tolist() == sorted(ri.tolist()) and pi.tolist() == sorted(pi.tolist())
            if _exact(vtype):
                assert ri.tolist() == pi.tolist()


# ------------------------------------------------------------------ multi-value
def _multi_layout(rng, vtype, dim, metric):
    """[(blob, label)] of a multi-value index: labels 1..30 are tie groups at the front (1-5 copies of one of two vectors, labels
    ascending in row order), then labels 31..229 with 1-5 rows each in shuffled row order, some rows shared across labels."""
    scale = 1.0 if metric != IP else 1.7
    base = _rows(rng, vtype, 2, dim, scale)
    out = []
    for lab in range(1, 31):
        out += [(base[lab % 2], lab)] * int(rng.integers(1, 6))
    rest = []
    for lab in range(31, 230):
        rest += [(v, lab) for v in _rows(rng, vtype, int(rng.integers(1, 6)), dim, scale)]
    for j in range(0, 40, 4):  # the same vector under two labels
        rest[j + 1] = (rest[j][0].copy(), rest[j + 1][1])
    order = rng.permutation(len(rest))
    return out + [rest[i] for i in order], base


@pytest.mark.parametrize("vtype,metric", CASES)
def test_multi_value_index_matches_reference(oracle, ref, vtype, metric):
    """A multi-value index (labels with 1-5 vectors, identical vectors inside a label and across labels) before and after
    deletes of multi-vector labels (whose swap-deletes move other labels' rows) and re-adds: top-k at
    k in {1, 10, 129, label_count, label_count+1}, range, batch iterators drained to the end, distance_from (min over the label's
    rows)."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(900 + ci)
    dim = DIMS[(ci + 1) % 3]
    rows, base = _multi_layout(rng, vtype, dim, metric)
    with _HalfTier(vtype):
        r = ol.RefIndex(vtype, dim, metric, multi=True)
        p = ol.PortIndex(vtype, dim, metric, multi=True, tier=TIER_AVX512)
        for blob, lab in rows:
            assert r.add(blob, lab) == p.add(blob, lab) == 1
        labels = sorted({lab for _, lab in rows})
        counts = {lab: sum(1 for _, l2 in rows if l2 == lab) for lab in labels}
        multi_labels = [lab for lab in labels if lab > 30 and counts[lab] > 1]
        queries = [_rows(rng, vtype, 1, dim)[0], base[0].copy()]
        for phase in range(2):
            assert r.size() == p.size()
            nl = len(labels)
            for q in queries:
                for k in (1, 10, 129, nl, nl + 1):
                    assert_same_list(vtype, r.topk(q, k), p.topk(q, k), k >= nl, ("topk", phase, k))
                ai, as_ = p.all_sorted(q)
                assert len(ai) == nl
                all_dist = dict(zip(ai.tolist(), as_.tolist()))
                for radius in _radii(as_):
                    for order in (0, 1):
                        check_range(vtype, r, p, q, radius, order, all_dist)
                for size, order in ((7, 0), (64, 1), (129, 0)):
                    check_batches(vtype, r, p, q, size, order)
                sq = _stored_query(p, q)
                for lab in labels[::7] + [labels[-1], 10**6]:
                    a, b = r.distance_from(lab, sq), p.distance_from(lab, sq)
                    if np.isnan(a) or np.isnan(b):
                        assert np.isnan(a) and np.isnan(b), lab
                    elif _exact(vtype):
                        assert np.float32(a).tobytes() == np.float32(b).tobytes(), lab
                    else:
                        assert abs(a - b) <= _tol(a), lab
            if phase == 0:
                # delete multi-vector labels (their rows are all over the index), then re-add some with fewer / more rows
                victims = [int(v) for v in rng.choice(multi_labels, 25, replace=False)]
                for lab in victims:
                    assert r.delete(lab) == p.delete(lab) == counts[lab]
                assert r.delete(10**6) == p.delete(10**6) == 0
                labels = [lab for lab in labels if lab not in victims]
                for lab in victims[:10] + [400, 401]:
                    c = int(rng.integers(1, 4))
                    for v in _rows(rng, vtype, c, dim):
                        assert r.add(v, lab) == p.add(v, lab) == 1
                    labels.append(lab)
                    counts[lab] = c
                labels.sort()


@pytest.mark.parametrize("vtype", TYPES)
def test_multi_value_distance_from_nan_rule(oracle, ref, vtype):
    """getDistanceFrom on a multi-value index folds `dist = (dist < d) ? dist : d` from +inf over the label's rows in
    insertion order (brute_force_multi.h:234-238): a NaN row makes the running value NaN and the next row replaces it, so the
    answer is NaN exactly when the label's LAST row is NaN against the query.  A cosine row of zeros is NaN against every
    query (0/0 in the normaliser, or the int8/uint8 norm slot being 0)."""
    dim = 9
    rng = np.random.default_rng(40 + vtype)
    a, b = _rows(rng, vtype, 2, dim)
    z = np.zeros(dim, dtype=ol.NP_DTYPE[vtype])
    if vtype == U8:
        z[:] = 0
    layouts = {1: [a, z], 2: [z, a], 3: [a, z, b], 4: [z, z], 5: [z], 6: [b, a], 7: [z, b, z, a]}
    with _HalfTier(vtype):
        r = ol.RefIndex(vtype, dim, COS, multi=True)
        p = ol.PortIndex(vtype, dim, COS, multi=True, tier=TIER_AVX512)
        for lab, vs in layouts.items():
            for v in vs:
                assert r.add(v, lab) == p.add(v, lab) == 1
        sq = _stored_query(p, _rows(rng, vtype, 1, dim)[0])
        got = {}
        for lab in list(layouts) + [99]:
            x, y = r.distance_from(lab, sq), p.distance_from(lab, sq)
            got[lab] = np.isnan(x)
            assert np.isnan(x) == np.isnan(y), (lab, x, y)
            if not np.isnan(x):
                assert abs(x - y) <= (0 if _exact(vtype) else _tol(x)), (lab, x, y)
        assert got == {1: True, 2: False, 3: False, 4: True, 5: True, 6: False, 7: False, 99: True}
