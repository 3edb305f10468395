"""Result TREES (nested aggregates) in the oracle: oracle/tree_oracle.c against
  * the known answers of the reference's Merge offset iterator (RS/index_result/src/core/proximity.rs:409-470), and
  * the reference's own src/ext/default.c + src/index_result/index_result.c + src/offset_vector.c compiled in place
    (oracle/_ref/libscorers_ref.so, RefTree*; its answers recorded under tests/golden/reference/), on seeded random trees: bit-equal
    scores, equal offsets / GetSlop.
CPU only."""
import struct

import numpy as np
import pytest

import oracle_lib as ol
from oracle_lib import KIND_AND, KIND_NUMERIC, KIND_OR, KIND_TERM, KIND_VIRTUAL, ResultTree

def term(positions=(), freq=None, weight=1.0, idf=1.5, bm25_idf=0.7):
    return {"kind": KIND_TERM, "freq": len(positions) if freq is None else freq, "weight": weight, "idf": idf, "bm25_idf": bm25_idf,
            "positions": list(positions)}


def agg(kind, children, weight=1.0):
    return {"kind": kind, "weight": weight, "children": children}


def from_deltas(deltas):
    return np.cumsum(deltas).tolist()


# ---- proximity.rs:409-470 ----------------------------------------------------------------------
def test_merge_two_children_yields_sorted_order():
    t = ResultTree(agg(KIND_OR, [term(from_deltas([2, 3, 4])), term(from_deltas([1, 3, 3]))]))
    assert t.offsets() == [1, 2, 4, 5, 7, 9]


def test_merge_one_child_exhausts_early():
    t = ResultTree(agg(KIND_OR, [term(from_deltas([3])), term(from_deltas([6, 4]))]))
    assert t.offsets() == [3, 6, 10]


def test_merge_three_children_yields_sorted_order():
    t = ResultTree(agg(KIND_OR, [term(from_deltas([5])), term(from_deltas([2, 6])), term(from_deltas([1, 3]))]))
    assert t.offsets() == [1, 2, 4, 5, 8]


def test_merge_all_children_empty_returns_none():
    t = ResultTree(agg(KIND_OR, [term([], freq=1), term([], freq=1)]))
    assert t.offsets() == []
    # ... but the aggregate still COUNTS as having offsets (kind mask = Term): inside a slop query it rejects the document
    assert t.has_offsets()


def test_single_child_union_delegates_to_child_iter():
    t = ResultTree(agg(KIND_OR, [term(from_deltas([2, 3, 5]))]))
    assert t.offsets() == [2, 5, 10]


def test_duplicates_are_kept_and_nested_merges_compose():
    inner = agg(KIND_OR, [term([3, 9]), term([3, 7])])
    t = ResultTree(agg(KIND_AND, [inner, term([1, 3, 20])]))
    assert t.offsets(1) == [3, 3, 7, 9]
    assert t.offsets(0) == [1, 3, 3, 3, 7, 9, 20]


# ---- proximity over a tree: hand-checked ----------------------------------------------------------
def test_phrase_over_an_expansion():
    # "(run|running) fast": running at 4, fast at 5 -> exact phrase; run at 1 only -> slop 3 needed
    q = agg(KIND_AND, [agg(KIND_OR, [term([1]), term([4])]), term([5])])
    t = ResultTree(q)
    assert t.within_range(0, True) and t.within_range(0, False)
    q2 = agg(KIND_AND, [agg(KIND_OR, [term([1])]), term([5])])
    t2 = ResultTree(q2)
    assert not t2.within_range(2, True) and t2.within_range(3, True)
    # a union of terms indexed without positions counts as "has offsets" and then yields nothing: never in range
    q3 = agg(KIND_AND, [agg(KIND_OR, [term([], freq=2), term([], freq=1)]), term([5]), term([6])])
    assert not ResultTree(q3).within_range(10, False)
    # the same terms directly under the AND are skipped instead
    q4 = agg(KIND_AND, [term([], freq=2), term([5]), term([6])])
    assert ResultTree(q4).within_range(0, True)


def test_tree_equals_flat_when_unions_have_one_child():
    rng = np.random.default_rng(5)
    for _ in range(200):
        n = int(rng.integers(2, 5))
        pos = [sorted(set(rng.integers(1, 40, int(rng.integers(1, 6))).tolist())) for _ in range(n)]
        flat = [ol.varint_deltas(p) for p in pos]
        slop = None if rng.random() < 0.2 else int(rng.integers(0, 6))
        in_order = bool(rng.integers(0, 2)) or slop is None
        tree = ResultTree(agg(KIND_AND, [agg(KIND_OR, [term(p)]) for p in pos]))
        assert tree.within_range(slop, in_order) == bool(ol.within_range(flat, slop, in_order))


# ---- random trees against the reference's own code ---------------------------------------------------
def random_tree(rng, depth=0):
    def leaf():
        r = rng.random()
        if r < 0.70:
            npos = int(rng.integers(0, 6)) if rng.random() < 0.85 else 0
            p = sorted(set(rng.integers(1, 300, npos).tolist())) if npos else []
            if p and rng.random() < 0.3:
                p = sorted(set(p + rng.integers(300, 70_000, 2).tolist()))  # multi-byte varints
            return term(p, freq=max(1, len(p)) if rng.random() < 0.8 else int(rng.integers(1, 9)), weight=float(rng.choice([1.0, 0.5, 2.0, 0.3])),
                        idf=float(rng.uniform(0.1, 9.0)), bm25_idf=float(rng.uniform(0.01, 6.0)))
        if r < 0.85:
            return {"kind": KIND_VIRTUAL, "freq": int(rng.integers(0, 2)), "weight": float(rng.choice([0.0, 1.0, 0.7]))}
        return {"kind": KIND_NUMERIC, "freq": 1, "weight": float(rng.choice([1.0, 0.4]))}

    nk = int(rng.integers(1, 5))
    kids = []
    for _ in range(nk):
        if depth < 2 and rng.random() < 0.4:
            kids.append(random_tree(rng, depth + 1))
        else:
            kids.append(leaf())
    return agg(KIND_AND if rng.random() < 0.5 else KIND_OR, kids, weight=float(rng.choice([1.0, 1.0, 0.5, 3.0])))


def bits(x):
    return struct.pack("<d", x)


@pytest.mark.usefixtures("ref")
def test_offsets_has_offsets_and_get_slop_equal_the_reference():
    rng = np.random.default_rng(11)
    seen_nested = 0
    for _ in range(400):
        t = ResultTree(random_tree(rng))
        for node in range(len(t.nodes)):
            assert t.offsets(node) == t.ref_offsets(node)
            assert t.has_offsets(node) == t.ref_has_offsets(node)
        assert t.min_offset_delta() == t.ref_min_offset_delta()
        seen_nested += int((t.kind[1:] <= KIND_OR).any() and (t.kind[1:] >= KIND_AND).any())
    assert seen_nested > 100


@pytest.mark.usefixtures("ref")
def test_kind_mask_quirks_equal_the_reference():
    # an aggregate of numeric children only: mask = Numeric, which is neither Virtual nor exactly Numeric|Metric -> "has offsets"
    for kids in ([{"kind": KIND_NUMERIC, "freq": 1, "weight": 1.0}], [{"kind": KIND_VIRTUAL, "freq": 1, "weight": 1.0}],
                 [{"kind": KIND_VIRTUAL, "freq": 1, "weight": 1.0}, {"kind": KIND_NUMERIC, "freq": 1, "weight": 1.0}],
                 [term([], freq=1)], [agg(KIND_OR, [{"kind": KIND_VIRTUAL, "freq": 1, "weight": 1.0}])]):
        t = ResultTree(agg(KIND_AND, [agg(KIND_OR, kids), term([4, 9])]))
        assert t.has_offsets(1) == t.ref_has_offsets(1), kids
        assert t.min_offset_delta() == t.ref_min_offset_delta(), kids


@pytest.mark.usefixtures("ref")
@pytest.mark.parametrize("scorer", [ol.SCORER_BM25STD, ol.SCORER_BM25, ol.SCORER_TFIDF, ol.SCORER_TFIDF_DOCNORM, ol.SCORER_DOCSCORE,
                                    ol.SCORER_BM25STD_TANH, ol.SCORER_DISMAX])
def test_tree_scores_are_bit_equal_to_the_reference(scorer):
    rng = np.random.default_rng(100 + scorer)
    for i in range(300):
        t = ResultTree(random_tree(rng))
        doc_len, max_freq = int(rng.integers(0, 400)), int(rng.integers(0, 12))
        doc_score = float(np.float32(rng.choice([1.0, 0.5, 0.0, 2.5])))
        avg = float(rng.uniform(5.0, 300.0))
        min_score = float(rng.choice([0.0, 0.0, 0.05, 1.0]))
        a = t.score(scorer, doc_len, max_freq, doc_score, 10_000, avg, slop=-1, min_score=min_score, tanh_factor=4.0)
        b = t.ref_score(scorer, doc_len, max_freq, doc_score, 10_000, avg, slop=-1, min_score=min_score, tanh_factor=4)
        assert bits(a) == bits(b), (i, a, b)


# ---- EXPLAINSCORE: the PRODUCT's host-side explanation builder (libii_b200.so II_ExplainTree, no device) against the reference's
# scorers run with scrExp set (the EXPLAIN strings of src/ext/default.c, re-rooted by strExpCreateParent) ------------------------
def product_explain(t, scorer, doc_len, max_freq, doc_score, avg, slop, min_score, tanh_factor=4):
    import ctypes as C

    from redisearch_b200 import postings

    L = postings.lib()
    buf = C.create_string_buffer(1 << 16)
    sc = C.c_double(0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    L.II_ExplainTree(scorer, len(t.nodes), p(t.parent), p(t.kind), p(t.freq), p(t.weight), p(t.idf), p(t.bm25), b"t", doc_len, max_freq,
                     doc_score, avg, slop, min_score, tanh_factor, C.byref(sc), buf, len(buf))
    return sc.value, buf.value.decode()


@pytest.mark.usefixtures("ref")
@pytest.mark.parametrize("scorer", [ol.SCORER_BM25STD, ol.SCORER_BM25, ol.SCORER_TFIDF, ol.SCORER_TFIDF_DOCNORM, ol.SCORER_DOCSCORE,
                                    ol.SCORER_BM25STD_TANH, ol.SCORER_DISMAX])
def test_explainscore_strings_equal_the_reference(scorer):
    rng = np.random.default_rng(700 + scorer)
    shapes = set()
    for i in range(250):
        t = ResultTree(random_tree(rng))
        doc_len, max_freq = int(rng.integers(0, 400)), int(rng.integers(0, 12))
        doc_score = float(np.float32(rng.choice([1.0, 0.5, 0.0, 2.5])))
        avg = float(rng.uniform(5.0, 300.0))
        min_score = float(rng.choice([0.0, 0.0, 0.05, 1.0]))
        slop = t.min_offset_delta()
        ref_score, ref_text = t.ref_explain(scorer, doc_len, max_freq, doc_score, 10_000, avg, slop=slop, min_score=min_score)
        got_score, got_text = product_explain(t, scorer, doc_len, max_freq, doc_score, avg, slop, min_score)
        assert got_text == ref_text, (i, got_text, ref_text)
        assert bits(got_score) == bits(ref_score) or scorer == ol.SCORER_BM25STD_TANH and abs(got_score - ref_score) < 1e-15
        shapes.add(ref_text.count("\n"))
    assert len(shapes) >= 4 or scorer == ol.SCORER_DOCSCORE  # trees of several sizes, the early-out forms included


@pytest.mark.usefixtures("ref")
def test_wide_and_deep_trees_equal_the_reference():
    """up to 32 children per aggregate (the harness' and the device kernels' table size) and four levels of nesting: scores of every
    scorer bit-equal, offsets / GetSlop equal, explanations byte-equal"""
    rng = np.random.default_rng(4242)

    def wide(depth):
        nk = int(rng.integers(1, 33 if depth == 0 else 7))
        kids = []
        for _ in range(nk):
            if depth < 3 and rng.random() < 0.25:
                kids.append(wide(depth + 1))
            else:
                p = sorted(set(rng.integers(1, 2000, int(rng.integers(0, 5))).tolist()))
                kids.append(term(p, freq=max(1, len(p)), weight=float(rng.choice([1.0, 0.5])), idf=float(rng.uniform(0.1, 9.0)),
                                 bm25_idf=float(rng.uniform(0.01, 6.0))))
        return agg(KIND_AND if rng.random() < 0.5 else KIND_OR, kids, weight=float(rng.choice([1.0, 0.7, 2.0])))

    for i in range(60):
        t = ResultTree(wide(0))
        assert t.offsets(0) == t.ref_offsets(0)
        slop = t.min_offset_delta()
        assert slop == t.ref_min_offset_delta()
        for scorer in (ol.SCORER_BM25STD, ol.SCORER_BM25, ol.SCORER_TFIDF, ol.SCORER_TFIDF_DOCNORM, ol.SCORER_DISMAX):
            a = t.score(scorer, 120, 7, 1.0, 10_000, 88.5, slop=-1)
            b = t.ref_score(scorer, 120, 7, 1.0, 10_000, 88.5, slop=-1)
            assert bits(a) == bits(b), (i, scorer, a, b)
            assert product_explain(t, scorer, 120, 7, 1.0, 88.5, slop, 0.0)[1] == t.ref_explain(scorer, 120, 7, 1.0, 10_000, 88.5, slop=slop)[1]
