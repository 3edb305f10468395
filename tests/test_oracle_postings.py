"""Pins oracle/postings_oracle.c and oracle/scorer_oracle.c to the reference.

The posting path of the reference is Rust and cannot be built here (no toolchain), so the restatement
is pinned by the reference's OWN golden vectors and known answers (tests/golden/postings_golden.json,
each entry citing its source file:line).  The scorers are C: oracle/_ref/libscorers_ref.so IS the
reference's src/ext/default.c, and the restatement must agree with it bit for bit.  CPU only.
"""
import ctypes as C
import json
import math
import os

import numpy as np
import pytest

import oracle_lib as ol

G = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "postings_golden.json")))


@pytest.fixture(scope="module")
def L():
    return ol.postings()


def _qint(L, vals):
    arr = (C.c_uint32 * len(vals))(*vals)
    out = (C.c_uint8 * 32)()
    n = L.orc_qint_encode(arr, len(vals), out)
    back = (C.c_uint32 * len(vals))()
    m = L.orc_qint_decode(out, len(vals), back)
    assert m == n and list(back) == list(vals)
    return bytes(out[:n])


def test_qint_known_lengths_and_roundtrip(L):
    for case in G["qint_lengths"]:
        assert len(_qint(L, case["values"])) == case["bytes"]
    rng = np.random.default_rng(0)
    for _ in range(500):
        n = int(rng.integers(2, 5))
        vals = [int(rng.integers(0, 2 ** int(rng.integers(1, 33)))) for _ in range(n)]
        _qint(L, vals)


def test_varint_golden_bytes(L):
    for value, expected in G["varint_bytes"]:
        out = (C.c_uint8 * 16)()
        n = L.orc_varint_encode(value, out)
        assert list(out[:n]) == expected, value
        v = C.c_uint64()
        assert L.orc_varint_decode(out, C.byref(v)) == n and v.value == value
    for value, ln in G["varint_lengths"]:
        out = (C.c_uint8 * 16)()
        assert L.orc_varint_encode(value, out) == ln


def _single_record_bytes(codec, delta, freq, mask, offsets=b""):
    """Encode one record whose delta from the block's first entry is `delta` and return its bytes."""
    base = 1 << 32  # the reference tests use doc_id = 4294967296 and prev = doc_id - delta
    ix = ol.InvIndex(codec)
    ix.add(base, 7, 1, b"\1")
    first_len = len(ix.blocks()[0][3])
    grew = ix.add(base + delta, freq, mask, offsets) if delta else None
    if delta == 0:
        # delta 0 can only be the first record of a block: encode it as such
        ix = ol.InvIndex(codec)
        ix.add(base, freq, mask, offsets)
        return ix.blocks()[0][3]
    blocks = ix.blocks()
    assert len(blocks) == 1 and grew == len(blocks[0][3]) - first_len
    return blocks[0][3][first_len:]


def test_codec_golden_bytes():
    for freq, delta, expected in G["freqs_only"]:
        assert list(_single_record_bytes(ol.CODEC_FREQS_ONLY, delta, freq, 1)) == expected
    for delta, freq, mask, offs, expected in G["full"]:
        assert list(_single_record_bytes(ol.CODEC_FULL, delta, freq, mask, bytes(offs))) == expected
    for delta, freq, mask, expected in G["freqs_fields"]:
        assert list(_single_record_bytes(ol.CODEC_FREQS_FIELDS, delta, freq, mask)) == expected
    for delta, mask, expected in G["fields_only"]:
        assert list(_single_record_bytes(ol.CODEC_FIELDS_ONLY, delta, 1, mask)) == expected
    for delta, expected in G["doc_ids_only"]:
        assert list(_single_record_bytes(ol.CODEC_DOCIDS_ONLY, delta, 1, 1)) == expected
    for delta, expected in G["raw_doc_ids_only"]:
        assert list(_single_record_bytes(ol.CODEC_RAW_DOCIDS_ONLY, delta, 1, 1)) == expected
    # the codecs that carry term offsets without the full record, and the u128 field-mask (*Wide) variants
    for delta, freq, offs, expected in G["freqs_offsets"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FREQS_OFFSETS, delta, freq, 1, bytes(offs))) == expected
    for delta, offs, expected in G["offsets_only"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_OFFSETS_ONLY, delta, 1, 1, bytes(offs))) == expected
    for delta, mask, offs, expected in G["fields_offsets"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FIELDS_OFFSETS, delta, 1, mask, bytes(offs))) == expected
    for delta, mask, offs, expected in G["fields_offsets_wide"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FIELDS_OFFSETS_WIDE, delta, 1, int(mask), bytes(offs))) == expected
    for delta, freq, mask, offs, expected in G["full_wide"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FULL_WIDE, delta, freq, int(mask), bytes(offs))) == expected
    for delta, freq, mask, expected in G["freqs_fields_wide"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FREQS_FIELDS_WIDE, delta, freq, int(mask))) == expected
    for delta, mask, expected in G["fields_only_wide"]["cases"]:
        assert list(_single_record_bytes(ol.CODEC_FIELDS_ONLY_WIDE, delta, 1, int(mask))) == expected


@pytest.mark.parametrize("codec", range(ol.N_CODECS))
def test_blocks_and_reader_roundtrip(codec):
    """index/core.rs:235-358 + reader/core.rs: 100 (1000) entries per block, first record delta 0,
    a delta that overflows u32 opens a new block, repeated docIds are dropped."""
    rng = np.random.default_rng(codec)
    ids = np.cumsum(rng.integers(1, 50, 2500)).astype(np.uint64)
    ids[1200:] += np.uint64(1 << 33)  # force a >u32 delta
    freqs = rng.integers(1, 300, len(ids))
    masks = rng.integers(1, 1 << 20, len(ids)).tolist()
    if codec in ol.CODECS_WIDE:  # field masks beyond 32 / 64 bits
        masks = [m << int(s_) for m, s_ in zip(masks, rng.integers(0, 100, len(ids)))]
    ix = ol.InvIndex(codec)
    for i, d in enumerate(ids.tolist()):
        ob = bytes(rng.integers(1, 100, int(rng.integers(0, 4)), dtype=np.uint8).tolist()) if codec in ol.CODECS_WITH_OFFSETS else b""
        ix.add(d, int(freqs[i]), masks[i], ob)
    assert ix.add(int(ids[-1]), 5, 5) == 0  # duplicate docId silently skipped
    per = 1000 if codec in (ol.CODEC_DOCIDS_ONLY, ol.CODEC_RAW_DOCIDS_ONLY) else 100
    blocks = ix.blocks()
    assert all(b[2] <= per for b in blocks)
    if codec != ol.CODEC_RAW_DOCIDS_ONLY:
        assert any(b[0] == int(ids[1200]) for b in blocks)  # the overflow opened a block at that doc
    got = ix.read_all()
    assert [g[0] for g in got] == ids.tolist()
    if codec in ol.CODECS_WITH_FREQ:
        assert [g[1] for g in got] == freqs.tolist()
    else:
        assert all(g[1] == 1 for g in got)
    if codec in ol.CODECS_WITH_MASK:
        assert [g[2] for g in got] == masks
        # FilterMaskReader (reader/field_mask.rs) over the wide masks too
        flt = (1 << 3) | (1 << 70)
        assert [g[0] for g in ix.read_all(flt)] == [int(d) for d, m_ in zip(ids.tolist(), masks) if m_ & flt]
    # seek: first record >= target, from the start and monotonically
    L = ol.postings()
    r = ix.reader()
    d, f, m = C.c_uint64(), C.c_uint32(), C.c_uint32()
    pos = 0
    for t in sorted(rng.choice(int(ids[-1]) + 10, 200, replace=False).tolist()):
        if pos < len(ids) and t <= int(ids[pos - 1] if pos else 0):
            continue
        ok = L.orc_reader_seek(r, t, C.byref(d), C.byref(f), C.byref(m))
        j = int(np.searchsorted(ids, t))
        if j >= len(ids):
            assert not ok
            break
        assert ok and d.value == int(ids[j])
        pos = j + 1
    L.orc_reader_free(r)


def _children_for(result_set, num_children):
    nxt = 1
    out = []
    for _ in range(num_children):
        ids = set(result_set)
        # unique ids must not collide with the result set (the Rust fixture relies on dedup of equal ids only)
        added = 0
        while added < 100:
            ids.add(nxt)
            nxt += 1
            added += 1
        out.append(sorted(ids))
    return out


def _expected_intersection(children):
    s = set(children[0])
    for c in children[1:]:
        s &= set(c)
    return sorted(s)


@pytest.mark.parametrize("num_children", G["intersection_num_children"][:2] + [16])
@pytest.mark.parametrize("case", range(3))
def test_intersection_read_and_skipto_cases(num_children, case):
    """rqe_iterators/tests/integration/intersection.rs:59-273 (read_all_combinations, skip_to_all_combinations)."""
    L = ol.postings()
    rs = G["intersection_result_sets"][case]
    children = _children_for(rs, num_children)
    expected = _expected_intersection(children)
    idx = [ol.InvIndex(ol.CODEC_FREQS_ONLY, c, [1] * len(c)) for c in children]
    hits = ol.run_intersect(idx)
    assert [h[0] for h in hits] == expected
    assert all(len(h[1]) == num_children for h in hits)
    # skip_to(i) from a rewound iterator lands on the first result >= i
    for i in range(1, expected[-1] + 2, max(1, expected[-1] // 300)):
        readers = [ix.reader() for ix in idx]
        arr = (C.c_void_p * len(readers))(*readers)
        t = (C.c_uint64 * 1)(i)
        st = (C.c_int * 1)()
        landed = (C.c_uint64 * 1)()
        L.orc_intersect_skipto(arr, len(readers), t, 1, st, landed)
        nxt = [e for e in expected if e >= i]
        if not nxt:
            assert st[0] == 2
        else:
            assert landed[0] == nxt[0] and st[0] == (0 if nxt[0] == i else 1)
        for r in readers:
            L.orc_reader_free(r)


def test_cpp_intersection_known_answer():
    """tests/cpptests/test_cpp_index.cpp:542-601."""
    g = G["cpp_intersection"]
    a = np.arange(1, g["size"] + 1) * g["steps"][0]
    b = np.arange(1, g["size"] + 1) * g["steps"][1]
    ia = ol.InvIndex(ol.CODEC_FULL, a, [1] * len(a), [1] * len(a))
    ib = ol.InvIndex(ol.CODEC_FULL, b, [1] * len(b), [1] * len(b))
    hits = ol.run_intersect([ia, ib])
    assert len(hits) == g["hits"]
    for count, (doc, ch) in enumerate(hits):
        assert doc == (count * 2 + 2) * 2
        assert sum(f for _, f in ch) == g["freq"]
    L = ol.postings()
    readers = [ia.reader(), ib.reader()]
    arr = (C.c_void_p * 2)(*readers)
    t = (C.c_uint64 * 3)(8, 12, 200000)
    st = (C.c_int * 3)()
    landed = (C.c_uint64 * 3)()
    L.orc_intersect_skipto(arr, 2, t, 3, st, landed)
    assert list(st) == [0, 0, 0] and list(landed) == [8, 12, 200000]


@pytest.mark.parametrize("quick", [False, True])
def test_union_full_and_quick(quick):
    """union_flat.rs:218-524: every docId present in any child, ascending; full mode aggregates all
    children positioned on it, quick mode reports one."""
    rng = np.random.default_rng(11)
    lists = [np.unique(rng.integers(1, 5000, n)) for n in (50, 400, 1500, 7)]
    idx = [ol.InvIndex(ol.CODEC_FREQS_ONLY, l, rng.integers(1, 9, len(l))) for l in lists]
    hits = ol.run_intersect(idx, union=True, quick=quick)
    expected = sorted(set().union(*[set(l.tolist()) for l in lists]))
    assert [h[0] for h in hits] == expected
    for doc, ch in hits:
        present = {i for i, l in enumerate(lists) if doc in set(l.tolist())}
        if quick:
            assert len(ch) == 1 and ch[0][0] in present
        else:
            assert {c for c, _ in ch} == present


def test_idf_known_answers(L):
    for total, term, expected in G["idf"]:
        assert L.orc_idf(total, term) == expected
    for total, term, expected, eps in G["idf_bm25"]:
        assert abs(L.orc_idf_bm25(total, term) - expected) <= eps
    assert L.orc_idf(100, 0) == L.orc_idf(100, 1)
    assert L.orc_idf_bm25(5, 10) == L.orc_idf_bm25(10, 10)


# ------------------------------------------------------------------ scorers
def test_bm25std_golden_explainscore(L):
    """tests/pytests/test_scorers.py:198-221."""
    g = G["bm25std_explain"]
    idf = L.orc_idf_bm25(g["num_docs"], g["term_docs"])
    assert f"{idf:.2f}" == "0.13"
    for doc_len, total, leaf in g["cases"]:
        s = ol.oracle_score(ol.SCORER_BM25STD, [g["freq"]] * 2, [0, 0], [idf, idf], [1.0, 1.0], 1.0, doc_len, 10, 1.0,
                            g["num_docs"], g["avg_doc_len"])
        assert f"{s:.2f}" == f"{total:.2f}"
        s1 = ol.oracle_score(ol.SCORER_BM25STD, [g["freq"]], [0], [idf], [1.0], 1.0, doc_len, 10, 1.0, g["num_docs"], g["avg_doc_len"])
        assert f"{s1:.2f}" == f"{leaf:.2f}"


def test_bm25_legacy_golden_explainscore():
    """tests/pytests/test_scorers.py:159-178."""
    g = G["bm25_explain"]
    for doc_score, slop in g["cases"]:
        s = ol.oracle_score(ol.SCORER_BM25, [g["freq"]] * 2, [g["idf"]] * 2, [0, 0], [1.0, 1.0], 1.0, 10, 10, doc_score, 3,
                            g["avg_doc_len"], slop=slop)
        words = s * slop / doc_score
        assert f"{words:.2f}" == f"{g['words_bm25']:.2f}"


@pytest.mark.parametrize("scorer", [ol.SCORER_BM25STD, ol.SCORER_BM25, ol.SCORER_TFIDF, ol.SCORER_TFIDF_DOCNORM,
                                    ol.SCORER_DOCSCORE, ol.SCORER_BM25STD_TANH, ol.SCORER_DISMAX])
def test_scorers_bit_equal_to_reference_default_c(ref, scorer):
    """oracle/_ref/libscorers_ref.so is the reference's own src/ext/default.c."""
    rng = np.random.default_rng(100 + scorer)
    for _ in range(300):
        n = int(rng.integers(1, 7))
        freqs = rng.integers(1, 60, n).tolist()
        num_docs = int(rng.integers(n, 10**7))
        dfs = rng.integers(1, num_docs + 1, n)
        idf = [ol.postings().orc_idf(num_docs, int(d)) for d in dfs]
        bidf = [ol.postings().orc_idf_bm25(num_docs, int(d)) for d in dfs]
        weights = rng.choice([1.0, 0.5, 0.3, 2.0, 1.7], n).tolist()
        aggw = float(rng.choice([1.0, 0.7, 0.3]))
        doc_len = int(rng.integers(1, 3000))
        max_freq = int(rng.integers(1, 100))
        doc_score = float(np.float32(rng.choice([1.0, 0.5, 0.1, 0.0, 0.77])))
        avg = float(rng.uniform(5, 700))
        slop = int(rng.integers(1, 5))
        min_score = float(rng.choice([0.0, 0.0, 0.05]))
        tanh = int(rng.integers(1, 20))
        a = ol.oracle_score(scorer, freqs, idf, bidf, weights, aggw, doc_len, max_freq, doc_score, num_docs, avg, slop, min_score, float(tanh))
        b = ol.reference_score(scorer, freqs, idf, bidf, weights, aggw, doc_len, max_freq, doc_score, num_docs, avg, slop, min_score, tanh)
        assert np.float64(a).tobytes() == np.float64(b).tobytes(), (scorer, a, b)


def test_reference_scorers_reproduce_their_own_golden(ref):
    """Sanity of the harness itself: the reference's BM25STD through libscorers_ref gives 0.54/0.52/0.51."""
    g = G["bm25std_explain"]
    idf = math.log(1 + 0.5 / 3.5)
    for doc_len, total, _ in g["cases"]:
        s = ol.reference_score(ol.SCORER_BM25STD, [10, 10], [0, 0], [idf, idf], [1.0, 1.0], 1.0, doc_len, 10, 1.0, 3, g["avg_doc_len"])
        assert f"{s:.2f}" == f"{total:.2f}"


def test_union_reference_edge_cases(L):
    """rqe_iterators/tests/integration/union_common.rs:243-452 — the reference's own known answers."""
    E = G["union_edge_cases"]

    def run(children, **kw):
        idx = [ol.InvIndex(ol.CODEC_DOCIDS_ONLY, np.array(c, dtype=np.uint64)) for c in children]
        return idx, [h[0] for h in ol.run_intersect(idx, union=True, **kw)]

    for name in ("disjoint", "overlapping", "empty_mixed", "all_empty"):
        for quick in (False, True):
            _, got = run(E[name]["children"], quick=quick)
            assert got == E[name]["expected"], (name, quick, got)
    for name in ("skip_exact", "skip_not_found", "skip_past_eof"):
        idx = [ol.InvIndex(ol.CODEC_DOCIDS_ONLY, np.array(c, dtype=np.uint64)) for c in E[name]["children"]]
        readers = [ix.reader() for ix in idx]
        arr = (C.c_void_p * len(readers))(*readers)
        t = (C.c_uint64 * 1)(*E[name]["targets"])
        st, landed = (C.c_int * 1)(), (C.c_uint64 * 1)()
        L.orc_union_skipto(arr, len(readers), t, 1, st, landed)
        assert list(st) == E[name]["status"], name
        if "landed" in E[name]:
            assert list(landed) == E[name]["landed"], name
        for r in readers:
            L.orc_reader_free(r)


def test_intersection_reference_edge_cases(L):
    """rqe_iterators/tests/integration/intersection.rs:325-521, 876-931 — the reference's own known answers."""
    E = G["intersection_edge_cases"]
    for name, case in E.items():
        if name.startswith("_"):
            continue
        idx = [ol.InvIndex(ol.CODEC_DOCIDS_ONLY, np.array(c, dtype=np.uint64)) for c in case["children"]]
        if "expected" in case:
            assert [h[0] for h in ol.run_intersect(idx)] == case["expected"], name
        for target, status, landed in case.get("skips", []):  # each skip on a fresh (rewound) iterator
            readers = [ix.reader() for ix in idx]
            arr = (C.c_void_p * len(readers))(*readers)
            t = (C.c_uint64 * 1)(target)
            st, ld = (C.c_int * 1)(), (C.c_uint64 * 1)()
            L.orc_intersect_skipto(arr, len(readers), t, 1, st, ld)
            assert st[0] == status, (name, target, st[0])
            if status != 2:
                assert ld[0] == landed, (name, target, ld[0])
            for r in readers:
                L.orc_reader_free(r)


def test_proximity_known_answers_of_the_reference():
    """RS/index_result/src/core/proximity.rs tests (:318-392): in-order / unordered slop checks over varint-delta offsets."""
    vw1, vw2 = bytes([1, 8, 4, 3, 6]), bytes([4, 3, 25])  # positions 1,9,13,16,22 and 4,7,32
    for slop, exp in ((0, False), (1, False), (2, True), (3, True), (4, True), (5, True)):
        assert ol.within_range([vw1, vw2], slop, True) is exp, ("in_order", slop)
    for slop, exp in ((0, False), (1, True), (2, True), (3, True), (4, True)):
        assert ol.within_range([vw1, vw2], slop, False) is exp, ("unordered", slop)
    assert ol.within_range([bytes([3]), bytes([4])], 0, True)          # in_order_exact_consecutive
    assert not ol.within_range([bytes([10]), bytes([5])], 100, True)   # in_order_out_of_order_terms
    assert not ol.within_range([bytes([10]), bytes([5])], 3, False)    # unordered_reversed_order_ok
    assert ol.within_range([bytes([10]), bytes([5])], 4, False)
    # a child without offsets is left out of the check; one stream left = trivially in range (is_within_range :282-290)
    assert ol.within_range([b"", bytes([5])], 0, True) and ol.within_range([bytes([5])], 0, False)
    # no slop limit, order only
    assert ol.within_range([bytes([1]), bytes([90])], None, True) and not ol.within_range([bytes([90]), bytes([1])], None, True)
    # multi-byte varints (the -1 bias per continuation): 300 = [0x81, 0x2c]
    enc = lambda v: bytes(ol_varint(v))
    assert ol.within_range([enc(300), enc(302)], 1, True) and not ol.within_range([enc(300), enc(303)], 1, True)


def test_numeric_codec_golden_bytes():
    """RS/inverted_index/src/codec/numeric.rs against the byte vectors of inverted_index/tests/integration/codec/numeric.rs:220-600
    (tiny / positive / negative integers, f32, f64, infinities, 0-7 delta bytes) and its stored-value edge cases (:62-86)."""
    D7 = 72_057_594_037_927_935
    f64_3124 = [203, 161, 69, 182, 243, 253, 8, 64]
    cases = [
        (0, 2.0, [0b010_00_000]), (2, 7.0, [0b111_00_001, 2]), (D7, 0.0, [0b000_00_111] + [255] * 7), (0, 0.0, [0]), (0, -0.0, [0]),
        (1, 16.0, [0b000_10_001, 1, 16]), (0, 256.0, [0b001_10_000, 0, 1]), (D7, float(2**64 - 1), [0b111_10_111] + [255] * 15),
        (0, -16.0, [0b000_11_000, 16]), (1, -16.0, [0b000_11_001, 1, 16]), (0, -256.0, [0b001_11_000, 0, 1]),
        (D7, -float(2**64 - 1), [0b111_11_111] + [255] * 15),
        (0, 3.125, [0b000_01_000, 0, 0, 72, 64]), (D7, 3.125, [0b000_01_111] + [255] * 7 + [0, 0, 72, 64]),
        (0, -3.125, [0b010_01_000, 0, 0, 72, 64]), (D7, -3.125, [0b010_01_111] + [255] * 7 + [0, 0, 72, 64]),
        (0, math.inf, [0b001_01_000]), (D7, math.inf, [0b001_01_111] + [255] * 7),
        (0, -math.inf, [0b011_01_000]), (D7, -math.inf, [0b011_01_111] + [255] * 7),
        (0, 3.124, [0b100_01_000] + f64_3124), (D7, 3.124, [0b100_01_111] + [255] * 7 + f64_3124),
        (0, -3.124, [0b110_01_000] + f64_3124), (D7, -3.124, [0b110_01_111] + [255] * 7 + f64_3124),
    ]
    for delta, value, expected in cases:
        assert list(ol.numeric_encode(delta, value)) == expected, (delta, value)
        n, d, v = ol.numeric_decode(bytes(expected))
        assert n == len(expected) and d == delta and (v == value or abs(value) >= 2.0**63), (delta, value, v)
    # float compression (numeric.rs:625-700): 3.124 is within 0.01 of its f32, 1e-9 is stored as the canonical zero... only when it
    # collapses: |1e-9 - f32(1e-9)| < 0.01 and f32(1e-9) != 0 -> f32
    assert len(ol.numeric_encode(0, 3.124, compress=True)) == 5 and len(ol.numeric_encode(0, 3.124)) == 9
    n, _, v = ol.numeric_decode(ol.numeric_encode(0, 3.124, compress=True))
    assert v == float(np.float32(3.124))
    for value in (0.0, -0.0, 1.0, 7.0, 8.0, -1.0, -8.0, 0.5, -0.5, 100.500001, 1e-9, 9_007_199_254_740_993.0, 4_503_599_627_370_496.0,
                  1.7976931348623157e308, -1.7976931348623157e308, 2.2250738585072014e-308, math.inf, -math.inf):
        for compress in (False, True):
            n, _, v = ol.numeric_decode(ol.numeric_encode(5, value, compress))
            if not compress or value in (math.inf, -math.inf):
                assert v == value and (math.copysign(1, v) == math.copysign(1, value) or value == 0)
            else:
                assert abs(v - value) < 0.01
            # stored_value is idempotent (numeric.rs:44-57)
            assert ol.numeric_decode(ol.numeric_encode(0, v, compress))[2] == v


def test_min_offset_delta_equals_the_reference(ref):
    """GetSlop of the legacy scorers: the restatement against the reference's own index_result.c, and its doc-comment example."""
    assert ol.min_offset_delta([[2, 4, 8], [0, 5, 12]]) == 1           # index_result.c:47-50: abs(4-5)
    assert ol.min_offset_delta([[5]]) == 1 and ol.min_offset_delta([[], []]) == 1 and ol.min_offset_delta([[], [], []]) == 2
    assert ol.min_offset_delta([[1], [10]]) == 9 and ol.min_offset_delta([[1], [4], [8]]) == 5  # sqrt(9 + 16)
    rng = np.random.default_rng(77)
    for _ in range(3000):
        n = int(rng.integers(1, 7))
        positions, virtual = [], []
        for _i in range(n):
            kind = rng.integers(0, 8)
            cnt = 0 if kind == 0 else int(rng.integers(1, 9))
            positions.append(np.sort(rng.choice(np.arange(1, 60), size=cnt, replace=False)).tolist())
            virtual.append(kind == 1)
        a = ol.min_offset_delta(positions, virtual)
        b = ol.reference_min_offset_delta(positions, virtual)
        assert a == b, (positions, virtual, a, b)


def ol_varint(v):
    out = (C.c_uint8 * 16)()
    n = ol.postings().orc_varint_encode(v, out)
    return bytes(out[:n])
