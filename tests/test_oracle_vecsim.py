"""Pins oracle/vecsim_oracle.c (our CPU restatement) to the reference:
  * against oracle/_ref/libvecsim_ref.so — the reference's own VecSim sources compiled in place, its answers recorded on an
    AVX-512F host under tests/golden/reference/ — on seeded random inputs (bit-equal where the arithmetic is order-defined), and
  * against the known answers of the reference's unit tests
    (deps/VectorSimilarity/tests/unit/test_bruteforce.cpp, test_spaces.cpp).
CPU only.
"""
import os

import numpy as np
import pytest

import oracle_lib as ol
from oracle_lib import BF16, COS, F16, F32, I8, IP, L2, TIER_AVX512, TIER_SCALAR, U8

DIMS = [1, 2, 3, 4, 7, 8, 9, 15, 16, 17, 24, 31, 32, 33, 40, 47, 48, 63, 64, 65, 100, 128, 255, 256, 768, 771]


def _bits(x):
    return np.float32(x).tobytes()


def _rand(rng, vtype, dim, metric):
    x = rng.uniform(-1, 1, dim).astype(np.float32)
    blob = ol.to_type(x, vtype)
    if vtype in (I8, U8) and metric == COS:
        buf = np.zeros(dim + 4, dtype=np.uint8)
        buf[:dim] = blob.view(np.uint8)
        ol.port().orc_normalize(ol._p(buf), dim, vtype)
        return buf
    return blob


# ------------------------------------------------------------------ distances vs the reference
@pytest.mark.parametrize("metric", [L2, IP])
def test_fp32_distance_bit_equal_to_reference_tier(oracle, ref, metric):
    """fp32: the AVX-512 emulation must equal the reference's dispatched kernel bit for bit on an
    AVX-512F host; with every SIMD tier masked off the reference falls back to its scalar
    baseline, which must equal our scalar restatement (test_spaces.cpp:683-736 spirit)."""
    rng = np.random.default_rng(1234 + metric)
    for tier, mask in ((TIER_AVX512, None), (TIER_SCALAR, "avx512f,avx,avx2,sse,sse3,sse4_1,fma3,f16c")):
        if mask:
            os.environ["REF_CPU_MASK"] = mask
        try:
            for dim in DIMS:
                for _ in range(8):
                    a = rng.uniform(-1, 1, dim).astype(np.float32)
                    b = rng.uniform(-1, 1, dim).astype(np.float32)
                    r = ol.reference_distance(F32, metric, dim, a, b)
                    o = oracle.orc_distance(F32, metric, dim, ol._p(a), ol._p(b), tier)
                    assert _bits(r) == _bits(o), (tier, dim, r, o)
        finally:
            os.environ.pop("REF_CPU_MASK", None)


@pytest.mark.parametrize("vtype", [I8, U8])
@pytest.mark.parametrize("metric", [L2, IP, COS])
def test_int_distance_exact(oracle, ref, vtype, metric):
    """int8/uint8 accumulate exactly in int32, so every reference tier and our port agree bit for bit
    (IP.cpp:248-285, L2.cpp:150-174)."""
    rng = np.random.default_rng(99 + vtype * 3 + metric)
    for dim in DIMS:
        for _ in range(4):
            a = _rand(rng, vtype, dim, metric)
            b = _rand(rng, vtype, dim, metric)
            r = ol.reference_distance(vtype, metric, dim, a, b)
            o = oracle.orc_distance(vtype, metric, dim, ol._p(a), ol._p(b), TIER_SCALAR)
            assert _bits(r) == _bits(o), (dim, r, o)


@pytest.mark.parametrize("vtype", [F16, BF16])
@pytest.mark.parametrize("metric", [L2, IP])
def test_half_distance_close_to_fp32_accumulate_tier(oracle, ref, vtype, metric):
    """fp16/bf16: our port accumulates in fp32 like the reference's scalar / AVX512F / bf16 tiers.
    The AVX512-FP16 tier (fp16 accumulation) is masked off — SURVEY.md §0 finding 5."""
    rng = np.random.default_rng(7 + vtype + metric)
    os.environ["REF_CPU_MASK"] = "avx512_fp16"
    try:
        for dim in DIMS:
            a = _rand(rng, vtype, dim, metric)
            b = _rand(rng, vtype, dim, metric)
            r = ol.reference_distance(vtype, metric, dim, a, b)
            o = oracle.orc_distance(vtype, metric, dim, ol._p(a), ol._p(b), TIER_SCALAR)
            scale = 1.0 if metric == IP else 0.0
            assert abs(r - o) <= 1e-4 * max(abs(r), scale) + 1e-6, (dim, r, o)
    finally:
        os.environ.pop("REF_CPU_MASK", None)


@pytest.mark.parametrize("vtype", [F32, F16, BF16, I8, U8])
def test_normalize_bit_equal(oracle, ref, vtype):
    rng = np.random.default_rng(5 + vtype)
    for dim in [1, 3, 8, 17, 128, 768]:
        x = rng.uniform(-1, 1, dim).astype(np.float32)
        blob = ol.to_type(x, vtype)
        extra = 4 if vtype in (I8, U8) else 0
        a = np.zeros(blob.nbytes + extra, dtype=np.uint8)
        a[: blob.nbytes] = blob.view(np.uint8)
        b = a.copy()
        a = ol.reference_normalize(a, dim, vtype)
        oracle.orc_normalize(ol._p(b), dim, vtype)
        assert a.tobytes() == b.tobytes(), dim


# ------------------------------------------------------------------ index semantics vs the reference
def _fill(ix, blobs, label0=0):
    ix.add_many(blobs, label0)


@pytest.mark.parametrize("vtype,metric", [(F32, L2), (F32, IP), (F32, COS), (F16, COS), (BF16, L2), (I8, COS), (U8, L2), (I8, IP)])
def test_topk_matches_reference_index(oracle, ref, vtype, metric):
    rng = np.random.default_rng(31 + vtype * 7 + metric)
    n, dim, k = 3000, 96, 10
    x = rng.uniform(-1, 1, (n, dim)).astype(np.float32)
    blobs = ol.to_type(x, vtype)
    os.environ["REF_CPU_MASK"] = "avx512_fp16"
    try:
        r = ol.RefIndex(vtype, dim, metric)
        p = ol.PortIndex(vtype, dim, metric, tier=TIER_AVX512)
        _fill(r, blobs, 1)
        _fill(p, blobs, 1)
        exact = vtype in (I8, U8, F32)
        for qi in range(5):
            q = ol.to_type(rng.uniform(-1, 1, dim).astype(np.float32), vtype)
            for order in (0, 1):
                ri, rs = r.topk(q, k, order)
                pi, ps = p.topk(q, k, order)
                if exact:
                    assert ri.tolist() == pi.tolist()
                    assert rs.tobytes() == ps.tobytes()
                else:
                    assert set(ri.tolist()) == set(pi.tolist())
                    np.testing.assert_allclose(np.sort(rs), np.sort(ps), rtol=1e-4, atol=1e-5)
    finally:
        os.environ.pop("REF_CPU_MASK", None)


def test_swap_delete_and_update_match_reference(oracle, ref):
    rng = np.random.default_rng(77)
    n, dim = 500, 16
    x = rng.uniform(-1, 1, (n, dim)).astype(np.float32)
    r = ol.RefIndex(F32, dim, L2)
    p = ol.PortIndex(F32, dim, L2, tier=TIER_AVX512)
    _fill(r, x, 0)
    _fill(p, x, 0)
    for lab in rng.choice(n, 120, replace=False).tolist():
        assert r.delete(lab) == p.delete(lab) == 1
    assert r.delete(10**9) == p.delete(10**9) == 0
    for lab in [3, 5, 8]:  # update in place / re-add
        v = rng.uniform(-1, 1, dim).astype(np.float32)
        assert r.add(v, lab) == p.add(v, lab)
    assert r.size() == p.size()
    q = rng.uniform(-1, 1, dim).astype(np.float32)
    ri, rs = r.topk(q, 25)
    pi, ps = p.topk(q, 25)
    assert ri.tolist() == pi.tolist()
    np.testing.assert_allclose(rs, ps, rtol=1e-6)
    for lab in [0, 1, 3, 10**9]:
        a, b = r.distance_from(lab, q), p.distance_from(lab, q)
        assert (np.isnan(a) and np.isnan(b)) or abs(a - b) <= 1e-6 * abs(a)


def test_range_and_batches_match_reference(oracle, ref):
    rng = np.random.default_rng(8)
    n, dim = 2000, 32
    x = rng.uniform(-1, 1, (n, dim)).astype(np.float32)
    r = ol.RefIndex(F32, dim, L2)
    p = ol.PortIndex(F32, dim, L2, tier=TIER_AVX512)
    _fill(r, x, 1)
    _fill(p, x, 1)
    q = rng.uniform(-1, 1, dim).astype(np.float32)
    for radius in [0.0, 6.0, 9.0, 1e9]:
        for order in (0, 1):
            ri, rs = r.range(q, radius, order)
            pi, ps = p.range(q, radius, order)
            assert ri.tolist() == pi.tolist()
    allp, alls = p.all_sorted(q)
    got = []
    for ids, scores in r.batches(q, 300, 0):
        got += ids.tolist()
    assert got == allp.tolist()


@pytest.mark.parametrize("dim", [4, 75, 76, 300, 301, 750, 751, 768])
def test_prefer_adhoc_tree_matches_reference(oracle, ref, dim):
    """brute_force.h:380-451 — drive both through every leaf by faking the index size with tiny
    vectors is too costly; instead compare on real small/medium indexes and on the thresholds."""
    for n in [100, 5500, 5501, 6000]:
        r = ol.RefIndex(F32, dim, L2)
        p = ol.PortIndex(F32, dim, L2)
        x = np.zeros((n, dim), dtype=np.float32)
        _fill(r, x, 0)
        _fill(p, x, 0)
        for frac in [0.0, 0.1, 0.15, 0.16, 0.35, 0.36, 0.55, 0.56, 0.75, 0.76, 1.0, 2.0]:
            s = int(frac * n)
            assert r.prefer_adhoc(s, 10, True) == p.prefer_adhoc(s, 10, True), (n, dim, frac)


# ------------------------------------------------------------------ known answers from the reference's unit tests
@pytest.mark.parametrize("vtype", [F32, F16, BF16])
def test_known_answers_bruteforce_l2(oracle, vtype):
    """test_bruteforce.cpp:781-812: vectors (i,i,i,i), query (50,..): id distance (idx+1)/2, score 4*((idx+1)/2)^2."""
    dim, n, k = 4, 100, 11
    p = ol.PortIndex(vtype, dim, L2)
    for i in range(n):
        p.add(ol.to_type(np.full(dim, float(i), dtype=np.float32), vtype), i)
    ids, scores = p.topk(ol.to_type(np.full(dim, 50.0, dtype=np.float32), vtype), k)
    assert len(ids) == k
    for idx, (i, s) in enumerate(zip(ids.tolist(), scores.tolist())):
        assert abs(i - 50) == (idx + 1) // 2
        assert s == 4 * ((idx + 1) // 2) ** 2
    assert len(p.topk(np.zeros(dim, dtype=np.float32), 0)[0]) == 0


def test_known_answers_bruteforce_ip(oracle):
    """test_bruteforce.cpp:747-779: top-11 by inner product are the 11 largest vectors."""
    dim, n, k = 4, 100, 11
    p = ol.PortIndex(F32, dim, IP)
    for i in range(n):
        p.add(np.full(dim, float(i), dtype=np.float32), i)
    ids, _ = p.topk(np.full(dim, 50.0, dtype=np.float32), k)
    assert set(ids.tolist()) == set(range(n - k, n))


def test_known_answers_spaces(oracle):
    """test_spaces.cpp:68-140 style known answers on exactly representable data: v1[i]=i, v2[i]=i+1.5."""
    dim = 5
    a = np.arange(dim, dtype=np.float32)
    b = a + np.float32(1.5)
    for tier in (TIER_SCALAR, TIER_AVX512):
        assert oracle.orc_distance(F32, L2, dim, ol._p(a), ol._p(b), tier) == dim * 2.25
        assert oracle.orc_distance(F32, IP, dim, ol._p(a), ol._p(b), tier) == 1.0 - float(np.dot(a, b))
    ai = np.array([1, 2, 3, 4, 5], dtype=np.int8)
    assert oracle.orc_distance(I8, L2, dim, ol._p(ai), ol._p(ai), 0) == 0.0
    assert oracle.orc_distance(I8, IP, dim, ol._p(ai), ol._p(ai), 0) == 1.0 - 55.0


def test_streaming_topk_equals_the_reference_index(ref):
    """bench.py's parity check at the full 10M x 768 size feeds the device's own rows back chunk by chunk to
    ol.StreamingTopK (the reference's distance kernels + heap over a flat array): it must answer exactly like the
    reference's BruteForceIndex::topKQuery over the same rows, ties at the boundary included."""
    n, dim, k = 30_000, 96, 10
    rows = ol.synth_rows(ol.F32, 1, 0, n, dim)
    rows[5000:5010] = rows[100]  # exact duplicates: score ties resolved like the heap does
    for r in rows:
        ol.port().orc_normalize(ol._p(r), dim, ol.F32)
    qs = ol.synth_rows(ol.F32, 2, 0, 4, dim)
    qs[3] = rows[100]
    for r in qs:
        ol.port().orc_normalize(ol._p(r), dim, ol.F32)
    ix = ol.PortIndex(ol.F32, dim, ol.IP, tier=ol.TIER_AVX512)
    ix.add_many(rows, 1)
    for kind in ("port", "reference"):
        st = ol.StreamingTopK(ol.F32, ol.COS, dim, qs, k, 3)
        st.kind = kind
        for c in range(0, n, 7000):
            st.feed(rows[c:c + 7000], 1 + c)
        for i in range(len(qs)):
            a, b = ix.topk(qs[i], k)
            l, s = st.result(i)
            assert a.tolist() == l.tolist(), (kind, i)
            assert b.astype(np.float32).tobytes() == s.tobytes()
