"""GPU: the FLAT index's "all scores" path through the C-ABI — scan_scores_kernel<DT,MT> for every (type, metric), then
range_compact_kernel (range queries) or the cursor-chunked select_scores_kernel + final_select_kernel (batch iterators, top-k
with k > 128, every top-k of a multi-value index) and the host logic of csrc/vecsim_index.cpp — against the oracle
(oracle/vecsim_oracle.c, pinned to the reference on these paths by tests/test_oracle_vecsim_scan_paths.py) and, for the
batch-iterator scripts and the NaN rule, against the reference's own answers replayed from tests/golden/reference/.

Bars (as in test_vecsim_parity.py): fp32 / int8 / uint8 ids in order and score bits equal; fp16 / bf16 scores within
2e-4 * max(|score|, 1) position by position, ids equal except for labels whose oracle distance is within that tolerance of the
k-th score or of the radius.  Largest fp16 / bf16 deviation from the oracle measured on these paths (B200, every check of
this file): 7.2e-7 * max(|score|, 1), well under the 2e-4 bar; the module prints it at the end of a run.

Score ties: the device orders candidates by (score, row id), the reference's heap by (score, label); they differ at the k-th
boundary only after swap-deletes permuted labels against row ids (DESIGN.md §3.2).  Every tie group below has labels ascending
in row order and is never moved by a swap-delete, so the expected order is (score, label) whatever that deviation does.
"""
import os

import numpy as np
import pytest

import oracle_lib as ol
from oracle_lib import BF16, COS, F16, F32, I8, IP, L2, TIER_AVX512, U8

pytestmark = pytest.mark.gpu

TYPES = [F32, F16, BF16, I8, U8]
METRICS = [L2, IP, COS]
CASES = [(t, m) for t in TYPES for m in METRICS]
DIMS = [7, 17, 33]
HALF_TOL = 2e-4
_dev = {"max": 0.0}


@pytest.fixture(scope="module")
def vs():
    from redisearch_b200 import vecsim

    yield vecsim
    print(f"\nlargest fp16/bf16 deviation from the oracle on the scan paths: {_dev['max']:.3e}")


def _exact(vtype):
    return vtype in (F32, I8, U8)


class _HalfTier:
    """the reference's fp16 / bf16 distances by its fp32-accumulating tiers, as everywhere in the suite (SURVEY.md §0)"""

    def __init__(self, vtype):
        self.on = vtype in (F16, BF16)

    def __enter__(self):
        if self.on:
            os.environ["REF_CPU_MASK"] = "avx512_fp16"

    def __exit__(self, *a):
        os.environ.pop("REF_CPU_MASK", None)


def _tol(s):
    return HALF_TOL * np.maximum(np.abs(s), 1.0)


def _rows(rng, vtype, n, dim, scale=1.0):
    return ol.to_type(rng.uniform(-scale, scale, (n, dim)).astype(np.float32), vtype)


def _pair(vs, vtype, dim, metric, multi=False):
    return vs.VecSimIndex(vtype, dim, metric, multi=multi), ol.PortIndex(vtype, dim, metric, multi=multi, tier=TIER_AVX512)


def _add_rows(g, p, blobs, labels):
    labels = np.asarray(labels, dtype=np.uint64)
    assert g.add_many(blobs, labels=labels) == len(blobs)
    for b, lab in zip(blobs, labels.tolist()):
        p.add(b, lab)


def _canon(ids, scores):
    ids, scores = np.asarray(ids, dtype=np.int64), np.asarray(scores, dtype=np.float64)
    o = np.lexsort((ids, scores))
    return ids[o], scores[o]


def same(vtype, got, want, what="", complete=False, open_start=False):
    """got = the device's (ids, scores) in its reply order, want = the oracle's in (score, label) order.  fp16 / bf16: a label
    on one side only must lie within the tolerance of the last score (or of the first, with `open_start`: a batch)."""
    gi, gs = np.asarray(got[0], dtype=np.int64), np.asarray(got[1], dtype=np.float64)
    wi, ws = np.asarray(want[0], dtype=np.int64), np.asarray(want[1], dtype=np.float64)
    assert len(gi) == len(wi), (what, len(gi), len(wi))
    if _exact(vtype):
        assert gi.tolist() == wi.tolist(), what
        assert gs.astype(np.float32).tobytes() == ws.astype(np.float32).tobytes(), what
        return
    if len(ws):
        dev = np.abs(gs - ws) / np.maximum(np.abs(ws), 1.0)
        _dev["max"] = max(_dev["max"], float(dev.max()))
        assert np.all(np.abs(gs - ws) <= _tol(ws)), (what, float(dev.max()))
        only = set(gi.tolist()) ^ set(wi.tolist())
        assert not (complete and only), what
        cut = ws[-1]
        wmap = dict(zip(wi.tolist(), ws.tolist()))
        gmap = dict(zip(gi.tolist(), gs.tolist()))
        for lab in only:
            s = wmap.get(lab, gmap.get(lab))
            assert abs(s - cut) <= 2 * _tol(cut) or (open_start and abs(s - ws[0]) <= 2 * _tol(ws[0])), (what, lab)


def same_range(vtype, got, want, radius, all_dist, what=""):
    if _exact(vtype):
        same(vtype, got, want, what)
        return
    gmap, wmap = dict(zip(got[0].tolist(), got[1].tolist())), dict(zip(want[0].tolist(), want[1].tolist()))
    for lab in set(gmap) ^ set(wmap):  # only labels farther than the tolerance from the radius must agree
        assert abs(all_dist[lab] - radius) <= 2 * _tol(radius), (what, lab, all_dist[lab], radius)
    for lab in set(gmap) & set(wmap):
        d = abs(gmap[lab] - wmap[lab])
        _dev["max"] = max(_dev["max"], d / max(abs(wmap[lab]), 1.0))
        assert d <= _tol(wmap[lab]), (what, lab)


def radii(ds):
    """0; an observed distance (included: `<=`); the float below it (excluded); a double that rounds to it (both sides cast
    the radius to float, brute_force.h:306); 1e9.  From the oracle's sorted distances, since IP and int8/uint8 cosine
    distances can be negative or above 1; the C-ABI takes non-negative radii only (vec_sim.cpp:365-367)."""
    pos = ds[ds >= 0]
    out = [0.0, 1e9]
    if len(pos):
        d = np.float32(pos[len(pos) // 2])
        near = float(d) + float(np.spacing(d)) * 0.25
        assert np.float32(near) == d
        out += [float(d), near] + ([float(np.nextafter(d, np.float32(-np.inf)))] if d > 0 else [])
    return out


def check_range(vtype, g, p, q, what):
    ai, as_ = p.all_sorted(q)
    all_dist = dict(zip(ai.tolist(), as_.tolist()))
    with pytest.raises(ValueError):
        g.range(q, -1e-30)
    for radius in radii(as_):
        for order in (0, 1):
            gi, gs, code = g.range(q, radius, order)
            pi, ps = p.range(q, radius, order)
            assert code == 0
            if order == 1:
                assert gi.tolist() == sorted(gi.tolist())
                gi, gs = _canon(gi, gs)
                pi, ps = _canon(pi, ps)
            same_range(vtype, (gi, gs), (pi, ps), radius, all_dist, (what, "range", radius, order))
        if _exact(vtype) and radius == float(np.float32(radius)) and 0 < radius < 1e9:
            inside = int(np.sum(as_.astype(np.float32) <= np.float32(radius)))
            assert len(g.range(q, radius)[0]) == inside  # the radius itself is a distance: its labels are in


def drain(vs, vtype, g, p, q, size, what, orders=(0,)):
    """Drain a device batch iterator `size` at a time (cycling `orders`): the batches continue each other in (score, label)
    order with no repeats and no gaps, exactly label_count results, then an empty next."""
    ai, as_ = p.all_sorted(q)
    it = g.batch_iterator(q)
    got_i, got_s, j = [], [], 0
    while it.has_next():
        order = orders[j % len(orders)]
        bi, bs, code = it.next(size, order)
        assert code == 0 and 0 < len(bi) <= size, (what, size, j)
        if order == 1:
            assert bi.tolist() == sorted(bi.tolist())
            bi, bs = _canon(bi, bs)
        lo = len(got_i)
        same(vtype, (bi, bs), (ai[lo:lo + len(bi)], as_[lo:lo + len(bi)]), (what, "batch", size, j), open_start=True)
        got_i += bi.tolist()
        got_s += bs.tolist()
        j += 1
    assert len(got_i) == len(set(got_i)) == len(ai), (what, size)
    assert set(got_i) == set(ai.tolist())
    bi, _, code = it.next(size)
    assert code == 0 and len(bi) == 0
    it.free()


# ------------------------------------------------------------------ row-tile / grid edges, cursor chunking, range radii
@pytest.mark.parametrize("vtype,metric", CASES)
def test_single_value_row_tile_edges(vs, vtype, metric):
    """n in {1, 3, 4, 5, 129, 4099} (4-row tiles with a clamped last tile): top-k at k in {129, 256, 257, 1000, n, n+1},
    range radii around an observed distance in both orders, batch iterators of 1, 7, 128, 129 and 500 drained."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(7000 + ci)
    dim = DIMS[ci % 3]
    for n in (1, 3, 4, 5, 129, 4099):
        g, p = _pair(vs, vtype, dim, metric)
        _add_rows(g, p, _rows(rng, vtype, n, dim, 1.0 if metric != IP else 1.7), np.arange(1, n + 1))
        q = _rows(rng, vtype, 1, dim)[0]
        for k in sorted({129, 256, 257, 1000, n, n + 1}):
            gi, gs, code = g.topk(q, k)
            assert code == 0
            same(vtype, (gi, gs), p.topk(q, k), (n, "topk", k), complete=k >= n)
        check_range(vtype, g, p, q, n)
        for size in (1, 7, 128, 129, 500):
            if size == 1 and n > 129:
                continue
            drain(vs, vtype, g, p, q, size, n, orders=(0, 1) if size == 7 else (0,))
        g.close()


@pytest.mark.parametrize("vtype,metric", CASES)
def test_tie_groups_across_cursor_chunks(vs, vtype, metric):
    """Two blocks of 250 and 270 identical rows (labels ascending in row order), one tied with the row ranked ~60th and one
    with the row ranked ~700th against the query, so that tie groups span 128-entry chunks of select_from_scores: top-k
    at k in {129, 256, 257, 1000, n, n+1} and batch iterators must continue in (score, label) order through them."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(7100 + ci)
    dim, n0 = DIMS[(ci + 2) % 3], 1500
    x = _rows(rng, vtype, n0, dim, 1.0 if metric != IP else 1.7)
    q = _rows(rng, vtype, 1, dim)[0]
    p0 = ol.PortIndex(vtype, dim, metric, tier=TIER_AVX512)
    p0.add_many(x, 1)
    order = p0.all_sorted(q)[0]
    blocks = np.concatenate([np.repeat(x[order[60] - 1][None], 250, 0), np.repeat(x[order[700] - 1][None], 270, 0)])
    rows = np.concatenate([x, blocks])
    n = len(rows)
    g, p = _pair(vs, vtype, dim, metric)
    _add_rows(g, p, rows, np.arange(1, n + 1))
    ai, as_ = p.all_sorted(q)
    if _exact(vtype):
        assert np.sum(as_[60:320] == as_[60]) >= 251  # the first group starts at rank 60 and crosses 128 and 256
    for k in (129, 256, 257, 1000, n, n + 1):
        gi, gs, code = g.topk(q, k)
        assert code == 0
        same(vtype, (gi, gs), p.topk(q, k), ("topk", k), complete=k >= n)
    for size in (7, 128, 129, 500):
        drain(vs, vtype, g, p, q, size, "ties", orders=(0, 1))
    # several queries at once with k > 128 take the per-query path: same answers as one query at a time
    qs = np.stack([q, rows[order[60] - 1], _rows(rng, vtype, 1, dim)[0]])
    for k in (129, 300):
        labels, scores, rc = g.topk_batch(qs, k)
        assert rc == 0
        for i in range(len(qs)):
            gi, gs, _ = g.topk(qs[i], k)
            assert labels[i].astype(np.int64).tolist() == gi.tolist()
            assert scores[i].tobytes() == gs.tobytes()
            same(vtype, (gi, gs), p.topk(qs[i], k), ("topk_batch", k, i))
    g.close()


@pytest.mark.parametrize("vtype", TYPES)
def test_select_grid_stride_rounds(vs, vtype):
    """n = 200,003 rows: select_scores_kernel walks the score array in several grid-stride rounds and ends on a partial
    warp; scan_scores_kernel clamps the last 4-row tile."""
    metric = METRICS[TYPES.index(vtype) % 3]
    n, dim = 200_003, 17
    rows = ol.synth_rows(vtype, 11 + vtype, 0, n, dim)
    q = ol.synth_rows(vtype, 12 + vtype, 0, 1, dim)[0]
    g, p = _pair(vs, vtype, dim, metric)
    assert g.add_many(rows, label0=1) == n
    p.add_many(rows, 1)
    ai, as_ = p.all_sorted(q)
    for k in (129, 1000):
        gi, gs, code = g.topk(q, k)
        assert code == 0
        same(vtype, (gi, gs), (ai[:k], as_[:k]), ("topk", k))
    it = g.batch_iterator(q)
    lo = 0
    for j, (size, order) in enumerate(((500, 0), (129, 1), (1000, 0))):
        bi, bs, code = it.next(size, order)
        assert code == 0 and len(bi) == size
        if order == 1:
            bi, bs = _canon(bi, bs)
        same(vtype, (bi, bs), (ai[lo:lo + size], as_[lo:lo + size]), ("batch", j), open_start=True)
        lo += size
    it.free()
    pos = as_[as_ >= 0]
    radius = float(np.float32(pos[min(3000, len(pos) - 1)])) if len(pos) else 1e9  # uint8 IP: every distance is negative
    all_dist = dict(zip(ai.tolist(), as_.tolist()))
    gi, gs, code = g.range(q, radius)
    pi, ps = p.range(q, radius)
    assert code == 0
    same_range(vtype, (gi, gs), (pi, ps), radius, all_dist, "range")
    g.close()


# ------------------------------------------------------------------ batch iterator: order switches, reset, mutation
def _scripts(rng, vtype, dim, n):
    new = _rows(rng, vtype, 3, dim)
    plain = [("next", 7, 0), ("next", 129, 1), ("has_next",), ("next", 1, 0), ("reset",), ("next", 5, 0), ("next", 128, 1),
             ("next", 500, 0), ("has_next",), ("next", 10, 0)]
    # mutated after batch_new and before the first next (the first next reads the index), then again between two nexts
    # (later nexts continue from the scores of the first); a reset re-reads the index
    mutated = [("delete", 3), ("add", new[0], n + 10), ("delete", n // 2), ("next", 50, 0), ("delete", 5),
               ("add", new[1], n + 11), ("next", 129, 0), ("next", 1000, 1), ("has_next",), ("next", 3, 0), ("reset",),
               ("add", new[2], n + 12), ("next", 20, 0)]
    return plain, mutated


def _run_script_device(g, p, q, steps):
    it = g.batch_iterator(q)
    out = []
    for st in steps:
        if st[0] == "next":
            gi, gs, code = it.next(st[1], st[2])
            assert code == 0
            out.append((gi, gs))
        elif st[0] == "reset":
            it.reset()
            out.append(None)
        elif st[0] == "has_next":
            out.append(it.has_next())
        elif st[0] == "add":
            out.append(g.add(st[1], st[2]))
            p.add(st[1], st[2])
        else:
            out.append(g.delete(st[1]))
            p.delete(st[1])
    it.free()
    return out


@pytest.mark.parametrize("vtype,metric", CASES)
def test_batch_iterator_scripts_match_reference(vs, ref, vtype, metric):
    """Order switched between calls, reset midway, drained to exactly label_count results and then an empty next, and the
    index mutated after batch_new / between two nexts (bf_batch_iterator.h:176-189, 209-214) — against the reference's
    own batch iterator on the same script (single- and multi-value)."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(7200 + ci)
    dim, n = DIMS[(ci + 1) % 3], 300
    x = _rows(rng, vtype, n, dim, 1.0 if metric != IP else 1.7)
    multi_labels = np.concatenate([np.arange(1, n // 2 + 1), rng.integers(1, n // 2 + 1, n - n // 2)])
    q = _rows(rng, vtype, 1, dim)[0]
    plain, mutated = _scripts(rng, vtype, dim, n)
    want = {}  # the reference's half first: it is recorded before the device is touched
    with _HalfTier(vtype):
        for multi in (False, True):
            labels = multi_labels if multi else np.arange(1, n + 1)
            for name, steps in (("plain", plain), ("mutated", mutated)):
                r = ol.RefIndex(vtype, dim, metric, multi=multi)
                for b, lab in zip(x, labels.tolist()):
                    assert r.add(b, lab) == 1
                want[multi, name] = r.batch_script(q, steps)
    for multi in (False, True):
        labels = multi_labels if multi else np.arange(1, n + 1)
        for name, steps in (("plain", plain), ("mutated", mutated)):
            g, p = _pair(vs, vtype, dim, metric, multi)
            _add_rows(g, p, x, labels)
            got = _run_script_device(g, p, q, steps)
            for j, (st, a, b) in enumerate(zip(steps, got, want[multi, name])):
                what = (multi, name, j, st[0])
                if st[0] == "next":
                    ai, as_ = _canon(*a)
                    bi, bs = _canon(*b)
                    same(vtype, (ai, as_), (bi, bs), what, open_start=True)
                else:
                    assert a == b, what
            g.close()


# ------------------------------------------------------------------ multi-value indexes
def _multi_rows(rng, vtype, dim, metric):
    """labels 1..250: a tie group (1-2 copies each of one vector: identical rows inside a label and across labels, labels
    ascending in row order, at the front where no swap-delete moves them); labels 251..600: 1-5 rows each in shuffled row
    order"""
    scale = 1.0 if metric != IP else 1.7
    t = _rows(rng, vtype, 1, dim, scale)[0]
    blobs, labels = [], []
    for lab in range(1, 251):
        c = int(rng.integers(1, 3))
        blobs += [t] * c
        labels += [lab] * c
    rest = []
    for lab in range(251, 601):
        rest += [(v, lab) for v in _rows(rng, vtype, int(rng.integers(1, 6)), dim, scale)]
    for i in rng.permutation(len(rest)):
        blobs.append(rest[i][0])
        labels.append(rest[i][1])
    return np.stack(blobs), np.array(labels, dtype=np.uint64), t


def check_multi(vs, vtype, g, p, qs, labels, what):
    lc = len(labels)
    for qi, q in enumerate(qs):
        for k in (1, 10, 129, lc, lc + 1):
            gi, gs, code = g.topk(q, k)
            assert code == 0 and len(set(gi.tolist())) == len(gi)
            same(vtype, (gi, gs), p.topk(q, k), (what, qi, "topk", k), complete=k >= lc)
        check_range(vtype, g, p, q, (what, qi))
        for size in (64, 129):
            drain(vs, vtype, g, p, q, size, (what, qi), orders=(0, 1))
        sq = np.zeros(p.L.orc_stored_size(p.vtype, p.dim, p.metric), dtype=np.uint8)
        sq[: q.nbytes] = np.ascontiguousarray(q).view(np.uint8)
        if p.metric == COS:
            p.L.orc_normalize(ol._p(sq), p.dim, p.vtype)
        probe = np.array(list(labels[::3]) + [10**7], dtype=np.uint64)
        ad = g.adhoc_distances(q, probe)
        for lab, a in zip(probe.tolist(), ad.tolist()):
            b = p.distance_from(lab, sq)
            c = g.distance_from(lab, sq)
            for v in (a, c):
                if np.isnan(b):
                    assert np.isnan(v), (what, lab)
                elif _exact(vtype):
                    assert np.float32(v).tobytes() == np.float32(b).tobytes(), (what, lab)
                else:
                    assert abs(v - b) <= _tol(b), (what, lab)
    for k in (10, 129, lc):
        bl, bs, rc = g.topk_batch(np.stack(qs), k)
        assert rc == 0
        for i, q in enumerate(qs):
            gi, gs, _ = g.topk(q, k)
            m = len(gi)
            assert bl[i, :m].astype(np.int64).tolist() == gi.tolist() and bs[i, :m].tobytes() == gs.tobytes(), (what, k, i)


@pytest.mark.parametrize("vtype,metric", CASES)
def test_multi_value_index_paths(vs, vtype, metric):
    """A multi-value index: top-k at k in {1, 10, 129, label_count, label_count+1} (first occurrence per label in
    (score, row) order), topk_batch equal to the per-query answers, range (best score per label, only labels with a row
    inside the radius), batch iterators drained (no repeats, label_count results), distance_from / adhoc_distances (the
    min over the label's rows) — before and after deletes of multi-vector labels and re-adds."""
    ci = CASES.index((vtype, metric))
    rng = np.random.default_rng(7300 + ci)
    dim = DIMS[ci % 3]
    blobs, labels, t = _multi_rows(rng, vtype, dim, metric)
    g, p = _pair(vs, vtype, dim, metric, multi=True)
    _add_rows(g, p, blobs, labels)
    assert g.size() == p.size() == len(blobs)
    qs = [_rows(rng, vtype, 1, dim)[0], t.copy()]
    live = sorted(set(labels.tolist()))
    check_multi(vs, vtype, g, p, qs, live, "built")
    counts = {lab: int(np.sum(labels == lab)) for lab in live}
    victims = [int(v) for v in rng.choice([lab for lab in live if lab > 250 and counts[lab] > 1], 40, replace=False)]
    for lab in victims:
        assert g.delete(lab) == p.delete(lab) == counts[lab]
    live = [lab for lab in live if lab not in victims]
    for lab in victims[:15] + [900, 901]:
        c = int(rng.integers(1, 4))
        _add_rows(g, p, _rows(rng, vtype, c, dim), [lab] * c)
        live.append(lab)
    live.sort()
    assert g.size() == p.size()
    check_multi(vs, vtype, g, p, qs, live, "after deletes and re-adds")
    g.close()


@pytest.mark.parametrize("vtype", TYPES)
def test_multi_value_distance_nan_rows_match_reference(vs, ref, vtype):
    """A cosine row of zeros is NaN against every query.  The reference folds `(dist < d) ? dist : d` over a label's rows in
    order (brute_force_multi.h:234-238): NaN exactly when the last row is NaN.  distance_from and adhoc_distances (the
    ad-hoc step of hybrid queries) must give the reference's answer."""
    dim = 9
    rng = np.random.default_rng(40 + vtype)  # the rows of test_oracle_vecsim_scan_paths.py::test_multi_value_distance_from_nan_rule
    a, b = _rows(rng, vtype, 2, dim)
    z = np.zeros(dim, dtype=ol.NP_DTYPE[vtype])
    layouts = {1: [a, z], 2: [z, a], 3: [a, z, b], 4: [z, z], 5: [z], 6: [b, a], 7: [z, b, z, a]}
    q = _rows(rng, vtype, 1, dim)[0]
    r = ol.RefIndex(vtype, dim, COS, multi=True)
    p = ol.PortIndex(vtype, dim, COS, multi=True, tier=TIER_AVX512)
    for lab, rows_ in layouts.items():
        for v in rows_:
            assert r.add(v, lab) == 1
            p.add(v, lab)
    sq = np.zeros(p.L.orc_stored_size(vtype, dim, COS), dtype=np.uint8)
    sq[: q.nbytes] = np.ascontiguousarray(q).view(np.uint8)
    p.L.orc_normalize(ol._p(sq), dim, vtype)
    probe = list(layouts) + [99]
    with _HalfTier(vtype):
        want = [r.distance_from(lab, sq) for lab in probe]
    g = vs.VecSimIndex(vtype, dim, COS, multi=True)
    for lab, rows_ in layouts.items():
        for v in rows_:
            assert g.add(v, lab) == 1
    ad = g.adhoc_distances(q, np.array(probe, dtype=np.uint64))
    for lab, w, x in zip(probe, want, ad.tolist()):
        y = g.distance_from(lab, sq)
        o = p.distance_from(lab, sq)
        for v in (x, y, o):
            assert np.isnan(v) == np.isnan(w), (lab, v, w)
            if not np.isnan(w):
                assert abs(v - w) <= (0 if _exact(vtype) else _tol(w)), (lab, v, w)
    assert [bool(np.isnan(w)) for w in want] == [True, False, False, True, True, False, False, True]
    g.close()
