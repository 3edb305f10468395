"""GPU: VecSimB200_HybridTopK replays the HybridIterator state machine of src/iterators/hybrid_reader.c — mode choice
(:668-691), batches mode (prepareResults :372-443 with the batch-size formula :400-404 and alternatingIterate :140-169), the
policy review that restarts the query in ad-hoc mode (:346-370, :430-438) and ad-hoc mode (:289-335).

The oracle below is the same call sequence written against the REFERENCE's own VecSim (oracle/_ref: its batch iterator,
preferAdHocSearch, getDistanceFrom) with a plain sorted docId list as the child; its answers are recorded under tests/golden/reference/.
The device side gets a B200 iterator (the result of a posting-list union) as its child.  Compared: the final mode, the
number of batches, the docIds and the fp32 distance bits."""
import ctypes as C
import math

import numpy as np
import pytest

import oracle_lib as ol

pytestmark = pytest.mark.gpu
STANDARD_KNN, ADHOC, BATCHES, BATCHES_TO_ADHOC = 1, 2, 3, 4


class _Child:
    def __init__(self, ids):
        self.ids, self.pos, self.last = [int(x) for x in ids], 0, 0

    def rewind(self):
        self.pos, self.last = 0, 0

    def read(self):
        if self.pos >= len(self.ids):
            return False
        self.last = self.ids[self.pos]
        self.pos += 1
        return True

    def skip_to(self, doc):
        while self.pos < len(self.ids) and self.ids[self.pos] < doc:
            self.pos += 1
        return self.read()


def _less(a, b):  # cmpVecSimResByScore: score asc; among equal scores the smaller docId compares greater
    return a[0] < b[0] or (a[0] == b[0] and a[1] > b[1])


class _Heap:
    def __init__(self, k):
        self.k, self.v = k, []

    def push(self, h):
        if len(self.v) < self.k:
            self.v.append(h)
        else:
            worst = max(range(len(self.v)), key=lambda i: (self.v[i][0], -self.v[i][1]))
            self.v[worst] = h

    def upper(self):
        return max(self.v, key=lambda h: (h[0], -h[1]))[0]


def oracle_hybrid(ref, is_ref, q_raw, q_norm, k, child_ids, forced=0, batch_size=0):
    L = ol.ref_vecsim() if is_ref else None
    index_size = ref.size()
    child = _Child(child_ids)
    subset = min(len(child_ids), index_size)
    mode = forced or (ADHOC if ref.prefer_adhoc(subset, k, True) else BATCHES)
    heap = _Heap(k)
    iters = 0

    def adhoc():
        heap.v = []
        upper = math.inf
        child.rewind()
        while child.read():
            d = ref.distance_from(child.last, q_norm)
            if d != d:
                continue
            if len(heap.v) < k or d < upper:
                heap.push((np.float32(d), child.last))
                upper = heap.upper()

    if mode == ADHOC:
        adhoc()
    else:
        mode = BATCHES
        it = L.Ref_BatchNew(ref.h, ol._p(np.ascontiguousarray(q_raw))) if is_ref else None
        assert is_ref, "the batches oracle needs the reference's batch iterator"
        upper = math.inf
        est = min(len(child_ids), index_size)
        est_cap = est
        while L.Ref_BatchHasNext(it):
            iters += 1
            n_left = k - len(heap.v)
            bs = batch_size or int(np.float32(n_left) * (np.float32(index_size) / np.float32(est)) + 1)
            ids = np.empty(bs, dtype=np.uint64)
            sc = np.empty(bs, dtype=np.float64)
            m = L.Ref_BatchNext(it, bs, 1, bs, ol._p(ids), ol._p(sc))
            batch = list(zip(ids[:m].tolist(), sc[:m].tolist()))
            child.rewind()
            bi = 0
            cur = None

            def read_in_batch():
                nonlocal bi, cur
                if bi >= len(batch):
                    return False
                cur = batch[bi]
                bi += 1
                return True

            c_ok, v_ok = child.read(), read_in_batch()
            while c_ok and v_ok:
                if cur[0] == child.last:
                    if len(heap.v) < k or cur[1] < upper:
                        heap.push((np.float32(cur[1]), cur[0]))
                        upper = heap.upper()
                    c_ok, v_ok = child.read(), read_in_batch()
                elif cur[0] > child.last:
                    c_ok = child.skip_to(cur[0])
                elif bi < len(batch):
                    v_ok = False
                    while bi < len(batch):
                        cand = batch[bi]
                        bi += 1
                        if child.last > cand[0]:
                            continue
                        cur, v_ok = cand, True
                        break
                else:
                    break
            if len(heap.v) == k:
                break
            change = False
            if not (forced == BATCHES and batch_size):
                new_results = len(heap.v) - (k - n_left)
                cur_ratio = np.float32(new_results) / np.float32(n_left)
                est = (est + int(cur_ratio * np.float32(index_size))) // 2
                est = min(est, est_cap)
                if forced != BATCHES:
                    change = ref.prefer_adhoc(est, k, False)
                est = max(est, 1)
            if change:
                mode = BATCHES_TO_ADHOC
                adhoc()
                break
        L.Ref_BatchFree(it)
    res = sorted(heap.v, key=lambda h: (h[0], h[1]))
    return mode, iters, [h[1] for h in res], np.array([h[0] for h in res], dtype=np.float32)


def farthest_half(ref, q, n):
    """labels 1..n as a bitmap: set for the n // 2 rows the reference ranks farthest from q"""
    all_ids, _ = ref.topk(q, n)
    return np.packbits(np.isin(np.arange(1, n + 1), all_ids[n // 2:]))


@pytest.mark.usefixtures("ref")
@pytest.mark.parametrize("scenario", ["adhoc", "batches", "batches_then_adhoc", "forced_batches_fixed_size", "few_matches"])
def test_hybrid_state_machine_matches_the_reference_call_sequence(scenario):
    from redisearch_b200 import postings as ps
    from redisearch_b200 import vecsim as vs

    n, dim, k = 60_000, 32, 10
    rows = ol.synth_rows(ol.F32, 42, 0, n, dim)
    ref = ol.RefIndex(ol.F32, dim, ol.COS)
    ref.add_many(rows, 1)
    q = ol.synth_rows(ol.F32, 43, 0, 1, dim)[0]
    qn = q.copy()
    ol.port().orc_normalize(ol._p(qn), dim, ol.F32)
    rng = np.random.default_rng(8)
    forced, bsz = 0, 0
    if scenario == "adhoc":
        child_ids = np.sort(rng.choice(np.arange(1, n + 1), n // 20, replace=False))  # 5 %: ad-hoc from the start
    elif scenario == "batches":
        child_ids = np.sort(rng.choice(np.arange(1, n + 1), n // 2, replace=False))  # 50 %, uncorrelated: batches finish
    elif scenario == "batches_then_adhoc":
        # the FARTHEST half: batches keep finding nothing, the review switches
        child_ids = np.flatnonzero(np.unpackbits(ol.reference_call("farthest_half", farthest_half, (ref, q, n)))[:n]) + 1
    elif scenario == "forced_batches_fixed_size":
        child_ids = np.sort(rng.choice(np.arange(1, n + 1), n // 10, replace=False))
        forced, bsz = BATCHES, 500
    else:
        child_ids = np.sort(rng.choice(np.arange(1, n + 1), 4, replace=False))  # fewer matches than k
    exp_mode, exp_iters, exp_ids, exp_sc = ol.reference_call("oracle_hybrid", oracle_hybrid, (ref, True, q, qn, k, child_ids, forced, bsz))

    g = vs.VecSimIndex(vs.VecSimType_FLOAT32, dim, vs.VecSimMetric_Cosine)
    g.add_many(rows, label0=1)

    pl = ps.PostingList.from_arrays(child_ids.astype(np.uint64))
    it = ps.union([pl]).into_iterator()
    qp = vs.VecSimQueryParams()
    qp.searchMode, qp.batchSize = forced, bsz
    labels = np.zeros(k, dtype=np.uint64)
    scores = np.zeros(k, dtype=np.float64)
    cnt, mode, iters = C.c_size_t(0), C.c_int(0), C.c_size_t(0)
    rc = vs.lib().VecSimB200_HybridTopK(g.h, q.ctypes.data, k, C.cast(it, C.c_void_p), C.byref(qp), labels.ctypes.data, scores.ctypes.data,
                                        C.byref(cnt), C.byref(mode), C.byref(iters))
    it.contents.Free(it)
    assert rc == 0
    assert mode.value == exp_mode, (scenario, mode.value, exp_mode)
    if scenario == "adhoc":
        assert mode.value == ADHOC
    if scenario == "batches":
        assert mode.value == BATCHES
    if scenario == "batches_then_adhoc":
        assert mode.value == BATCHES_TO_ADHOC
    assert iters.value == exp_iters, (scenario, iters.value, exp_iters)
    assert labels[:cnt.value].tolist() == exp_ids, (scenario, labels[:cnt.value], exp_ids)
    assert scores[:cnt.value].astype(np.float32).tobytes() == exp_sc.tobytes()
