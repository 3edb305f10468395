"""ctypes loaders for the CHECKERS under oracle/ (test infrastructure; never used by the product).

  port()        oracle/liboracle.so          our CPU restatement (plain C)
  ref_vecsim()  oracle/_ref/libvecsim_ref.so the reference's own VecSim sources, compiled in place
  ref_scorers() oracle/_ref/libscorers_ref.so the reference's src/ext/default.c

oracle/_ref can only be built where the reference's sources are, so what the tests ask of it is recorded once under
tests/golden/reference/ and replayed everywhere (reference_tape, reference_call).
"""
import contextlib
import ctypes as C
import functools
import hashlib
import json
import lzma
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ODIR = os.path.join(ROOT, "oracle")
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "reference")

F32, BF16, F16, I8, U8 = 0, 2, 3, 4, 5
L2, IP, COS = 0, 1, 2
TIER_SCALAR, TIER_AVX512 = 0, 1
NP_DTYPE = {F32: np.float32, BF16: np.uint16, F16: np.uint16, I8: np.int8, U8: np.uint8}

_P, _SZ = C.c_void_p, C.c_size_t
_port = None
_ref = None


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def build_port():
    subprocess.run(["make", "-C", ODIR, "liboracle.so"], check=True, capture_output=True)


def port():
    global _port
    if _port is None:
        path = os.path.join(ODIR, "liboracle.so")
        if not os.path.exists(path):
            build_port()
        L = C.CDLL(path)
        L.orc_distance.restype = C.c_float
        L.orc_distance.argtypes = [C.c_int, C.c_int, _SZ, _P, _P, C.c_int]
        L.orc_normalize.argtypes = [_P, _SZ, C.c_int]
        L.orc_stored_size.restype = _SZ
        L.orc_stored_size.argtypes = [C.c_int, _SZ, C.c_int]
        L.orc_half_to_float.restype = C.c_float
        L.orc_half_to_float.argtypes = [C.c_uint16]
        L.orc_float_to_half.restype = C.c_uint16
        L.orc_float_to_half.argtypes = [C.c_float]
        L.orc_float_to_bf16.restype = C.c_uint16
        L.orc_float_to_bf16.argtypes = [C.c_float]
        L.orc_index_new.restype = _P
        L.orc_index_new.argtypes = [C.c_int, _SZ, C.c_int, C.c_int, C.c_int]
        L.orc_index_free.argtypes = [_P]
        L.orc_index_add.restype = C.c_int
        L.orc_index_add.argtypes = [_P, _P, _SZ]
        L.orc_index_add_bulk.argtypes = [_P, _P, _SZ, _SZ, _SZ]
        L.orc_index_delete.restype = C.c_int
        L.orc_index_delete.argtypes = [_P, _SZ]
        L.orc_index_size.restype = _SZ
        L.orc_index_size.argtypes = [_P]
        L.orc_index_topk.restype = _SZ
        L.orc_index_topk.argtypes = [_P, _P, _SZ, C.c_int, _P, _P]
        L.orc_index_range.restype = _SZ
        L.orc_index_range.argtypes = [_P, _P, C.c_double, C.c_int, _SZ, _P, _P]
        L.orc_index_distance_from.restype = C.c_double
        L.orc_index_distance_from.argtypes = [_P, _SZ, _P]
        L.orc_index_prefer_adhoc.restype = C.c_int
        L.orc_index_prefer_adhoc.argtypes = [_P, _SZ, _SZ, C.c_int]
        L.orc_index_all_sorted.restype = _SZ
        L.orc_index_all_sorted.argtypes = [_P, _P, _P, _P]
        L.orc_index_time_topk.restype = C.c_double
        L.orc_index_time_topk.argtypes = [_P, _P, _SZ, _SZ, _SZ, C.c_int, _P, _P]
        L.orc_scan_topk_chunk.argtypes = [C.c_int, C.c_int, C.c_int, _SZ, _P, _SZ, _SZ, _SZ, _P, _SZ, _SZ, _SZ, C.c_int, _P, _P, _P]
        L.orc_mix64.restype = C.c_uint64
        L.orc_mix64.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
        L.orc_synth_f32.restype = C.c_float
        L.orc_synth_f32.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
        L.orc_synth_rows.argtypes = [C.c_int, C.c_uint64, C.c_uint64, _SZ, _SZ, _P]
        _port = L
    return _port


def ref_vecsim():
    """None when oracle/_ref was not built (no /root/reference on this machine and no prebuilt .so)."""
    global _ref
    if _ref is None:
        path = os.path.join(ODIR, "_ref", "libvecsim_ref.so")
        if not os.path.exists(path):
            return None
        L = C.CDLL(path)
        L.Ref_IndexNew.restype = _P
        L.Ref_IndexNew.argtypes = [C.c_int, _SZ, C.c_int, C.c_int, _SZ]
        L.Ref_IndexFree.argtypes = [_P]
        L.Ref_AddVector.restype = C.c_int
        L.Ref_AddVector.argtypes = [_P, _P, _SZ]
        L.Ref_AddVectors.argtypes = [_P, _P, _SZ, _SZ, _P, _SZ]
        L.Ref_DeleteVector.restype = C.c_int
        L.Ref_DeleteVector.argtypes = [_P, _SZ]
        L.Ref_IndexSize.restype = _SZ
        L.Ref_IndexSize.argtypes = [_P]
        L.Ref_TopK.restype = _SZ
        L.Ref_TopK.argtypes = [_P, _P, _SZ, C.c_int, _SZ, _P, _P, _P]
        L.Ref_Range.restype = _SZ
        L.Ref_Range.argtypes = [_P, _P, C.c_double, C.c_int, _SZ, _P, _P, _P]
        L.Ref_GetDistanceFrom.restype = C.c_double
        L.Ref_GetDistanceFrom.argtypes = [_P, _SZ, _P]
        L.Ref_PreferAdHoc.restype = C.c_int
        L.Ref_PreferAdHoc.argtypes = [_P, _SZ, _SZ, C.c_int]
        L.Ref_BatchNew.restype = _P
        L.Ref_BatchNew.argtypes = [_P, _P]
        L.Ref_BatchNext.restype = _SZ
        L.Ref_BatchNext.argtypes = [_P, _SZ, C.c_int, _SZ, _P, _P]
        L.Ref_BatchHasNext.restype = C.c_int
        L.Ref_BatchHasNext.argtypes = [_P]
        L.Ref_BatchReset.argtypes = [_P]
        L.Ref_BatchFree.argtypes = [_P]
        L.Ref_Distance.restype = C.c_float
        L.Ref_Distance.argtypes = [C.c_int, C.c_int, _SZ, _P, _P]
        L.Ref_Distances.argtypes = [C.c_int, C.c_int, _SZ, _P, _SZ, _SZ, _P, _P]
        L.Ref_Normalize.argtypes = [_P, _SZ, C.c_int]
        L.Ref_ScanTopKChunk.argtypes = [C.c_int, C.c_int, _SZ, _P, _SZ, _SZ, _SZ, _P, _SZ, _SZ, _SZ, C.c_int, _P, _P, _P]
        L.Ref_TimeTopK.restype = C.c_double
        L.Ref_TimeTopK.argtypes = [_P, _P, _SZ, _SZ, _SZ, C.c_int, _P, _P]
        _ref = L
    return _ref


def host_has_avx512f() -> bool:
    try:
        with open("/proc/cpuinfo") as f:
            return " avx512f" in f.read()
    except OSError:
        return False


# ---------------------------------------------------------------------------------------------
# the reference's answers, recorded
# ---------------------------------------------------------------------------------------------
# A test that compares with the reference opens a tape (the `ref` fixture).  While it is open, every call marked @_recorded
# replays the answer stored in tests/golden/reference/<module>/<test>.json.xz.  When the tape closes, a digest of the calls'
# names and arguments (and of REF_CPU_MASK, which picks the reference's SIMD tier) checks that they were the ones the reference
# was asked.  With REFERENCE_RECORD=1 the calls run on oracle/_ref instead and the tape is written
# (tests/golden/make_fixtures.py reference).
_tape = None


def _plain(x):
    if isinstance(x, np.generic):
        return x.item()
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in sorted(x.items())}
    return x


def _feed(h, args):
    def feed(x):
        if isinstance(x, np.ndarray):
            h.update(f"{x.dtype.str}{x.shape}".encode())
            h.update(np.ascontiguousarray(x).tobytes())
        elif isinstance(x, (bytes, bytearray)):
            h.update(bytes(x))
        elif hasattr(x, "_tape_key"):
            feed(x._tape_key())
        elif isinstance(x, (list, tuple)):
            h.update(b"[")
            for v in x:
                feed(v)
            h.update(b"]")
        else:
            h.update(json.dumps(_plain(x)).encode())
        h.update(b"|")

    feed(args)


def _enc(x):
    if isinstance(x, np.ndarray):
        return {"nd": x.dtype.str, "v": x.tolist()}
    if isinstance(x, tuple):
        return {"tuple": [_enc(v) for v in x]}
    if isinstance(x, list):
        return [_enc(v) for v in x]
    return _plain(x)


def _dec(x):
    if isinstance(x, dict):
        if "tuple" in x:
            return tuple(_dec(v) for v in x["tuple"])
        return np.array(x["v"], dtype=x["nd"])
    if isinstance(x, list):
        return [_dec(v) for v in x]
    return x


def _live():
    return _tape is None or _tape["record"]


@contextlib.contextmanager
def reference_tape(module, test):
    """Replays (or, with REFERENCE_RECORD=1, records) the reference's answers for one test."""
    global _tape
    path = os.path.join(GOLDEN_REF, module, test + ".json.xz")
    record = os.environ.get("REFERENCE_RECORD") == "1"
    if record:
        assert ref_vecsim() is not None and ref_scorers() is not None, "recording needs oracle/_ref (build() with the reference at hand)"
        assert host_has_avx512f(), "the recorded answers are those of the reference's AVX-512 tier, which the tests hold the port's to"
        rec = {"calls": [], "digest": None}
    else:
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path}: no recorded reference answers for this test (tests/golden/make_fixtures.py reference)")
        with lzma.open(path, "rt") as f:
            rec = json.load(f)
    _tape = t = {"record": record, "calls": rec["calls"], "pos": 0, "path": path, "depth": 0, "h": hashlib.sha256()}
    try:
        yield
        if not record:
            assert t["pos"] == len(t["calls"]), f"{len(t['calls']) - t['pos']} recorded reference calls were not made: re-record {path}"
            assert t["h"].hexdigest() == rec["digest"], f"the reference calls differ from the recorded ones: re-record {path}"
    finally:
        if record:  # a GPU test records its reference half before it needs the device
            os.makedirs(os.path.dirname(path), exist_ok=True)
            with open(path, "wb") as f:
                f.write(lzma.compress(json.dumps({"digest": t["h"].hexdigest(), "calls": t["calls"]}, separators=(",", ":")).encode(),
                                      preset=9 | lzma.PRESET_EXTREME))
        _tape = None


def reference_call(name, fn, args, kwargs=None):
    """fn(*args, **kwargs) on the reference, or its recorded answer while a tape replays.  An argument with a _tape_key() enters the
    digest through it."""
    kwargs = kwargs or {}
    t = _tape
    if t is None or t["depth"]:
        return fn(*args, **kwargs)
    _feed(t["h"], [name, args, kwargs, os.environ.get("REF_CPU_MASK")])
    if t["record"]:
        t["depth"] += 1
        try:
            out = fn(*args, **kwargs)
        finally:
            t["depth"] -= 1
        t["calls"].append(_enc(out))
        return out
    assert t["pos"] < len(t["calls"]), f"{name}: more reference calls than recorded in {t['path']}"
    t["pos"] += 1
    return _dec(t["calls"][t["pos"] - 1])


def _recorded(fn):
    """Marks a call into oracle/_ref (see reference_call)."""

    @functools.wraps(fn)
    def call(*args, **kwargs):
        return reference_call(fn.__qualname__, fn, args, kwargs)

    return call


@_recorded
def reference_distance(vtype, metric, dim, a, b):
    """the reference's dispatched distance function (the tier REF_CPU_MASK leaves it)"""
    return ref_vecsim().Ref_Distance(vtype, metric, dim, _p(np.ascontiguousarray(a)), _p(np.ascontiguousarray(b)))


@_recorded
def reference_normalize(blob, dim, vtype):
    """a normalised copy of `blob` (bytes of the stored form, with the int8/uint8 norm slot) by the reference's normaliser"""
    out = np.array(blob, copy=True)
    ref_vecsim().Ref_Normalize(_p(out), dim, vtype)
    return out


# ---------------------------------------------------------------------------------------------
# convenience wrappers
# ---------------------------------------------------------------------------------------------
class PortIndex:
    def __init__(self, vtype, dim, metric, multi=False, tier=TIER_AVX512):
        self.L = port()
        self.h = self.L.orc_index_new(vtype, dim, metric, int(multi), tier)
        self.vtype, self.dim, self.metric = vtype, dim, metric

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_index_free(self.h)
            self.h = None

    def add(self, blob, label):
        blob = np.ascontiguousarray(blob)
        return self.L.orc_index_add(self.h, _p(blob), label)

    def add_many(self, blobs, label0=0):
        blobs = np.ascontiguousarray(blobs)
        self.L.orc_index_add_bulk(self.h, _p(blobs), blobs.strides[0], blobs.shape[0], label0)

    def delete(self, label):
        return self.L.orc_index_delete(self.h, label)

    def size(self):
        return self.L.orc_index_size(self.h)

    def topk(self, q, k, order=0):
        q = np.ascontiguousarray(q)
        cap = max(1, min(k, self.size()))
        labels = np.empty(cap, dtype=np.uint64)
        scores = np.empty(cap, dtype=np.float64)
        n = self.L.orc_index_topk(self.h, _p(q), k, order, _p(labels), _p(scores))
        return labels[:n].astype(np.int64), scores[:n]

    def range(self, q, radius, order=0):
        q = np.ascontiguousarray(q)
        cap = max(1, self.size())
        labels = np.empty(cap, dtype=np.uint64)
        scores = np.empty(cap, dtype=np.float64)
        n = self.L.orc_index_range(self.h, _p(q), radius, order, cap, _p(labels), _p(scores))
        return labels[:n].astype(np.int64), scores[:n]

    def distance_from(self, label, q):
        q = np.ascontiguousarray(q)
        return self.L.orc_index_distance_from(self.h, label, _p(q))

    def prefer_adhoc(self, subset, k, initial):
        return bool(self.L.orc_index_prefer_adhoc(self.h, subset, k, int(initial)))

    def all_sorted(self, q):
        q = np.ascontiguousarray(q)
        cap = max(1, self.size())
        labels = np.empty(cap, dtype=np.uint64)
        scores = np.empty(cap, dtype=np.float64)
        n = self.L.orc_index_all_sorted(self.h, _p(q), _p(labels), _p(scores))
        return labels[:n].astype(np.int64), scores[:n]


class RefIndex:
    """The reference's BruteForceIndex through oracle/ref_shim/ref_capi.cpp."""

    def __init__(self, vtype, dim, metric, multi=False, block_size=1024):
        self.L = ref_vecsim() if _live() else None  # a replayed test never touches the library
        self.h = self.L.Ref_IndexNew(vtype, dim, metric, int(multi), block_size) if self.L is not None else None
        self.vtype, self.dim, self.metric, self.multi, self.block_size = vtype, dim, metric, multi, block_size

    def __del__(self):
        if getattr(self, "h", None):
            self.L.Ref_IndexFree(self.h)
            self.h = None

    def _tape_key(self):  # the index's contents enter the digests through the recorded calls that made them
        return ("RefIndex", self.vtype, self.dim, self.metric, int(self.multi), self.block_size)

    @_recorded
    def add(self, blob, label):
        blob = np.ascontiguousarray(blob)
        return self.L.Ref_AddVector(self.h, _p(blob), label)

    @_recorded
    def add_many(self, blobs, label0=0):
        blobs = np.ascontiguousarray(blobs)
        self.L.Ref_AddVectors(self.h, _p(blobs), blobs.shape[0], blobs.strides[0], None, label0)

    @_recorded
    def delete(self, label):
        return self.L.Ref_DeleteVector(self.h, label)

    @_recorded
    def size(self):
        return self.L.Ref_IndexSize(self.h)

    @_recorded
    def topk(self, q, k, order=0):
        q = np.ascontiguousarray(q)
        cap = max(1, k)
        ids = np.empty(cap, dtype=np.uint64)
        scores = np.empty(cap, dtype=np.float64)
        code = C.c_int(0)
        n = self.L.Ref_TopK(self.h, _p(q), k, order, cap, _p(ids), _p(scores), C.byref(code))
        return ids[:n].astype(np.int64), scores[:n]

    @_recorded
    def range(self, q, radius, order=0):
        q = np.ascontiguousarray(q)
        cap = max(1, self.size())
        ids = np.empty(cap, dtype=np.uint64)
        scores = np.empty(cap, dtype=np.float64)
        code = C.c_int(0)
        n = self.L.Ref_Range(self.h, _p(q), radius, order, cap, _p(ids), _p(scores), C.byref(code))
        return ids[:n].astype(np.int64), scores[:n]

    @_recorded
    def distance_from(self, label, q):
        q = np.ascontiguousarray(q)
        return self.L.Ref_GetDistanceFrom(self.h, label, _p(q))

    @_recorded
    def prefer_adhoc(self, subset, k, initial):
        return bool(self.L.Ref_PreferAdHoc(self.h, subset, k, int(initial)))

    @_recorded
    def batches(self, q, n, order=0):
        """Drain a batch iterator n results at a time; returns a list of (ids, scores)."""
        q = np.ascontiguousarray(q)
        it = self.L.Ref_BatchNew(self.h, _p(q))
        out = []
        while self.L.Ref_BatchHasNext(it):
            ids = np.empty(n, dtype=np.uint64)
            scores = np.empty(n, dtype=np.float64)
            m = self.L.Ref_BatchNext(it, n, order, n, _p(ids), _p(scores))
            out.append((ids[:m].astype(np.int64), scores[:m]))
            if m == 0:
                break
        self.L.Ref_BatchFree(it)
        return out

    @_recorded
    def batch_script(self, q, steps):
        """One batch iterator driven by `steps`: ("next", n, order) | ("reset",) | ("has_next",) | ("add", blob, label) |
        ("delete", label), the last two on the index while the iterator lives.  Returns one entry per step: (ids, scores) for
        "next", a bool for "has_next", the return code for "add" / "delete", None for "reset"."""
        q = np.ascontiguousarray(q)
        it = self.L.Ref_BatchNew(self.h, _p(q))
        out = []
        for st in steps:
            if st[0] == "next":
                n = st[1]
                ids = np.empty(max(1, n), dtype=np.uint64)
                scores = np.empty(max(1, n), dtype=np.float64)
                m = self.L.Ref_BatchNext(it, n, st[2], n, _p(ids), _p(scores))
                out.append((ids[:m].astype(np.int64), scores[:m]))
            elif st[0] == "reset":
                self.L.Ref_BatchReset(it)
                out.append(None)
            elif st[0] == "has_next":
                out.append(bool(self.L.Ref_BatchHasNext(it)))
            elif st[0] == "add":
                blob = np.ascontiguousarray(st[1])
                out.append(self.L.Ref_AddVector(self.h, _p(blob), st[2]))
            else:
                out.append(self.L.Ref_DeleteVector(self.h, st[1]))
        self.L.Ref_BatchFree(it)
        return out


class StreamingTopK:
    """k nearest rows of a corpus that is handed over chunk by chunk (stored-form rows, e.g. copied back from the device):
    the reference's own distance kernels + heap when oracle/_ref is built (Ref_ScanTopKChunk), else the C restatement."""

    def __init__(self, vtype, metric, dim, queries_stored_form, k, threads):
        self.vtype, self.metric, self.dim, self.k, self.threads = vtype, metric, dim, k, max(1, threads)
        self.q = np.ascontiguousarray(queries_stored_form)
        nq = self.q.shape[0]
        self.ids = np.zeros((nq, k), dtype=np.uint64)
        self.scores = np.zeros((nq, k), dtype=np.float32)
        self.counts = np.zeros(nq, dtype=np.uint64)
        self.kind = "reference" if ref_vecsim() is not None else "port"

    def feed(self, rows, label0):
        rows = np.ascontiguousarray(rows)
        nq = self.q.shape[0]
        if self.kind == "reference":
            self.ids, self.scores, self.counts = _reference_scan_chunk(self.vtype, self.metric, self.dim, rows, label0, self.q, self.k,
                                                                       self.threads, self.ids, self.scores, self.counts)
        else:
            port().orc_scan_topk_chunk(self.vtype, self.metric, TIER_AVX512, self.dim, _p(rows), rows.strides[0], rows.shape[0], label0,
                                       _p(self.q), self.q.strides[0], nq, self.k, self.threads, _p(self.ids), _p(self.scores),
                                       _p(self.counts))

    def result(self, i):
        """(labels, scores) of query i ordered by (score, label) like a drained reference heap."""
        c = int(self.counts[i])
        order = np.lexsort((self.ids[i, :c], self.scores[i, :c]))
        return self.ids[i, :c][order].astype(np.int64), self.scores[i, :c][order]


@_recorded
def _reference_scan_chunk(vtype, metric, dim, rows, label0, q, k, threads, ids, scores, counts):
    """Ref_ScanTopKChunk: one chunk of rows into the per-query heaps; returns the heaps' new (ids, scores, counts)."""
    ids, scores, counts = ids.copy(), scores.copy(), counts.copy()
    ref_vecsim().Ref_ScanTopKChunk(vtype, metric, dim, _p(rows), rows.strides[0], rows.shape[0], label0, _p(q), q.strides[0], q.shape[0], k,
                                   threads, _p(ids), _p(scores), _p(counts))
    return ids, scores, counts


def synth_rows(vtype, seed, row0, nrows, dim):
    """Counter-based synthetic rows (oracle/vecsim_oracle.c orc_synth_rows)."""
    out = np.empty((nrows, dim), dtype=NP_DTYPE[vtype])
    port().orc_synth_rows(vtype, seed, row0, nrows, dim, _p(out))
    return out


def to_type(x32: np.ndarray, vtype: int) -> np.ndarray:
    """fp32 values -> blobs of `vtype` with the reference's conversions."""
    L = port()
    if vtype == F32:
        return np.ascontiguousarray(x32, dtype=np.float32)
    flat = np.ascontiguousarray(x32, dtype=np.float32).ravel()
    if vtype == F16:
        return np.array([L.orc_float_to_half(float(v)) for v in flat], dtype=np.uint16).reshape(x32.shape)
    if vtype == BF16:
        return np.array([L.orc_float_to_bf16(float(v)) for v in flat], dtype=np.uint16).reshape(x32.shape)
    if vtype == I8:
        return np.rint(127.0 * x32).astype(np.int8)
    return np.rint(127.5 * x32 + 127.5).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# postings / scorers (oracle/postings_oracle.c, scorer_oracle.c, oracle/_ref/libscorers_ref.so)
# ---------------------------------------------------------------------------------------------
(CODEC_FULL, CODEC_FREQS_ONLY, CODEC_FREQS_FIELDS, CODEC_FIELDS_ONLY, CODEC_DOCIDS_ONLY, CODEC_RAW_DOCIDS_ONLY, CODEC_FREQS_OFFSETS,
 CODEC_OFFSETS_ONLY, CODEC_FIELDS_OFFSETS, CODEC_FULL_WIDE, CODEC_FREQS_FIELDS_WIDE, CODEC_FIELDS_ONLY_WIDE,
 CODEC_FIELDS_OFFSETS_WIDE) = range(13)
N_CODECS = 13
CODECS_WITH_OFFSETS = (CODEC_FULL, CODEC_FREQS_OFFSETS, CODEC_OFFSETS_ONLY, CODEC_FIELDS_OFFSETS, CODEC_FULL_WIDE, CODEC_FIELDS_OFFSETS_WIDE)
CODECS_WITH_MASK = (CODEC_FULL, CODEC_FREQS_FIELDS, CODEC_FIELDS_ONLY, CODEC_FIELDS_OFFSETS, CODEC_FULL_WIDE, CODEC_FREQS_FIELDS_WIDE,
                    CODEC_FIELDS_ONLY_WIDE, CODEC_FIELDS_OFFSETS_WIDE)
CODECS_WIDE = (CODEC_FULL_WIDE, CODEC_FREQS_FIELDS_WIDE, CODEC_FIELDS_ONLY_WIDE, CODEC_FIELDS_OFFSETS_WIDE)
CODECS_WITH_FREQ = (CODEC_FULL, CODEC_FREQS_ONLY, CODEC_FREQS_FIELDS, CODEC_FREQS_OFFSETS, CODEC_FULL_WIDE, CODEC_FREQS_FIELDS_WIDE)
SCORER_BM25STD, SCORER_BM25, SCORER_TFIDF, SCORER_TFIDF_DOCNORM, SCORER_DOCSCORE, SCORER_BM25STD_TANH, SCORER_DISMAX = range(7)
SCORER_NAMES = {SCORER_BM25STD: b"BM25STD", SCORER_BM25: b"BM25", SCORER_TFIDF: b"TFIDF",
                SCORER_TFIDF_DOCNORM: b"TFIDF.DOCNORM", SCORER_DOCSCORE: b"DOCSCORE",
                SCORER_BM25STD_TANH: b"BM25STD.TANH", SCORER_DISMAX: b"DISMAX"}


class OrcHit(C.Structure):
    _fields_ = [("doc_id", C.c_uint64), ("n_children", C.c_uint32), ("child_index", C.c_uint32 * 16),
                ("child_freq", C.c_uint32 * 16)]


class OrcScoreDoc(C.Structure):
    _fields_ = [("n_terms", C.c_uint32), ("freq", C.POINTER(C.c_uint32)), ("idf", C.POINTER(C.c_double)),
                ("bm25_idf", C.POINTER(C.c_double)), ("weight", C.POINTER(C.c_double)), ("agg_weight", C.c_double),
                ("doc_len", C.c_uint32), ("max_freq", C.c_uint32), ("doc_score", C.c_float)]


class OrcTree(C.Structure):
    _fields_ = [("n_nodes", C.c_size_t), ("parent", C.c_void_p), ("kind", C.c_void_p), ("freq", C.c_void_p), ("weight", C.c_void_p),
                ("idf", C.c_void_p), ("bm25_idf", C.c_void_p), ("off_start", C.c_void_p), ("off_len", C.c_void_p), ("bytes", C.c_void_p)]


class OrcIndexStats(C.Structure):
    _fields_ = [("num_docs", C.c_uint64), ("num_terms", C.c_uint64), ("avg_doc_len", C.c_double)]


_post_bound = False


def postings():
    """liboracle.so with the postings / scorer prototypes bound."""
    global _post_bound
    L = port()
    if not _post_bound:
        L.orc_qint_encode.restype = _SZ
        L.orc_qint_encode.argtypes = [_P, C.c_int, _P]
        L.orc_qint_decode.restype = _SZ
        L.orc_qint_decode.argtypes = [_P, C.c_int, _P]
        L.orc_varint_encode.restype = _SZ
        L.orc_varint_encode.argtypes = [C.c_uint64, _P]
        L.orc_varint_decode.restype = _SZ
        L.orc_varint_decode.argtypes = [_P, _P]
        L.orc_ii_new.restype = _P
        L.orc_ii_new.argtypes = [C.c_int]
        L.orc_ii_free.argtypes = [_P]
        L.orc_ii_add.restype = _SZ
        L.orc_ii_add.argtypes = [_P, C.c_uint64, C.c_uint32, C.c_uint32, _P, C.c_uint32]
        L.orc_ii_add_wide.restype = _SZ
        L.orc_ii_add_wide.argtypes = [_P, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint64, _P, C.c_uint32]
        L.orc_reader_new_wide.restype = _P
        L.orc_reader_new_wide.argtypes = [_P, C.c_uint64, C.c_uint64]
        L.orc_reader_next_wide.restype = C.c_int
        L.orc_reader_next_wide.argtypes = [_P, _P, _P, _P, _P]
        L.orc_ii_num_blocks.restype = _SZ
        L.orc_ii_num_blocks.argtypes = [_P]
        L.orc_ii_num_docs.restype = _SZ
        L.orc_ii_num_docs.argtypes = [_P]
        L.orc_ii_block.argtypes = [_P, _SZ, _P, _P, _P, _P, _P]
        L.orc_reader_new.restype = _P
        L.orc_reader_new.argtypes = [_P, C.c_uint32]
        L.orc_reader_free.argtypes = [_P]
        L.orc_reader_rewind.argtypes = [_P]
        L.orc_reader_next.restype = C.c_int
        L.orc_reader_next.argtypes = [_P, _P, _P, _P]
        L.orc_reader_seek.restype = C.c_int
        L.orc_reader_seek.argtypes = [_P, C.c_uint64, _P, _P, _P]
        L.orc_intersect.restype = _SZ
        L.orc_intersect.argtypes = [_P, _SZ, _P, _SZ]
        L.orc_union.restype = _SZ
        L.orc_union.argtypes = [_P, _SZ, C.c_int, _P, _SZ]
        L.orc_intersect_skipto.restype = _SZ
        L.orc_intersect_skipto.argtypes = [_P, _SZ, _P, _SZ, _P, _P]
        L.orc_union_skipto.restype = _SZ
        L.orc_union_skipto.argtypes = [_P, _SZ, _P, _SZ, _P, _P]
        L.orc_idf.restype = C.c_double
        L.orc_idf.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_idf_bm25.restype = C.c_double
        L.orc_idf_bm25.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_score.restype = C.c_double
        L.orc_score.argtypes = [C.c_int, C.POINTER(OrcIndexStats), C.POINTER(OrcScoreDoc), C.c_int, C.c_double, C.c_double]
        L.orc_synth_df.restype = C.c_uint64
        L.orc_synth_df.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_synth_member.restype = C.c_int
        L.orc_synth_member.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, _P]
        L.orc_synth_doclen.restype = C.c_uint32
        L.orc_synth_doclen.argtypes = [C.c_uint64]
        L.orc_ii_fill_synth.restype = _SZ
        L.orc_ii_fill_synth.argtypes = [_P, C.c_uint64, C.c_uint64]
        L.orc_within_range.restype = C.c_int
        L.orc_within_range.argtypes = [_SZ, _P, _P, C.c_int, C.c_uint32, C.c_int]
        L.orc_numeric_encode.restype = _SZ
        L.orc_numeric_encode.argtypes = [C.c_uint64, C.c_double, C.c_int, _P]
        L.orc_numeric_decode.restype = _SZ
        L.orc_numeric_decode.argtypes = [_P, _P, _P]
        L.orc_numeric_in_range.restype = C.c_int
        L.orc_numeric_in_range.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int, C.c_int]
        L.orc_min_offset_delta.restype = C.c_int
        L.orc_min_offset_delta.argtypes = [_SZ, _P, _P, _SZ, _P]
        L.orc_score_tree.restype = C.c_double
        L.orc_score_tree.argtypes = [C.c_int, C.POINTER(OrcIndexStats), C.POINTER(OrcTree), C.c_uint32, C.c_uint32, C.c_float, C.c_int,
                                     C.c_double, C.c_double]
        L.orc_tree_offsets.restype = _SZ
        L.orc_tree_offsets.argtypes = [C.POINTER(OrcTree), _SZ, _P, _SZ]
        L.orc_tree_has_offsets.restype = C.c_int
        L.orc_tree_has_offsets.argtypes = [C.POINTER(OrcTree), _SZ]
        L.orc_tree_min_offset_delta.restype = C.c_int
        L.orc_tree_min_offset_delta.argtypes = [C.POINTER(OrcTree)]
        L.orc_tree_within_range.restype = C.c_int
        L.orc_tree_within_range.argtypes = [C.POINTER(OrcTree), C.c_int, C.c_uint32, C.c_int]
        L.orc_time_search3.restype = C.c_double
        L.orc_time_search3.argtypes = [_P, _SZ, _P, C.c_uint64, C.c_double, _SZ, C.c_int, _P, _P, _P]
        _post_bound = True
    return L


_ref_scorers = None


def ref_scorers():
    global _ref_scorers
    if _ref_scorers is None:
        path = os.path.join(ODIR, "_ref", "libscorers_ref.so")
        if not os.path.exists(path):
            return None
        L = C.CDLL(path)
        L.RefScore.restype = C.c_double
        L.RefScore.argtypes = [C.c_char_p, C.c_int, _SZ, _P, _P, _P, _P, C.c_double, C.c_uint32, C.c_uint32, C.c_float,
                               _SZ, C.c_double, C.c_int, C.c_double, C.c_uint64]
        L.RefHamming.restype = C.c_double
        L.RefHamming.argtypes = [C.c_char_p, _SZ, C.c_char_p, _SZ]
        L.RefMinOffsetDelta.restype = C.c_int
        L.RefMinOffsetDelta.argtypes = [C.c_int, _SZ, _P, _P, _SZ, _P]
        L.RefTreeLoad.restype = C.c_int
        L.RefTreeLoad.argtypes = [_SZ, _P, _P, _P, _P, _P, _P, _P, _P, C.c_char_p]
        L.RefTreeMinOffsetDelta.restype = C.c_int
        L.RefTreeHasOffsets.restype = C.c_int
        L.RefTreeHasOffsets.argtypes = [_SZ]
        L.RefTreeOffsets.restype = _SZ
        L.RefTreeOffsets.argtypes = [_SZ, _P, _SZ]
        L.RefTreeExplain.restype = _SZ
        L.RefTreeExplain.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_float, _SZ, C.c_double, C.c_int, C.c_double, C.c_uint64, _P, _P, _SZ]
        L.RefTreeScore.restype = C.c_double
        L.RefTreeScore.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_float, _SZ, C.c_double, C.c_int, C.c_double, C.c_uint64]
        _ref_scorers = L
    return _ref_scorers


class InvIndex:
    """oracle InvertedIndex + helpers."""

    def __init__(self, codec, doc_ids=None, freqs=None, masks=None):
        self.L = postings()
        self.codec = codec
        self.h = self.L.orc_ii_new(codec)
        if doc_ids is not None:
            for i, d in enumerate(doc_ids):
                self.add(int(d), int(freqs[i]) if freqs is not None else 1, int(masks[i]) if masks is not None else 1)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_ii_free(self.h)
            self.h = None

    def add(self, doc_id, freq=1, mask=1, offsets=b""):
        buf = (C.c_uint8 * max(1, len(offsets))).from_buffer_copy(offsets or b"\0")
        return self.L.orc_ii_add_wide(self.h, doc_id, freq, mask & 0xFFFFFFFFFFFFFFFF, mask >> 64, buf, len(offsets))

    def num_docs(self):
        return self.L.orc_ii_num_docs(self.h)

    def blocks(self):
        out = []
        for b in range(self.L.orc_ii_num_blocks(self.h)):
            first, last, n = C.c_uint64(), C.c_uint64(), C.c_uint16()
            buf, ln = C.POINTER(C.c_uint8)(), C.c_size_t()
            self.L.orc_ii_block(self.h, b, C.byref(first), C.byref(last), C.byref(n), C.byref(buf), C.byref(ln))
            out.append((first.value, last.value, n.value, bytes(buf[: ln.value])))
        return out

    def reader(self, mask=0):
        return self.L.orc_reader_new_wide(self.h, mask & 0xFFFFFFFFFFFFFFFF, mask >> 64)

    def read_all(self, mask=0):
        """[(docId, freq, fieldMask)]; the mask is 128 bits wide for the *Wide codecs, its low 32 bits otherwise"""
        r = self.reader(mask)
        d, f, lo, hi = C.c_uint64(), C.c_uint32(), C.c_uint64(), C.c_uint64()
        wide = self.codec in CODECS_WIDE
        out = []
        while self.L.orc_reader_next_wide(r, C.byref(d), C.byref(f), C.byref(lo), C.byref(hi)):
            out.append((d.value, f.value, (lo.value | (hi.value << 64)) if wide else (lo.value & 0xFFFFFFFF)))
        self.L.orc_reader_free(r)
        return out


def within_range(offset_bytes, max_slop, in_order):
    """proximity.rs is_within_range for term children; offset_bytes: list of bytes objects (varint deltas), max_slop None = no limit"""
    n = len(offset_bytes)
    bufs = [(C.c_uint8 * max(1, len(b))).from_buffer_copy(b or b"\0") for b in offset_bytes]
    ptrs = (C.c_void_p * n)(*[C.cast(b, C.c_void_p) for b in bufs])
    lens = (C.c_size_t * n)(*[len(b) for b in offset_bytes])
    return bool(postings().orc_within_range(n, ptrs, lens, 0 if max_slop is None else 1, 0 if max_slop is None else max_slop, int(in_order)))


def numeric_encode(delta, value, compress=False):
    out = (C.c_uint8 * 24)()
    n = postings().orc_numeric_encode(delta, value, int(compress), out)
    return bytes(out[:n])


def numeric_decode(data):
    buf = (C.c_uint8 * (len(data) + 16)).from_buffer_copy(bytes(data) + b"\0" * 16)
    d, v = C.c_uint64(), C.c_double()
    n = postings().orc_numeric_decode(buf, C.byref(d), C.byref(v))
    return n, d.value, v.value


def numeric_blocks(doc_ids, values, compress=False, per_block=100):
    """IndexBlocks of a numeric inverted index (index/core.rs:235-358 with the Numeric encoder: duplicates allowed, 100 entries per
    block, delta from the previous docId, a fresh block when the delta needs more than 7 bytes): [(first, last, n, bytes)]"""
    blocks, cur, first, last, n = [], b"", 0, 0, 0
    for d, v in zip(doc_ids, values):
        d = int(d)
        if n == 0 or (n >= per_block and d != last) or (d - last) >> 56:  # take_block: a full block is left for a NEW document only
            if n:
                blocks.append((first, last, n, cur))
            cur, first, last, n = b"", d, d, 0
        cur += numeric_encode(d - last, float(v), compress)
        last = d
        n += 1
    if n:
        blocks.append((first, last, n, cur))
    return blocks


def _slop_args(positions, virtual):
    n = len(positions)
    stride = max(1, max((len(p) for p in positions), default=1))
    npos = (C.c_uint32 * n)(*[len(p) for p in positions])
    flat = (C.c_uint32 * (n * stride))()
    for i, p in enumerate(positions):
        for j, v in enumerate(p):
            flat[i * stride + j] = v
    virt = (C.c_int * n)(*[int(bool(v)) for v in (virtual or [0] * n)])
    return n, npos, flat, stride, virt


def min_offset_delta(positions, virtual=None):
    """oracle GetSlop (IndexResult_MinOffsetDelta) over an aggregate of term leaves; positions: list of position lists"""
    n, npos, flat, stride, virt = _slop_args(positions, virtual)
    return postings().orc_min_offset_delta(n, npos, flat, stride, virt)


@_recorded
def reference_min_offset_delta(positions, virtual=None, is_union=False):
    """the reference's own src/index_result/index_result.c:51-108 (compiled in place into libscorers_ref.so)"""
    n, npos, flat, stride, virt = _slop_args(positions, virtual)
    return ref_scorers().RefMinOffsetDelta(int(is_union), n, npos, flat, stride, virt)


@_recorded
def reference_hamming(payload, qdata):
    """the reference's HammingDistanceScorer (src/ext/default.c:475-497); payload None = the document has no payload"""
    return ref_scorers().RefHamming(payload, len(payload) if payload else 0, qdata, len(qdata))


def run_intersect(indexes, union=False, quick=False):
    """Full iteration; returns list of (docId, [(orig_child, freq), ...])."""
    L = postings()
    readers = [ix.reader() for ix in indexes]
    arr = (C.c_void_p * len(readers))(*readers)
    cap = max(1, sum(ix.num_docs() for ix in indexes) if union else min(ix.num_docs() for ix in indexes))
    hits = (OrcHit * cap)()
    if union:
        n = L.orc_union(arr, len(readers), int(quick), hits, cap)
    else:
        n = L.orc_intersect(arr, len(readers), hits, cap)
    out = [(hits[i].doc_id, [(hits[i].child_index[j], hits[i].child_freq[j]) for j in range(hits[i].n_children)]) for i in range(n)]
    for r in readers:
        L.orc_reader_free(r)
    return out


def oracle_score(scorer, freqs, idf, bm25_idf, weights, agg_weight, doc_len, max_freq, doc_score, num_docs, avg_doc_len,
                 slop=1, min_score=0.0, tanh_factor=4.0):
    L = postings()
    n = len(freqs)
    fa = (C.c_uint32 * n)(*freqs)
    ia = (C.c_double * n)(*idf)
    ba = (C.c_double * n)(*bm25_idf)
    wa = (C.c_double * n)(*weights)
    d = OrcScoreDoc(n, fa, ia, ba, wa, agg_weight, doc_len, max_freq, doc_score)
    st = OrcIndexStats(num_docs, 0, avg_doc_len)
    return L.orc_score(scorer, C.byref(st), C.byref(d), slop, min_score, tanh_factor)


@_recorded
def reference_score(scorer, freqs, idf, bm25_idf, weights, agg_weight, doc_len, max_freq, doc_score, num_docs,
                    avg_doc_len, slop=1, min_score=0.0, tanh_factor=4, is_union=False):
    L = ref_scorers()
    n = len(freqs)
    fa = (C.c_uint32 * n)(*freqs)
    ia = (C.c_double * n)(*idf)
    ba = (C.c_double * n)(*bm25_idf)
    wa = (C.c_double * n)(*weights)
    return L.RefScore(SCORER_NAMES[scorer], int(is_union), n, fa, ia, ba, wa, agg_weight, doc_len, max_freq, doc_score,
                      num_docs, avg_doc_len, slop, min_score, int(tanh_factor))


# ---- result trees (nested aggregates): tree_oracle.c and the reference's own code over the same flattened arrays ----
KIND_TERM, KIND_AND, KIND_OR, KIND_VIRTUAL, KIND_NUMERIC = range(5)


def varint_deltas(positions):
    """ascending term positions -> the offsets payload of a record (RS/varint deltas)"""
    buf = (C.c_uint8 * 16)()
    out, last = bytearray(), 0
    for p in positions:
        n = postings().orc_varint_encode(int(p) - last, buf)
        out += bytes(buf[:n])
        last = int(p)
    return bytes(out)


class ResultTree:
    """One document's result as the scorers see it.  Nodes are dicts:
         {"kind": KIND_TERM, "freq", "weight", "idf", "bm25_idf", "positions": [...]}   (positions may be empty / absent)
         {"kind": KIND_AND | KIND_OR, "weight", "children": [...]}                      (freq = sum of the children's)
         {"kind": KIND_VIRTUAL | KIND_NUMERIC, "freq", "weight"}"""

    def __init__(self, root):
        self.nodes = []
        self._flatten(root, -1)
        n = len(self.nodes)
        self.parent = np.array([x[0] for x in self.nodes], dtype=np.int32)
        self.kind = np.array([x[1] for x in self.nodes], dtype=np.int32)
        self.freq = np.array([x[2] for x in self.nodes], dtype=np.uint32)
        self.weight = np.array([x[3] for x in self.nodes], dtype=np.float64)
        self.idf = np.array([x[4] for x in self.nodes], dtype=np.float64)
        self.bm25 = np.array([x[5] for x in self.nodes], dtype=np.float64)
        blobs = [x[6] for x in self.nodes]
        self.off_len = np.array([len(b) for b in blobs], dtype=np.uint32)
        self.off_start = np.concatenate([[0], np.cumsum(self.off_len)[:-1]]).astype(np.uint32) if n else np.zeros(0, np.uint32)
        self.bytes = b"".join(blobs) + b"\0"
        self._buf = C.create_string_buffer(self.bytes, len(self.bytes))
        self.c = OrcTree(n, _p(self.parent), _p(self.kind), _p(self.freq), _p(self.weight), _p(self.idf), _p(self.bm25),
                         _p(self.off_start), _p(self.off_len), C.cast(self._buf, C.c_void_p))

    def _flatten(self, node, parent):
        me = len(self.nodes)
        k = node["kind"]
        if k in (KIND_AND, KIND_OR):
            self.nodes.append(None)
            total = 0
            for ch in node["children"]:
                total += self._flatten(ch, me)
            self.nodes[me] = (parent, k, total, node.get("weight", 1.0), 0.0, 0.0, b"")
            return total
        blob = varint_deltas(node.get("positions", ())) if k == KIND_TERM else b""
        self.nodes.append((parent, k, node.get("freq", 1), node.get("weight", 1.0), node.get("idf", 0.0), node.get("bm25_idf", 0.0), blob))
        return node.get("freq", 1)

    # the C restatement
    def score(self, scorer, doc_len, max_freq, doc_score, num_docs, avg_doc_len, slop=-1, min_score=0.0, tanh_factor=4.0):
        st = OrcIndexStats(num_docs, 0, avg_doc_len)
        return postings().orc_score_tree(scorer, C.byref(st), C.byref(self.c), doc_len, max_freq, doc_score, slop, min_score, tanh_factor)

    def offsets(self, node=0):
        out = np.zeros(4096, dtype=np.uint32)
        n = postings().orc_tree_offsets(C.byref(self.c), node, _p(out), out.size)
        return out[:n].tolist()

    def has_offsets(self, node=0):
        return bool(postings().orc_tree_has_offsets(C.byref(self.c), node))

    def min_offset_delta(self):
        return postings().orc_tree_min_offset_delta(C.byref(self.c))

    def within_range(self, max_slop, in_order):
        return bool(postings().orc_tree_within_range(C.byref(self.c), 0 if max_slop is None else 1, 0 if max_slop is None else max_slop,
                                                     int(in_order)))

    # the reference's own code (libscorers_ref.so)
    def _tape_key(self):
        return (self.parent, self.kind, self.freq, self.weight, self.idf, self.bm25, self.bytes)

    def _ref_load(self):
        L = ref_scorers()
        rc = L.RefTreeLoad(len(self.nodes), _p(self.parent), _p(self.kind), _p(self.freq), _p(self.weight), _p(self.idf), _p(self.bm25),
                           _p(self.off_start), _p(self.off_len), C.cast(self._buf, C.c_char_p))
        assert rc == 0
        return L

    @_recorded
    def ref_score(self, scorer, doc_len, max_freq, doc_score, num_docs, avg_doc_len, slop=-1, min_score=0.0, tanh_factor=4):
        return self._ref_load().RefTreeScore(SCORER_NAMES[scorer], doc_len, max_freq, doc_score, num_docs, avg_doc_len, slop, min_score,
                                             int(tanh_factor))

    @_recorded
    def ref_explain(self, scorer, doc_len, max_freq, doc_score, num_docs, avg_doc_len, slop=-1, min_score=0.0, tanh_factor=4):
        """(score, explanation) of the reference's scorer run with scrExp set; one "<depth> <string>" line per node, pre-order"""
        L = self._ref_load()
        buf = C.create_string_buffer(1 << 16)
        sc = C.c_double(0)
        L.RefTreeExplain(SCORER_NAMES[scorer], doc_len, max_freq, doc_score, num_docs, avg_doc_len, slop, min_score, int(tanh_factor),
                         C.byref(sc), buf, len(buf))
        return sc.value, buf.value.decode()

    @_recorded
    def ref_offsets(self, node=0):
        L = self._ref_load()
        out = np.zeros(4096, dtype=np.uint32)
        n = L.RefTreeOffsets(node, _p(out), out.size)
        return out[:n].tolist()

    @_recorded
    def ref_has_offsets(self, node=0):
        return bool(self._ref_load().RefTreeHasOffsets(node))

    @_recorded
    def ref_min_offset_delta(self):
        return self._ref_load().RefTreeMinOffsetDelta()
