#!/usr/bin/env python
"""Regenerates the fixtures under tests/golden/ that pin the oracle to the reference.

  python tests/golden/make_fixtures.py abi       # needs /root/reference: struct layouts from its headers
  python tests/golden/make_fixtures.py postings  # transcription of the reference's own golden vectors
  python tests/golden/make_fixtures.py reference # needs oracle/_ref: records the reference's answers (tests/golden/reference/)

`postings` does not execute reference code (the posting path is Rust and no Rust toolchain exists
here): the vectors below are copied BY VALUE from the reference's test files, each with its source
file:line, so a reader can diff them against /root/reference.
"""
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
U16, U32 = 0xFFFF, 0xFFFFFFFF

POSTINGS = {
    "_source": "src/redisearch_rs (reference @ 075d9f36)",
    # qint/tests/qint.rs:17-115 — (values, encoded length)
    "qint_lengths": [
        {"values": [3333, 10], "bytes": 4},
        {"values": [1000000000, 70000, 20], "bytes": 9},
        {"values": [2500000000, 90000, 255, 1500000000], "bytes": 13},
        {"values": [0, 0, 0, 0], "bytes": 5},
    ],
    # varint/tests/varint.rs:74-108 (test_u32_encoded_bytes) and :6-16 (lengths)
    "varint_bytes": [
        [0, [0x00]], [1, [0x01]], [127, [0x7F]], [128, [0x80, 0x00]], [129, [0x80, 0x01]], [255, [0x80, 0x7F]],
        [256, [0x81, 0x00]], [16383, [0xFE, 0x7F]], [16384, [0xFF, 0x00]], [16511, [0xFF, 0x7F]],
        [16512, [0x80, 0x80, 0x00]], [2097151, [0xFE, 0xFE, 0x7F]], [2097152, [0xFE, 0xFF, 0x00]],
        [268435455, [0xFE, 0xFE, 0xFE, 0x7F]], [268435456, [0xFE, 0xFE, 0xFF, 0x00]],
        [U32, [0x8E, 0xFE, 0xFE, 0xFE, 0x7F]],
    ],
    "varint_lengths": [[123456789, 4], [987654321, 5], [0, 1], [9, 1]],
    # inverted_index/tests/integration/codec/freqs_only.rs:26-49 — (freq, delta, bytes)
    "freqs_only": [
        [0, 0, [0, 0, 0]], [0, 1, [0, 1, 0]], [2, 0, [0, 0, 2]], [2, 1, [0, 1, 2]], [256, 0, [4, 0, 0, 1]],
        [256, 256, [5, 0, 1, 0, 1]], [2, 65536, [2, 0, 0, 1, 2]], [U16 + 1, U16 + 1, [10, 0, 0, 1, 0, 0, 1]],
        [2, U32, [3, 255, 255, 255, 255, 2]], [U32, U32, [15, 255, 255, 255, 255, 255, 255, 255, 255]],
    ],
    # codec/full.rs:23-55 — (delta, freq, fieldMask, offsets, bytes)
    "full": [
        [0, 1, 1, [1, 2, 3], [0, 0, 1, 1, 3, 1, 2, 3]],
        [10, 5, U32, [1, 2, 3, 4], [48, 10, 5, 255, 255, 255, 255, 4, 1, 2, 3, 4]],
        [256, 1, 1, [1, 2, 3], [1, 0, 1, 1, 1, 3, 1, 2, 3]],
        [65536, 1, 1, [1, 2, 3], [2, 0, 0, 1, 1, 1, 3, 1, 2, 3]],
        [U16, 1, 1, [1, 2, 3], [1, 255, 255, 1, 1, 3, 1, 2, 3]],
        [U32, 1, 1, [1, 2, 3], [3, 255, 255, 255, 255, 1, 1, 3, 1, 2, 3]],
    ],
    # codec/freqs_fields.rs:48-61 — (delta, freq, fieldMask, bytes)
    "freqs_fields": [
        [0, 1, 1, [0, 0, 1, 1]], [10, 5, U32, [48, 10, 5, 255, 255, 255, 255]], [256, 1, 1, [1, 0, 1, 1, 1]],
        [65536, 1, 1, [2, 0, 0, 1, 1, 1]], [U16, 1, 1, [1, 255, 255, 1, 1]], [U32, 1, 1, [3, 255, 255, 255, 255, 1, 1]],
    ],
    # codec/fields_only.rs:44-56 — (delta, fieldMask, bytes)
    "fields_only": [
        [0, 1, [0, 0, 1]], [10, U32, [12, 10, 255, 255, 255, 255]], [256, 1, [1, 0, 1, 1]], [65536, 1, [2, 0, 0, 1, 1]],
        [U16, 1, [1, 255, 255, 1]], [U32, 1, [3, 255, 255, 255, 255, 1]],
        [U32, U32, [15, 255, 255, 255, 255, 255, 255, 255, 255]],
    ],
    # codec/doc_ids_only.rs:18-26 — (delta, bytes)
    "doc_ids_only": [[0, [0]], [10, [10]], [256, [129, 0]], [65536, [130, 255, 0]], [U16, [130, 254, 127]],
                     [U32, [142, 254, 254, 254, 127]]],
    # codec/raw_doc_ids_only.rs:18-26 — (delta, bytes)
    "raw_doc_ids_only": [[0, [0, 0, 0, 0]], [10, [10, 0, 0, 0]], [256, [0, 1, 0, 0]], [65536, [0, 0, 1, 0]],
                         [U16, [255, 255, 0, 0]], [U32, [255, 255, 255, 255]]],
    # rqe_iterators/tests/integration/intersection.rs:59-78 (NUM_CHILDREN_CASES, RESULT_SET_CASES); children are the
    # result set plus 100 ids unique to each child (create_children :30-52)
    "intersection_num_children": [2, 5, 25],
    "intersection_result_sets": [
        [1, 2, 3, 40, 50],
        [5, 6, 7, 24, 25, 46, 47, 48, 49, 50, 51, 234, 2345, 3456, 4567, 5678, 6789, 7890, 8901, 9012, 12345, 23456,
         34567, 45678, 56789],
        [9, 25, 30, 40, 50, 60, 70, 80, 90, 100, 110, 120, 130, 140, 150, 160, 170, 180, 190, 200, 210, 220, 230, 240,
         250],
    ],
    # tests/cpptests/test_cpp_index.cpp:542-601 (testIntersection): two lists of 100000 docs with id steps 4 and 2,
    # expects 50000 hits, docId (count*2+2)*2, aggregate freq 2; SkipTo(8)=OK, Read->12, SkipTo(200000)=OK, Read=EOF
    "cpp_intersection": {"size": 100000, "steps": [4, 2], "hits": 50000, "freq": 2},
    # idf/tests/tests.rs:25-158
    "idf": [[100, 10, 3.0], [0, 1, 1.0], [0, 0, 1.0], [1, 1, 1.0], [1000, 1, 9.0], [1000, 500, 1.0], [1000, 1000, 1.0]],
    "idf_bm25": [[100, 10, 2.2635, 1e-3]],
    # tests/pytests/test_scorers.py:198-221 (BM25STD: 3 docs, both terms in all 3 -> idf ln(1+0.5/3.5); F 10;
    # doc lens 23/35/45; avg 34.33 = 103/3) and :159-178 (BM25: IDF 1.00, F 10, avg len 30, doc scores / slops)
    "bm25std_explain": {"num_docs": 3, "term_docs": 3, "freq": 10, "avg_doc_len": 103.0 / 3.0,
                        "cases": [[23, 0.54, 0.27], [35, 0.52, 0.26], [45, 0.51, 0.26]]},
    "bm25_explain": {"idf": 1.0, "freq": 10, "avg_doc_len": 30.0, "words_bm25": 0.70, "leaf": 0.35,
                     "cases": [[0.5, 1], [1.0, 2], [0.1, 3]]},
}


def abi():
    probe = os.path.join(ROOT, "tests", "abi", "abi_probe.c")
    exe = "/tmp/abi_probe_ref"
    subprocess.run(["gcc", '-DHDR="VecSim/vec_sim.h"', "-I/root/reference/deps/VectorSimilarity/src", probe, "-o", exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    open(os.path.join(HERE, "vecsim_abi_layout.txt"), "w").write(out)
    probe2 = os.path.join(ROOT, "tests", "abi", "ii_abi_probe.c")
    if os.path.exists(probe2):
        R = "/root/reference"
        inc = [f"-I{R}/src", f"-I{R}/deps", f"-I{R}/src/redisearch_rs/headers", f"-I{R}/deps/rmalloc", f"-I{R}/src/buffer",
               f"-I{R}/deps/VectorSimilarity/src", f"-I{R}/src/coord"]
        subprocess.run(["gcc", "-std=gnu11", "-O1", "-w", "-D_GNU_SOURCE", "-DREFERENCE_HEADERS", *inc, probe2, "-o", exe + "2"], check=True)
        out = subprocess.run([exe + "2"], check=True, capture_output=True, text=True).stdout
        open(os.path.join(HERE, "ii_abi_layout.txt"), "w").write(out)


def postings():
    with open(os.path.join(HERE, "postings_golden.json"), "w") as f:
        json.dump(POSTINGS, f, indent=1)


# the modules whose tests take the `ref` fixture
REFERENCE_TESTS = ["test_oracle_vecsim.py", "test_oracle_vecsim_scan_paths.py", "test_oracle_trees.py", "test_oracle_postings.py",
                   "test_hybrid_state_machine.py", "test_vecsim_scan_paths.py"]


def reference():
    """Runs every test that compares with the reference on oracle/_ref itself and writes what it was asked and answered.  A GPU
    test records its reference half before it touches the device, so on a machine without one it fails after recording."""
    env = dict(os.environ, REFERENCE_RECORD="1")
    tests = [os.path.join(ROOT, "tests", t) for t in REFERENCE_TESTS]
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", *tests], env=env, cwd=ROOT)


if __name__ == "__main__":
    {"abi": abi, "postings": postings, "reference": reference}[sys.argv[1]]()
