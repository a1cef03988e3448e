#!/usr/bin/env python
"""Generate tests/golden/*.json by running the UNMODIFIED reference (oracle/_ref/libopal_ref.so,
compiled from /root/reference/src/opal.cpp by oracle/Makefile) in the build container.

Run:  make -C oracle && python tests/golden/make_golden.py
The GPU box has no /root/reference; it only reads the committed JSON files.

Vectors (each one also names the reference fixture it comes from):
  readme.json    README.md:33-66 example, 4 modes x 3 search types x 2 overflow methods
  config1.json   BASELINE configs[0]: test_data/query/O74807.fasta vs test_data/db/uniprot_sprot15.fasta,
                 BLOSUM50 3/1, SW, search types 0/1/2 (sequences embedded as alphabet indices)
  testcpp.json   src/test.cpp:35-99 inputs (glibc srand(42)), 4 modes, OPAL_SEARCH_ALIGNMENT,
                 OPAL_OVERFLOW_SIMPLE: per-target score/end/start + alignment digest, and `Maximum`
  protein.json   seeded random protein DB (BLOSUM62 11/1), 4 modes score+end; SW alignments
  api.json       reuse rule, CharSW, invalid mode (SURVEY.md section 4, probes B-D)
  oracle_vs_ref.json
                 every call tests/test_oracle_vs_ref.py compares (seeded random protein and small-alphabet cases,
                 score+end, SW alignments, per-target NW/HW/OV alignments): (rc, records), null where the
                 reference crashed.  `python tests/golden/make_golden.py oracle_vs_ref` writes this file alone.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from _util import (MODES, OPAL_OVERFLOW_BUCKETS, OPAL_OVERFLOW_SIMPLE, README_DB, README_MATRIX,  # noqa: E402
                   README_QUERY, REF_SO, OpalCLibrary, SequenceDB, dump_results, free_alignments,
                   glibc_testcpp_data, new_results, run_forked, search_dump)
from opal_b200 import datasets, matrices  # noqa: E402

REFROOT = "/root/reference"


def save(name, obj):
    with open(os.path.join(HERE, name), "w") as f:
        json.dump(obj, f, separators=(",", ":"))
    print("wrote", name, os.path.getsize(os.path.join(HERE, name)), "bytes")


def main():
    ref = OpalCLibrary(REF_SO)

    # ---- README example
    db = SequenceDB.from_sequences(README_DB)
    out = {}
    for m, code in MODES.items():
        for st in (0, 1, 2):
            for ovf in (OPAL_OVERFLOW_SIMPLE, OPAL_OVERFLOW_BUCKETS):
                rc, d = search_dump(ref, README_QUERY, db, 3, 1, README_MATRIX, 4, st, code, ovf)
                out[f"{m}/{st}/{ovf}"] = {"rc": rc, "results": d}
    save("readme.json", out)

    # ---- config 1
    b50 = matrices.blosum50()
    q = datasets.read_fasta(f"{REFROOT}/test_data/query/O74807.fasta", b50)[0]
    seqs = datasets.read_fasta(f"{REFROOT}/test_data/db/uniprot_sprot15.fasta", b50)
    db = SequenceDB.from_sequences(seqs)
    out = {"query": q.tolist(), "db": [s.tolist() for s in seqs], "gapOpen": 3, "gapExt": 1, "matrix": "blosum50"}
    for st in (0, 1, 2):
        rc, d = search_dump(ref, q, db, 3, 1, b50.flat(), 24, st, MODES["SW"], OPAL_OVERFLOW_BUCKETS)
        out[f"SW/{st}"] = {"rc": rc, "results": d}
    # the other three modes on the same data, score+end (alignment stage of the reference is unsafe there)
    for m in ("NW", "HW", "OV"):
        rc, d = search_dump(ref, q, db, 3, 1, b50.flat(), 24, 1, MODES[m], OPAL_OVERFLOW_BUCKETS)
        out[f"{m}/1"] = {"rc": rc, "results": d}
    save("config1.json", out)

    # ---- the reference's own self-test inputs
    tq, tdb = glibc_testcpp_data()
    tm = matrices.simple(4, 3, -1).flat()
    out = {}
    for m, code in MODES.items():
        r = run_forked(lambda: search_dump(ref, tq, tdb, 11, 1, tm, 4, 2, code, OPAL_OVERFLOW_SIMPLE, digest=True))
        assert r is not None, f"reference died in its own self-test, mode {m}"
        rc, d = r
        out[m] = {"rc": rc, "maximum": max(max(x[1] for x in d), 0), "results": d}
        print(m, "Maximum:", out[m]["maximum"])
    save("testcpp.json", out)

    # ---- seeded random protein DB
    b62 = matrices.blosum62()
    rng = np.random.default_rng(7)
    pq = datasets.random_residues(57, rng, b62)
    lens = np.concatenate([rng.integers(1, 12, 24), rng.integers(12, 300, 72)])
    seqs = [datasets.random_residues(int(n), rng, b62) for n in lens]
    for i in range(0, 96, 7):  # a few homologs so SW/OV scores are not all tiny
        seqs[i] = datasets.mutate(pq, 0.8, rng, b62)
    db = SequenceDB.from_sequences(seqs)
    out = {"query": pq.tolist(), "db": [s.tolist() for s in seqs], "gapOpen": 11, "gapExt": 1, "matrix": "blosum62"}
    for m, code in MODES.items():
        for st in (0, 1):
            rc, d = search_dump(ref, pq, db, 11, 1, b62.flat(), 23, st, code, OPAL_OVERFLOW_BUCKETS)
            out[f"{m}/{st}"] = {"rc": rc, "results": d}
    rc, d = search_dump(ref, pq, db, 11, 1, b62.flat(), 23, 2, MODES["SW"], OPAL_OVERFLOW_BUCKETS)
    out["SW/2"] = {"rc": rc, "results": d}
    save("protein.json", out)

    # ---- API semantics: reuse rule, CharSW, invalid mode
    out = {}
    db = SequenceDB.from_sequences(README_DB)
    res = new_results(4)
    ref.search_database(README_QUERY, db, 3, 1, README_MATRIX, 4, res, 0, MODES["SW"], OPAL_OVERFLOW_SIMPLE)
    res["score"][1] = 9999  # poison: a rerun at the same level must keep it
    ref.search_database(README_QUERY, db, 3, 1, README_MATRIX, 4, res, 0, MODES["SW"], OPAL_OVERFLOW_SIMPLE)
    out["reuse_score_then_score"] = dump_results(res)
    ref.search_database(README_QUERY, db, 3, 1, README_MATRIX, 4, res, 1, MODES["SW"], OPAL_OVERFLOW_SIMPLE)
    out["reuse_then_score_end"] = dump_results(res)
    ref.search_database(README_QUERY, db, 3, 1, README_MATRIX, 4, res, 2, MODES["SW"], OPAL_OVERFLOW_SIMPLE)
    out["reuse_then_alignment"] = dump_results(res)
    free_alignments(res)
    big = np.array([2, -1, -3, 0, -1, 4, -5, -1, -3, -5, 1, -10, 0, -1, -10, 40], dtype=np.int32)
    cq = np.array([3] * 6 + [0, 1, 2], dtype=np.uint8)
    cdb = SequenceDB.from_sequences([[3] * 6, [0, 1, 2, 0], [3, 3, 0, 1], [2, 2, 2]])
    res = new_results(4)
    rc, res = ref.search_database_char_sw(cq, cdb, 3, 1, big, 4, res)
    out["char_sw"] = {"rc": rc, "results": dump_results(res, with_alignment=False),
                      "query": cq.tolist(), "db": [cdb.sequence(i).tolist() for i in range(4)], "matrix": big.tolist()}
    res = new_results(4)
    rc, res = ref.search_database(README_QUERY, db, 3, 1, README_MATRIX, 4, res, 0, 7, OPAL_OVERFLOW_SIMPLE)
    out["invalid_mode"] = {"rc": rc, "results": dump_results(res)}
    save("api.json", out)
    oracle_vs_ref(ref)


def oracle_vs_ref(ref):
    from test_oracle_vs_ref import all_cases, run_reference
    save("oracle_vs_ref.json", {key: run_reference(ref, args) for key, args in all_cases()})


if __name__ == "__main__":
    if sys.argv[1:] == ["oracle_vs_ref"]:
        oracle_vs_ref(OpalCLibrary(REF_SO))
    else:
        main()
