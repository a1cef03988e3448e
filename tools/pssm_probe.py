"""Matrix search against the same search through a position-specific scoring matrix (PSSM = matrix rows of the query):
the sweep is the same code, only the profile build and the per-search upload differ.

  python tools/pssm_probe.py [--out FILE]

1. BASELINE configs[2]: the 570k-sequence database, its 20 queries x NW / HW / OV, score + end, 12 searches in flight:
   opalb200_db_search_batch_modes (matrix) and opalb200_db_search_batch_pssm, alternated twice; outputs must be equal.
2. BASELINE configs[3]: SW top-1000 with OPAL_SEARCH_ALIGNMENT (opalb200_db_search_topk / _topk_pssm), query P18080.
Prints GCUPS (query residues x database residues / device time of the batch), the PSSM / matrix ratio, the card name
and its power limit."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from opal_b200 import datasets, free_alignments, get_alignment, matrices  # noqa: E402
from opal_b200.handle import OpalB200  # noqa: E402


def records(res):
    return [tuple(int(res[f][i]) for f in ("score", "endLocationQuery", "endLocationTarget", "startLocationQuery",
                                          "startLocationTarget", "alignmentLength")) + (get_alignment(res, i).tobytes(),)
            for i in range(len(res))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()
    say(f"card: {card[0] if card else 'unknown'}")
    eng = OpalB200()
    sm = matrices.blosum62()
    p18080 = sm.encode(datasets.P18080)
    db = datasets.config3_db(sm, query=p18080)
    h = eng.create_db(db, 0)
    queries = datasets.config3_queries(sm)
    searches = [(q, m) for m in ("NW", "HW", "OV") for q in queries]
    qs, modes = [q for q, _ in searches], [m for _, m in searches]
    pssms = [sm.matrix[q.astype(np.int64)].astype(np.int32) for q in qs]
    cells = float(sum(len(q) for q in qs)) * float(db.total_residues)
    say(f"configs[2]: {len(db)} sequences, {db.total_residues} residues; {len(qs)} searches (20 queries x NW/HW/OV), "
        f"score + end, 12 in flight; {cells / 1e12:.2f} T cells per batch")
    # warm-up of both paths (module load, plans, layouts)
    rc, *_ = h.search_batch(qs[:6], 11, 1, sm.flat(), 23, 1, modes[:6], in_flight=12)
    assert rc == 0, eng.last_error()
    rc, *_ = h.search_batch_pssm(pssms[:6], 11, 1, 1, modes[:6], in_flight=12)
    assert rc == 0, eng.last_error()
    best = {"matrix": [], "pssm": []}
    ref = None
    for rep in range(2):
        for kind in ("matrix", "pssm"):
            t0 = time.perf_counter()
            if kind == "matrix":
                rc, S, E, T, ms = h.search_batch(qs, 11, 1, sm.flat(), 23, 1, modes, in_flight=12)
            else:
                rc, S, E, T, ms = h.search_batch_pssm(pssms, 11, 1, 1, modes, in_flight=12)
            wall = (time.perf_counter() - t0) * 1e3
            assert rc == 0, eng.last_error()
            if ref is None:
                ref = (S, E, T)
            else:
                assert all(np.array_equal(a, b) for a, b in zip(ref, (S, E, T))), f"{kind} run {rep}: outputs differ"
            best[kind].append(ms)
            say(f"  run {rep} {kind:6s}: device {ms:9.1f} ms  {cells / ms / 1e6:7.0f} GCUPS   wall {wall:9.1f} ms")
    say("  outputs: matrix and PSSM batches array-equal (scores, end query, end target) in every run")
    m, p = min(best["matrix"]), min(best["pssm"])
    say(f"  best: matrix {cells / m / 1e6:.0f} GCUPS, PSSM {cells / p / 1e6:.0f} GCUPS, PSSM / matrix = {m / p:.3f}")

    # configs[3]: SW, top 1000, alignment
    pq = sm.matrix[p18080.astype(np.int64)].astype(np.int32)
    for rep in range(2):
        t0 = time.perf_counter()
        rc1, i1, r1 = h.search_topk(p18080, 11, 1, sm.flat(), 23, 2, "SW", 1000)
        t1 = time.perf_counter()
        rc2, i2, r2 = h.search_topk_pssm(pq, 11, 1, 2, "SW", 1000, query=p18080)
        t2 = time.perf_counter()
        assert rc1 == rc2 == 0, eng.last_error()
        assert np.array_equal(i1, i2) and records(r1) == records(r2)
        say(f"configs[3] top-1000 SW ALIGNMENT, run {rep}: matrix {(t1 - t0) * 1e3:.1f} ms, PSSM {(t2 - t1) * 1e3:.1f} ms "
            f"(wall, records equal)")
        free_alignments(r1)
        free_alignments(r2)
    h.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
