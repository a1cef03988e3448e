"""Many queries' top-k hits in one call (opalb200_db_search_batch_topk) against a loop of single top-k calls
(opalb200_db_search_topk), on the BASELINE configs[2] workload: the 570k-sequence database and its 20 queries, SW,
BLOSUM62 11/1, top-1000, at OPAL_SEARCH_SCORE_END and at OPAL_SEARCH_ALIGNMENT.

  python tools/batch_topk_probe.py [--out FILE]

Per search level the three variants (loop of 20 calls, batch with 3 and with 12 searches in flight) are alternated
twice; every run's indices and records (alignments included) must equal the first loop's.  Times are wall clock around
the calls (each call ends with its records on the host), summed over the loop's 20 calls.  Prints the card name and its power limit."""
import argparse
import os
import subprocess
import sys
import time

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
    db = datasets.config3_db(sm, query=sm.encode(datasets.P18080))
    h = eng.create_db(db, 0)
    queries = datasets.config3_queries(sm)
    k = 1000
    say(f"configs[2]: {len(db)} sequences, {db.total_residues} residues; {len(queries)} queries, SW, BLOSUM62 11/1, top-{k}")

    def loop(st):  # (results, ms inside the calls)
        out, ms = [], 0.0
        for q in queries:
            t0 = time.perf_counter()
            rc, idx, res = h.search_topk(q, 11, 1, sm.flat(), 23, st, "SW", k)
            ms += (time.perf_counter() - t0) * 1e3
            assert rc == 0, eng.last_error()
            out.append((idx.tolist(), records(res)))
            free_alignments(res)
        return out, ms

    def batch(st, in_flight):
        t0 = time.perf_counter()
        rc, idx, res = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, st, "SW", k, in_flight=in_flight)
        ms = (time.perf_counter() - t0) * 1e3
        assert rc == 0, eng.last_error()
        out = [(idx[s].tolist(), records(res[s])) for s in range(len(queries))]
        for r in res:
            free_alignments(r)
        return out, ms

    for st, name in ((1, "SCORE_END"), (2, "ALIGNMENT")):
        batch(st, 12)  # warm-up: contexts, plans, module load
        ref = None
        best = {}
        for rep in range(2):
            for label, run in (("loop of 20", lambda: loop(st)), ("batch, 3 in flight", lambda: batch(st, 3)),
                               ("batch, 12 in flight", lambda: batch(st, 12))):
                out, wall = run()
                if ref is None:
                    ref = out
                else:
                    assert out == ref, f"{name} {label} run {rep}: results differ from the loop"
                best[label] = min(best.get(label, 1e30), wall)
                say(f"  {name} run {rep} {label:20s}: {wall:9.1f} ms")
        say(f"  {name} best: " + ", ".join(f"{label} {ms:.1f} ms" for label, ms in best.items()) +
            f"; batch(12) / loop = {best['batch, 12 in flight'] / best['loop of 20']:.3f}; indices and records identical")
    h.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
