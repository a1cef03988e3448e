"""Scoring (query, candidate) pairs on the resident database (opalb200_db_search_pairs) against the route that existed
before it: one opalb200_db_search per query with a skip mask that leaves only its candidates.

  python tools/pairs_probe.py [--out FILE] [--queries 1000] [--per 500]

Workload: the BASELINE configs[2] database (570k sequences) is resident.  Each query is a mutated copy (40 - 90 %
identity) of a database entry shorter than 5,000 residues, so query lengths follow the database's Swiss-Prot-shaped
length distribution; its candidates are that entry (its planted homolog) and `per` - 1 random entries.  BLOSUM62, gaps
11 / 1, SW score + end and NW score + end.  Per mode:
  * the pairs call over all queries: device time (CUDA events, first launch to last kernel end, best of three), sum of
    Q x T over the pairs, GCUPS;
  * the skip-mask route on the first 50 queries (wall clock and summed device time) and the pairs call on the same
    50 queries;
  * the bulk path (opalb200_db_search_batch, 3 in flight) for the first 50 queries against the whole database: GCUPS;
  * every pair of the timed call is compared with the full searches' entry (bulk batches of 50 queries).
Prints the card name and its power limit."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from opal_b200 import datasets, matrices  # noqa: E402
from opal_b200.handle import OpalB200  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--per", type=int, default=500)
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
    rng = np.random.default_rng(20261022)
    db = datasets.config3_db(sm)
    n, nq, per = len(db), args.queries, args.per
    src = rng.choice(np.nonzero(db.lengths < 5000)[0], nq, replace=False)
    queries = [datasets.mutate(db.sequence(int(i)), rng.uniform(0.4, 0.9), rng, sm) for i in src]
    qlen = np.array([len(q) for q in queries], dtype=np.int64)
    pt = np.concatenate([np.concatenate([[i], rng.choice(n, per - 1, replace=False)]) for i in src]).astype(np.int32)
    pq = np.repeat(np.arange(nq), per).astype(np.int32)
    cells = int((qlen[pq] * db.lengths[pt]).sum())
    m50 = 50 * per
    cells50 = int((qlen[pq[:m50]] * db.lengths[pt[:m50]]).sum())
    say(f"configs[2]: {n} sequences, {db.total_residues} residues; {nq} queries (lengths median {int(np.median(qlen))}, "
        f"max {qlen.max()}), {per} candidates each = {len(pq)} pairs, {cells / 1e9:.2f} G cells; BLOSUM62 11/1")
    h = eng.create_db(db, 0)
    for mode in ("SW", "NW"):
        say(f"{mode}, score + end:")
        h.search_pairs(queries, pq, pt, 11, 1, sm.flat(), 23, 1, mode)  # warm-up: module load, allocations
        best, wall = 1e30, 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            rc, sc, eq, et, ms = h.search_pairs(queries, pq, pt, 11, 1, sm.flat(), 23, 1, mode)
            wall = min(wall, (time.perf_counter() - t0) * 1e3)
            assert rc == 0, eng.last_error()
            best = min(best, ms)
        stats = h.last_stats()
        say(f"  pairs call, {nq} queries: device {best:.1f} ms, wall {wall:.1f} ms, {cells / best / 1e6:.0f} GCUPS "
            f"(R = {stats['R']}, largest G = {stats['G']}, most passes = {stats['passes']}, re-run at 32 bits: {stats['rerun32']})")

        # where the time goes: the cells the 16-bit sweep runs (every task: passes x G x R rows over T0 + G - 1 columns,
        # two pairs of one query per task, the longer one's columns; the planner's rule for G and passes restated here),
        # and the same call without the candidates longer than 5,000 residues (the longest single tasks)
        R = stats["R"]
        swept = 0
        for q in range(nq):
            g = 1
            while g < 32 and g * R < qlen[q]:
                g *= 2
            passes = -(-int(qlen[q]) // (g * R))
            t = np.sort(db.lengths[pt[q * per:(q + 1) * per]])[::-1]
            t = t[t > 0][::2].astype(np.int64)
            swept += 2 * passes * g * R * int((t + g - 1).sum())
        short = db.lengths[pt] <= 5000
        cells_short = int((qlen[pq[short]] * db.lengths[pt[short]]).sum())
        bs = 1e30
        for _ in range(2):
            rc, _, _, _, ms = h.search_pairs(queries, pq[short], pt[short], 11, 1, sm.flat(), 23, 1, mode)
            assert rc == 0, eng.last_error()
            bs = min(bs, ms)
        say(f"  where the time goes: the sweep runs {swept / 1e9:.1f} G cells for {cells / 1e9:.1f} G real ones ({cells / swept:.2f}: "
            f"rows padded to G x R, fill and drain of G - 1 columns, the shorter member of a task); without the "
            f"{int((~short).sum())} candidates longer than 5,000 residues: {bs:.1f} ms, {cells_short / bs / 1e6:.0f} GCUPS of real cells, "
            f"{cells_short / bs / 1e6 * swept / cells:.0f} GCUPS of swept ones")

        # the skip-mask route on the first 50 queries, then the pairs call on the same pairs
        route_wall, route_dev = 0.0, 0.0
        skip = np.ones(n, dtype=np.uint8)
        for q in range(50):
            cand = pt[q * per:(q + 1) * per]
            skip[cand] = 0
            t0 = time.perf_counter()
            rc, rsc, req, ret, ms = h.search(queries[q], 11, 1, sm.flat(), 23, 1, mode, skip=skip)
            route_wall += (time.perf_counter() - t0) * 1e3
            route_dev += ms
            skip[cand] = 1
            assert rc == 0, eng.last_error()
            sl = slice(q * per, (q + 1) * per)
            assert np.array_equal(rsc[cand], sc[sl]) and np.array_equal(req[cand], eq[sl]) and np.array_equal(ret[cand], et[sl])
        p50, w50 = 1e30, 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            rc, sc50, eq50, et50, ms = h.search_pairs(queries[:50], pq[:m50], pt[:m50], 11, 1, sm.flat(), 23, 1, mode)
            w50 = min(w50, (time.perf_counter() - t0) * 1e3)
            p50 = min(p50, ms)
            assert rc == 0 and np.array_equal(sc50, sc[:m50]) and np.array_equal(eq50, eq[:m50]) and np.array_equal(et50, et[:m50])
        say(f"  skip-mask route, 50 queries: wall {route_wall:.1f} ms ({route_wall / 50:.2f} ms per query), device {route_dev:.1f} ms")
        say(f"  pairs call, same 50 queries: wall {w50:.1f} ms ({w50 / 50:.3f} ms per query), device {p50:.2f} ms, "
            f"{cells50 / p50 / 1e6:.0f} GCUPS; route / pairs wall = {route_wall / w50:.0f}x")

        # bulk path and the check of every pair of the timed call against the full searches
        bulk_ms, bulk_cells = None, None
        for lo in range(0, nq, 50):
            hi = min(nq, lo + 50)
            rc, fsc, feq, fet, ms = h.search_batch(queries[lo:hi], 11, 1, sm.flat(), 23, 1, mode, in_flight=3)
            assert rc == 0, eng.last_error()
            if lo == 0:
                bulk_ms, bulk_cells = ms, int(qlen[:hi].sum()) * int(db.total_residues)
            for q in range(lo, hi):
                sl, cand = slice(q * per, (q + 1) * per), pt[q * per:(q + 1) * per]
                ok = (np.array_equal(fsc[q - lo][cand], sc[sl]) and np.array_equal(feq[q - lo][cand], eq[sl]) and
                      np.array_equal(fet[q - lo][cand], et[sl]))
                assert ok, f"{mode}: pairs of query {q} differ from the full search"
        say(f"  bulk path, first 50 queries over the whole database: {bulk_ms:.1f} ms, {bulk_cells / bulk_ms / 1e6:.0f} GCUPS")
        say(f"  all {len(pq)} pairs of the timed call equal the full searches' entries")
    h.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
