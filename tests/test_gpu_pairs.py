"""GPU tests of opalb200_db_search_pairs[_results]: a list of (query, database entry) pairs scored on the resident
database.  Pair p must be exactly entry pairTarget[p] of the full search of queries[pairQuery[p]] -- scores, end
locations, records at every search level -- and what the oracle gives against a one-sequence database; with repeated
and shuffled pairs, many queries per call, several passes, 32-bit re-runs, several devices and the argument errors."""
import ctypes

import numpy as np
import pytest

from _util import MODES, SequenceDB, dump_results, free_alignments
from opal_b200 import datasets, matrices

pytestmark = pytest.mark.gpu

OPAL_ERR_INVALID_MODE, OPAL_ERR_INVALID_ARGUMENT = 3, 4
GO, GE = 11, 1


def _db(rng, sm, planted, n=400):
    """Random targets of 1 - 420 residues with planted homologs of every query, three zero-length targets and one of
    4,000 residues."""
    seqs = [datasets.random_residues(int(x), rng, sm) for x in rng.integers(1, 420, n)]
    for k, q in enumerate(p for p in planted if len(p) > 0):
        for j in range(3):
            seqs[11 * k + 37 * j + 1] = datasets.mutate(q, 0.75, rng, sm)
    for i in (7, 150, 299):
        seqs[i] = np.zeros(0, np.uint8)
    seqs[42] = datasets.random_residues(4000, rng, sm)
    return SequenceDB.from_sequences(seqs)


def _queries(rng, sm):
    """Q = 0 and 1, ~130 rows, and 1,300 rows (several passes)."""
    return [datasets.random_residues(n, rng, sm) for n in (130, 0, 1, 1300, 128, 133, 131, 129)]


def _pairs(rng, nq, n, per=60, extra=(7, 150, 299, 42, 1, 38)):
    """Every query against a random sample of targets (the empty ones, the longest and planted ones included), some
    pairs repeated, all shuffled so that queries of different lengths are interleaved."""
    pq, pt = [], []
    for q in range(nq):
        t = np.concatenate([rng.choice(n, per, replace=False), extra])
        pq += [q] * len(t)
        pt += t.tolist()
    pq, pt = np.array(pq), np.array(pt)
    again = rng.choice(len(pq), 40, replace=False)
    pq, pt = np.concatenate([pq, pq[again]]), np.concatenate([pt, pt[again]])
    perm = rng.permutation(len(pq))
    return pq[perm].astype(np.int32), pt[perm].astype(np.int32)


def _setup(seed):
    rng = np.random.default_rng(seed)
    sm = matrices.blosum62()
    queries = _queries(rng, sm)
    db = _db(rng, sm, queries)
    pq, pt = _pairs(rng, len(queries), len(db))
    return rng, sm, queries, db, pq, pt


def _full(h, queries, sm, st, mode):
    out = []
    for q in queries:
        rc, sc, eq, et, _ = h.search(q, GO, GE, sm.flat(), 23, st, mode)
        assert rc == 0, h.eng.last_error()
        out.append((sc, eq, et))
    return out


@pytest.mark.parametrize("st", [0, 1])
@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pairs_equal_full_search(product, mode, st):
    _, sm, queries, db, pq, pt = _setup(301)
    h = product.create_db(db, 0)
    try:
        full = _full(h, queries, sm, st, mode)
        rc, sc, eq, et, ms = h.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, st, mode)
        assert rc == 0, product.last_error()
        assert ms > 0
        for a, got in enumerate((sc, eq, et)):
            want = np.array([full[q][a][t] for q, t in zip(pq, pt)])
            assert np.array_equal(got, want), (mode, st, a, np.nonzero(got != want)[0][:5])
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pair_records_equal_full_search_records(product, mode):
    _, sm, queries, db, pq, pt = _setup(302)
    h = product.create_db(db, 0)
    try:
        for st in (0, 1, 2):
            want = []
            for q in queries:
                rc, res = h.search_results(q, GO, GE, sm.flat(), 23, st, mode)
                assert rc == 0, product.last_error()
                want.append(dump_results(res))
                free_alignments(res)
            rc, res = h.search_pairs_results(queries, pq, pt, GO, GE, sm.flat(), 23, st, mode)
            assert rc == 0, product.last_error()
            got = dump_results(res)
            free_alignments(res)
            for p in range(len(pq)):
                assert got[p] == want[pq[p]][pt[p]], (mode, st, p, int(pq[p]), int(pt[p]))
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pairs_against_the_oracle_on_one_sequence_databases(product, oracle, mode):
    """Score and end location against opalSearchDatabase of the oracle over a database of the pair's target alone (SW
    reports no end location for a score of 0)."""
    rng, sm, queries, db, pq, pt = _setup(303)
    sample = rng.choice(len(pq), 24, replace=False)
    h = product.create_db(db, 0)
    try:
        rc, sc, eq, et, _ = h.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, 1, mode)
        assert rc == 0, product.last_error()
    finally:
        h.close()
    for p in sample:
        rc, want = oracle.search_database(queries[pq[p]], db.subset([pt[p]]), GO, GE, sm.flat(), 23, None, 1, MODES[mode])
        assert rc == 0
        w = [int(want[f][0]) for f in ("score", "endLocationQuery", "endLocationTarget")]
        if mode == "SW" and w[0] == 0:
            w[1:] = [-1, -1]
        assert [sc[p], eq[p], et[p]] == w, (mode, int(p), len(queries[pq[p]]), int(db.lengths[pt[p]]))


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pairs_rerun_at_32_bits(product, mode):
    """DNA +5 / -4, gaps 16 / 4: a 10,000-residue query whose planted near-copies score above 32,767, targets up to
    100 kb."""
    rng = np.random.default_rng(304)
    sm = matrices.simple(4, 5, -4)
    q = rng.integers(0, 4, 10000, dtype=np.uint8)
    db = datasets.dna_db(1500, 304, query=q, n_at_max=3, n_planted=4)
    queries = [q, rng.integers(0, 4, 700, dtype=np.uint8)]
    big = np.nonzero(db.lengths >= 9000)[0]
    pt = np.concatenate([big, rng.choice(len(db), 150, replace=False), big[:3]]).astype(np.int32)
    pq = np.concatenate([np.zeros(len(big), np.int32), rng.integers(0, 2, 150), np.ones(3, np.int32)]).astype(np.int32)
    h = product.create_db(db, 0)
    try:
        full = [h.search(x, 16, 4, sm.flat(), 4, 1, mode) for x in queries]
        assert all(f[0] == 0 for f in full)
        rc, sc, eq, et, _ = h.search_pairs(queries, pq, pt, 16, 4, sm.flat(), 4, 1, mode)
        assert rc == 0, product.last_error()
        stats = h.last_stats()
        for a, got in enumerate((sc, eq, et)):
            want = np.array([full[x][1 + a][t] for x, t in zip(pq, pt)])
            assert np.array_equal(got, want), (mode, a, np.nonzero(got != want)[0][:5])
        if mode in ("SW", "OV"):  # NW / HW route these pairs to 32 bits from the start
            assert sc.max() > 32767 and stats["rerun32"] > 0, stats
    finally:
        h.close()


def test_pairs_longest_target_against_a_long_query(product):
    """The longest target of a configs[2]-shaped database (35,213 residues) against a 5,478-residue query."""
    sm = matrices.blosum62()
    rng = np.random.default_rng(305)
    db = datasets.protein_db(3000, 305, sm, tail_fraction=0.002, exact_max=True)
    longest = int(np.argmax(db.lengths))
    assert db.lengths[longest] == datasets.MAX_PROTEIN_LEN
    q = datasets.random_residues(5478, rng, sm)
    pt = np.array([longest, 0, 1, longest, 2], np.int32)
    pq = np.zeros(len(pt), np.int32)
    h = product.create_db(db, 0)
    try:
        for mode in ("SW", "NW", "HW", "OV"):
            rc0, fsc, feq, fet, _ = h.search(q, GO, GE, sm.flat(), 23, 1, mode)
            rc, sc, eq, et, _ = h.search_pairs([q], pq, pt, GO, GE, sm.flat(), 23, 1, mode)
            assert rc0 == 0 and rc == 0, product.last_error()
            assert np.array_equal(sc, fsc[pt]) and np.array_equal(eq, feq[pt]) and np.array_equal(et, fet[pt]), mode
    finally:
        h.close()


def test_pairs_argument_errors(product):
    _, sm, queries, db, pq, pt = _setup(306)
    n = len(db)
    h = product.create_db(db, 0)
    lib = h.eng.lib

    def call(pq_, pt_, mode="SW", qs=queries, matrix_len=23):
        return h.search_pairs(qs, pq_, pt_, GO, GE, sm.flat(), matrix_len, 1, mode)

    def untouched(pq_, pt_, **kw):
        keep, ptrs, qlens, a, b, m = h._pairs_args(kw.get("qs", queries), pq_, pt_)
        outs = [np.full(m, -777, np.int32) for _ in range(3)]
        rc = lib.opalb200_db_search_pairs(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, m, a.ctypes.data, b.ctypes.data,
                                          GO, GE, sm.flat().ctypes.data, 23, 1, kw.get("mode", MODES["SW"]),
                                          *[o.ctypes.data for o in outs], None)
        assert all((o == -777).all() for o in outs)
        return rc

    try:
        bad_q = pq.copy(); bad_q[5] = len(queries)
        assert untouched(bad_q, pt) == OPAL_ERR_INVALID_ARGUMENT and "pair 5" in product.last_error()
        for t in (-1, n):
            bad_t = pt.copy(); bad_t[9] = t
            assert untouched(pq, bad_t) == OPAL_ERR_INVALID_ARGUMENT and "pair 9" in product.last_error()
        assert untouched(pq, pt, mode=7) == OPAL_ERR_INVALID_MODE
        wide = [q.copy() for q in queries]
        wide[3][10] = 23  # a residue code >= alphabetLength
        assert untouched(pq, pt, qs=wide) == OPAL_ERR_INVALID_ARGUMENT
        # NULL arrays with a count > 0
        m = len(pq)
        sc = np.full(m, -777, np.int32)
        keep, ptrs, qlens, a, b, _ = h._pairs_args(queries, pq, pt)
        for args in ((None, b.ctypes.data, sc.ctypes.data), (a.ctypes.data, None, sc.ctypes.data), (a.ctypes.data, b.ctypes.data, None)):
            rc = lib.opalb200_db_search_pairs(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, m, args[0], args[1], GO, GE,
                                              sm.flat().ctypes.data, 23, 0, MODES["SW"], args[2], None, None, None)
            assert rc == OPAL_ERR_INVALID_ARGUMENT
        rc = lib.opalb200_db_search_pairs(h.handle, len(keep), None, None, m, a.ctypes.data, b.ctypes.data, GO, GE,
                                          sm.flat().ctypes.data, 23, 0, MODES["SW"], sc.ctypes.data, None, None, None)
        assert rc == OPAL_ERR_INVALID_ARGUMENT and (sc == -777).all()
        rc = lib.opalb200_db_search_pairs_results(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, m, a.ctypes.data,
                                                  b.ctypes.data, GO, GE, sm.flat().ctypes.data, 23, None, 2, MODES["SW"])
        assert rc == OPAL_ERR_INVALID_ARGUMENT
        # deviceMs is not written on a failure
        ms = ctypes.c_float(-5.0)
        bad_q = pq.copy(); bad_q[0] = -1
        rc = lib.opalb200_db_search_pairs(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, m, bad_q.ctypes.data, b.ctypes.data,
                                          GO, GE, sm.flat().ctypes.data, 23, 0, MODES["SW"], sc.ctypes.data, None, None, ctypes.byref(ms))
        assert rc == OPAL_ERR_INVALID_ARGUMENT and ms.value == -5.0 and (sc == -777).all()
        # no pairs: 0, nothing read beyond the counts, nothing written (whatever the search type and outputs)
        assert lib.opalb200_db_search_pairs(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, 0, None, None, GO, GE,
                                            sm.flat().ctypes.data, 23, 2, MODES["SW"], None, None, None, ctypes.byref(ms)) == 0
        assert ms.value == -5.0
        assert lib.opalb200_db_search_pairs_results(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, 0, None, None, GO, GE,
                                                    sm.flat().ctypes.data, 23, None, 7, MODES["SW"]) == 0
        rc, sc0, _, _, _ = call(np.zeros(0, np.int32), np.zeros(0, np.int32))
        assert rc == 0 and sc0.size == 0
        assert lib.opalb200_db_search_pairs(h.handle, len(keep), ptrs.ctypes.data, qlens.ctypes.data, 0, None, None, GO, GE,
                                            sm.flat().ctypes.data, 23, 1, MODES["SW"], None, None, None, None) == 0
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pair_records_reuse_rule(product, oracle, mode):
    """Records prefilled at SCORE and at SCORE_END, then searched at ALIGNMENT: as opalSearchDatabase with the same
    prefilled records."""
    rng, sm, queries, db, pq, pt = _setup(307)
    sample = rng.choice(len(pq), 30, replace=False)
    pq, pt = pq[sample], pt[sample]
    h = product.create_db(db, 0)
    try:
        for level in (0, 1):
            rc, pre = h.search_pairs_results(queries, pq, pt, GO, GE, sm.flat(), 23, level, mode)
            assert rc == 0, product.last_error()
            want = []
            for p in range(len(pq)):
                rec = np.ascontiguousarray(pre[p:p + 1].copy())
                rc, w = oracle.search_database(queries[pq[p]], db.subset([pt[p]]), GO, GE, sm.flat(), 23, rec, 2, MODES[mode])
                assert rc == 0
                want.append(dump_results(w)[0])
                free_alignments(w)
            rc, got = h.search_pairs_results(queries, pq, pt, GO, GE, sm.flat(), 23, 2, mode, results=pre)
            assert rc == 0, product.last_error()
            assert dump_results(got) == want, (mode, level)
            free_alignments(got)
    finally:
        h.close()


def _devices(product, want=3):
    """Every device, or -- on a one-GPU host -- the same ordinal several times: several shards on one device run the same
    dealing, fan-out, scatter and per-shard alignment code (as in test_gpu_multi_device.py)."""
    n = product.device_count()
    return list(range(n)) if n >= 2 else [0] * want


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pairs_on_several_devices_equal_one_device(product, mode):
    _, sm, queries, db, pq, pt = _setup(308)
    devs = _devices(product)
    h1 = product.create_db(db, 0)
    hn = product.create_db(db, devs)
    try:
        assert hn.devices() == len(devs)
        a = h1.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, 1, mode)
        b = hn.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, 1, mode)
        assert a[0] == 0 and b[0] == 0, product.last_error()
        for x, y in zip(a[1:4], b[1:4]):
            assert np.array_equal(x, y), mode
        for level in (None, 0, 1):  # fresh records, and records prefilled at SCORE / SCORE_END (the reuse rule per shard)
            recs = []
            for h in (h1, hn):
                pre = None
                if level is not None:
                    rc, pre = h1.search_pairs_results(queries, pq, pt, GO, GE, sm.flat(), 23, level, mode)
                    assert rc == 0, product.last_error()
                rc, r = h.search_pairs_results(queries, pq, pt, GO, GE, sm.flat(), 23, 2, mode, results=pre)
                assert rc == 0, product.last_error()
                recs.append(dump_results(r))
                free_alignments(r)
            assert recs[0] == recs[1], (mode, level)
    finally:
        h1.close()
        hn.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_pairs_with_only_short_queries_use_the_short_strips(product, mode):
    """Queries of at most 8 residues: the step-time model prices the R = 8 kernels lowest, and they must give the full
    search's results."""
    rng = np.random.default_rng(310)
    sm = matrices.blosum62()
    queries = [datasets.random_residues(n, rng, sm) for n in (1, 2, 3, 5, 8, 8, 4, 7)]
    db = _db(rng, sm, queries)
    pq, pt = _pairs(rng, len(queries), len(db))
    h = product.create_db(db, 0)
    try:
        full = _full(h, queries, sm, 1, mode)
        rc, sc, eq, et, _ = h.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, 1, mode)
        assert rc == 0, product.last_error()
        assert h.last_stats()["R"] == 8
        for a, got in enumerate((sc, eq, et)):
            want = np.array([full[q][a][t] for q, t in zip(pq, pt)])
            assert np.array_equal(got, want), (mode, a, np.nonzero(got != want)[0][:5])
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["NW", "HW"])
def test_pairs_range_tracking_sends_global_pairs_to_32_bits(product, mode):
    """NW / HW pairs that pass the a-priori border rule of the 16-bit class (a 3,700-residue DNA query, +10 / -4, gaps
    16 / 4: the border -16 - 3700 x 4 stays above both modes' limits) but whose scores leave the tracked range: an exact
    copy of the query scores 37,000.  They are flagged by the range tracking, re-run at 32 bits, and equal the full
    search."""
    rng = np.random.default_rng(311)
    sm = matrices.simple(4, 10, -4)
    q = rng.integers(0, 4, 3700, dtype=np.uint8)
    near = np.where(rng.random(len(q)) < 0.99, q, rng.integers(0, 4, len(q))).astype(np.uint8)
    seqs = [rng.integers(0, 4, int(x), dtype=np.uint8) for x in rng.integers(100, 3500, 60)] + [q.copy(), near]
    db = SequenceDB.from_sequences(seqs)
    queries = [q, rng.integers(0, 4, 900, dtype=np.uint8)]
    pt = np.array([60, 61] + list(range(0, 60, 3)) + [60, 5, 61], np.int32)
    pq = np.array([0, 0] + [0] * 20 + [1, 1, 1], np.int32)
    h = product.create_db(db, 0)
    try:
        full = [h.search(x, 16, 4, sm.flat(), 4, 1, mode) for x in queries]
        assert all(f[0] == 0 for f in full)
        rc, sc, eq, et, _ = h.search_pairs(queries, pq, pt, 16, 4, sm.flat(), 4, 1, mode)
        assert rc == 0, product.last_error()
        stats = h.last_stats()
        for a, got in enumerate((sc, eq, et)):
            want = np.array([full[x][1 + a][t] for x, t in zip(pq, pt)])
            assert np.array_equal(got, want), (mode, a, np.nonzero(got != want)[0][:5])
        assert sc[0] == 37000 and stats["rerun32"] > 0 and stats["R"] > 0, stats  # R > 0: the 16-bit class ran
    finally:
        h.close()


def test_pairs_at_the_timed_size(product):
    """100 queries x 500 candidates on the 570k-sequence configs[2] database (queries are mutated copies of database
    entries, so every candidate list holds a homolog)."""
    sm = matrices.blosum62()
    rng = np.random.default_rng(309)
    db = datasets.config3_db(sm)
    n = len(db)
    src = rng.choice(np.nonzero(db.lengths < 3000)[0], 100, replace=False)
    queries = [datasets.mutate(db.sequence(int(i)), 0.7, rng, sm) for i in src]
    pt = np.concatenate([np.concatenate([[i], rng.choice(n, 499, replace=False)]) for i in src]).astype(np.int32)
    pq = np.repeat(np.arange(100), 500).astype(np.int32)
    h = product.create_db(db, 0)
    try:
        for mode in ("SW", "NW"):
            rc, sc, eq, et, ms = h.search_pairs(queries, pq, pt, GO, GE, sm.flat(), 23, 1, mode)
            assert rc == 0, product.last_error()
            for q in range(100):
                rcf, fsc, feq, fet, _ = h.search(queries[q], GO, GE, sm.flat(), 23, 1, mode)
                assert rcf == 0
                sl = slice(500 * q, 500 * (q + 1))
                t = pt[sl]
                assert np.array_equal(sc[sl], fsc[t]) and np.array_equal(eq[sl], feq[t]) and np.array_equal(et[sl], fet[t]), (mode, q)
    finally:
        h.close()
