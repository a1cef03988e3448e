"""GPU tests of opalb200_db_search_batch_topk[_pssm]: many searches' score -> top-k -> alignment in one call.  Row s of a
batch must be exactly what opalb200_db_search_topk[_pssm] returns for search s alone, at every search level, with
mixed modes, any number of searches in flight, one or several shards, and the single call's error codes."""
import numpy as np
import pytest

from _pssm import matrix_pssm, noisy_pssm
from _util import MODES, SequenceDB, dump_results, free_alignments
from opal_b200 import datasets, matrices

pytestmark = pytest.mark.gpu

OPAL_ERR_INVALID_MODE, OPAL_ERR_INVALID_ARGUMENT = 3, 4


def _db(rng, sm, planted, n=400):
    """Random targets with planted homologs of every query, a few zero-length targets and one of 4,000 residues."""
    seqs = [datasets.random_residues(int(x), rng, sm) for x in rng.integers(1, 420, n)]
    for k, q in enumerate(p for p in planted if len(p) > 0):
        for j in range(3):
            seqs[11 * k + 37 * j + 1] = datasets.mutate(q, 0.75, rng, sm)
    for i in (7, 150, 299):
        if i < n:
            seqs[i] = np.zeros(0, np.uint8)
    seqs[42] = datasets.random_residues(4000, rng, sm)
    return SequenceDB.from_sequences(seqs)


def _queries(rng, sm):
    """Q = 0, Q = 1, one query of more than 1,056 rows (several passes) and ~130-residue queries."""
    return [datasets.random_residues(n, rng, sm) for n in (130, 0, 1, 1300, 128, 133, 131, 129)]


def _rows(res):
    out = [dump_results(r) for r in res]
    for r in res:
        free_alignments(r)
    return out


def _loop(h, queries, modes, st, k, sm):
    idx, rows = [], []
    for q, mode in zip(queries, modes):
        rc, i, r = h.search_topk(q, 11, 1, sm.flat(), 23, st, mode, k)
        assert rc == 0, h.eng.last_error()
        idx.append(i.tolist())
        rows.append(dump_results(r))
        free_alignments(r)
    return idx, rows


@pytest.mark.parametrize("in_flight", [1, 3, 16])
def test_batch_equals_loop_of_single_calls(product, in_flight):
    rng = np.random.default_rng(101)
    sm = matrices.blosum62()
    queries = _queries(rng, sm)
    db = _db(rng, sm, queries)
    modes = ["SW", "NW", "HW", "OV", "SW", "OV", "HW", "NW"]
    h = product.create_db(db, 0)
    try:
        for st in (0, 1, 2):
            rc, idx, res = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, st, modes, 25, in_flight=in_flight)
            assert rc == 0, product.last_error()
            assert idx.shape == (len(queries), 25) and res.shape == (len(queries), 25)
            got = _rows(res)
            want_idx, want = _loop(h, queries, modes, st, 25, sm)
            assert idx.tolist() == want_idx, st
            for s in range(len(queries)):
                assert got[s] == want[s], (st, s, modes[s])
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_batch_equals_the_two_call_protocol(product, mode):
    """Row s at ALIGNMENT = opalSearchDatabase score + end, top k by (score desc, index asc), then ALIGNMENT over the
    k-entry sub-database with the prefilled records."""
    rng = np.random.default_rng(102)
    sm = matrices.blosum62()
    queries = [datasets.random_residues(n, rng, sm) for n in (110, 90, 140)]
    db = _db(rng, sm, queries, n=300)
    k = 37
    h = product.create_db(db, 0)
    try:
        rc, idx, res = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, mode, k)
        assert rc == 0, product.last_error()
        got = _rows(res)
        for s, q in enumerate(queries):
            rc, full = product.search_database(q, db, 11, 1, sm.flat(), 23, None, 1, MODES[mode])
            assert rc == 0
            order = sorted(range(len(db)), key=lambda i: (-int(full["score"][i]), i))[:k]
            rc, res2 = product.search_database(q, db.subset(order), 11, 1, sm.flat(), 23, full[order].copy(), 2, MODES[mode])
            assert rc == 0
            assert idx[s].tolist() == order
            assert got[s] == dump_results(res2), s
            free_alignments(res2)
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_batch_ties_empties_and_reruns(product, mode):
    """Tie-heavy scores (tiny alphabet), zero-length targets, 32-bit re-runs (scaled matrix), k from 0 to beyond n."""
    rng = np.random.default_rng(19)
    a = 3
    m = (matrices.simple(a, 2, -1).matrix * 300).ravel().astype(np.int32)
    queries = [rng.integers(0, a, n).astype(np.uint8) for n in (150, 60, 150)]
    seqs = [rng.integers(0, a, int(n)).astype(np.uint8) for n in rng.integers(0, 40, 260)]
    for i in (3, 17, 101):
        seqs[i] = np.zeros(0, np.uint8)
    seqs[50] = queries[0].copy()                        # beyond 16 bits
    seqs[51] = np.concatenate([queries[0][:100], queries[0][:100]])
    for i in range(200, 230):
        seqs[i] = seqs[199].copy()
    db = SequenceDB.from_sequences(seqs)
    n = len(db)
    h = product.create_db(db, 0)
    try:
        for k in (1, 31, n - 1, n, n + 5, 0):
            rc, idx, res = h.search_batch_topk(queries, 900, 300, m, a, 1, mode, k, in_flight=2)
            assert rc == 0, product.last_error()
            assert idx.shape == (len(queries), min(k, n))
            for s, q in enumerate(queries):
                rc1, i1, r1 = h.search_topk(q, 900, 300, m, a, 1, mode, k)
                assert rc1 == 0 and idx[s].tolist() == i1.tolist(), (mode, k, s)
                assert dump_results(res[s]) == dump_results(r1)
    finally:
        h.close()


def test_pssm_batch(product):
    rng = np.random.default_rng(104)
    sm = matrices.blosum62()
    queries = _queries(rng, sm)[:5]
    db = _db(rng, sm, queries)
    modes = ["SW", "OV", "HW", "NW", "SW"]
    h = product.create_db(db, 0)
    try:
        # S[query] scores exactly like the matrix: equal to the matrix batch row for row, alignments included
        rc, i1, r1 = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, modes, 30)
        rc2, i2, r2 = h.search_batch_topk_pssm([matrix_pssm(q, sm.flat(), 23) for q in queries], 11, 1, 2, modes, 30, queries=queries)
        assert rc == 0 and rc2 == 0, product.last_error()
        assert np.array_equal(i1, i2) and _rows(r1) == _rows(r2)
        # random PSSMs: equal to a loop of search_topk_pssm
        ps = [noisy_pssm(q, sm.flat(), 23, rng) for q in queries]
        for st in (1, 2):
            rc, idx, res = h.search_batch_topk_pssm(ps, 11, 1, st, modes, 30, queries=queries, in_flight=4)
            assert rc == 0, product.last_error()
            got = _rows(res)
            for s, (p, q) in enumerate(zip(ps, queries)):
                rc1, i, r = h.search_topk_pssm(p, 11, 1, st, modes[s], 30, query=q)
                assert rc1 == 0 and idx[s].tolist() == i.tolist() and got[s] == dump_results(r), (st, s)
                free_alignments(r)
        # below ALIGNMENT the residues are not needed; at ALIGNMENT they are
        rc, idx, res = h.search_batch_topk_pssm(ps, 11, 1, 1, "SW", 10)
        assert rc == 0 and idx.shape == (5, 10)
        rc, idx, res = h.search_batch_topk_pssm(ps, 11, 1, 2, "SW", 10)
        assert rc == OPAL_ERR_INVALID_ARGUMENT and idx.shape == (5, 0)
    finally:
        h.close()


def test_batch_on_several_shards_equals_one_device(product):
    rng = np.random.default_rng(105)
    sm = matrices.blosum62()
    queries = _queries(rng, sm)
    db = _db(rng, sm, queries, n=500)
    modes = ["SW", "HW", "OV", "NW"] * 2
    devs = [0, 1] if product.device_count() >= 2 else [0, 0]
    h1 = product.create_db(db, 0)
    hn = product.create_db(db, devs)
    try:
        assert hn.devices() == 2
        for st in (1, 2):
            rc1, i1, r1 = h1.search_batch_topk(queries, 11, 1, sm.flat(), 23, st, modes, 60)
            rcn, i_n, rn = hn.search_batch_topk(queries, 11, 1, sm.flat(), 23, st, modes, 60, in_flight=4)
            assert rc1 == 0 and rcn == 0, product.last_error()
            assert np.array_equal(i1, i_n) and _rows(r1) == _rows(rn), st
        # hits of both shards are aligned: every target index of the database appears among them
        rc, idx, res = hn.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, "SW", len(db))
        assert rc == 0 and sorted(idx[0].tolist()) == list(range(len(db)))
        assert (res["alignmentLength"][0] > 0).sum() > 0
        _rows(res)
    finally:
        h1.close()
        hn.close()


def test_errors_write_nothing_and_keep_the_handle(product):
    rng = np.random.default_rng(106)
    sm = matrices.blosum62()
    queries = [datasets.random_residues(n, rng, sm) for n in (80, 90, 100, 110, 120)]
    db = _db(rng, sm, queries, n=200)
    maxcode = int(max(db.sequence(i).max() for i in range(len(db)) if db.lengths[i] > 0))
    h = product.create_db(db, 0)
    lib = product.lib
    try:
        rc, want_idx, want = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, "SW", 20)
        assert rc == 0
        want = _rows(want)

        def raw(modes, alen=23, go=11, pssms=None):
            """The C call with pre-filled sentinels: returns (rc, found, indices untouched, records untouched)."""
            import ctypes
            from opal_b200 import new_results
            from opal_b200.capi import result_pointers
            ns, k = len(queries), 20
            res = new_results(ns * k)
            res["score"] = -12345
            rp = result_pointers(res)
            idx = np.full(ns * k, -7, dtype=np.int32)
            found = ctypes.c_int(99)
            qbufs = [np.ascontiguousarray(q) for q in queries]
            qp = np.array([q.ctypes.data for q in qbufs], dtype=np.uint64)
            ql = np.array([len(q) for q in queries], dtype=np.int32)
            md = np.array(modes, dtype=np.int32)
            if pssms is None:
                sm_ = np.ascontiguousarray(sm.flat(), dtype=np.int32)
                rc = lib.opalb200_db_search_batch_topk(h.handle, ns, qp.ctypes.data, ql.ctypes.data, md.ctypes.data, go, 1,
                                                      sm_.ctypes.data, alen, 2, k, idx.ctypes.data, rp.ctypes.data,
                                                      ctypes.byref(found), 3)
            else:
                keep = [p for p in pssms if p is not None]
                pp = np.array([0 if p is None else p.ctypes.data for p in pssms], dtype=np.uint64)
                rc = lib.opalb200_db_search_batch_topk_pssm(h.handle, ns, qp.ctypes.data, pp.ctypes.data, ql.ctypes.data,
                                                           md.ctypes.data, 23, go, 1, 2, k, idx.ctypes.data, rp.ctypes.data,
                                                           ctypes.byref(found), 3)
                del keep
            return rc, found.value, bool((idx == -7).all()), bool((res["score"] == -12345).all() and (res["scoreSet"] == 0).all())

        sw = MODES["SW"]
        cases = [
            ("bad mode", dict(modes=[sw, sw, sw, 17, sw]), OPAL_ERR_INVALID_MODE),
            ("short alphabet", dict(modes=[sw] * 5, alen=maxcode), OPAL_ERR_INVALID_ARGUMENT),
            ("negative gap", dict(modes=[sw] * 5, go=-1), OPAL_ERR_INVALID_ARGUMENT),
            ("NULL PSSM", dict(modes=[sw] * 5, pssms=[matrix_pssm(q, sm.flat(), 23) if s != 3 else None
                                                      for s, q in enumerate(queries)]), OPAL_ERR_INVALID_ARGUMENT),
        ]
        for name, kw, code in cases:
            rc, found, idx_untouched, rec_untouched = raw(**kw)
            assert rc == code, (name, rc, product.last_error())
            assert found == 0 and idx_untouched and rec_untouched, name
        # a bad search at index 3 only: the single call on it gives the same code
        rc1, _, _ = h.search_topk(queries[3], 11, 1, sm.flat(), 23, 2, 17, 20)
        assert rc1 == OPAL_ERR_INVALID_MODE
        # k = 0: the matrix call returns 0 without checking, as the single call does
        rc, idx, res = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, [sw, sw, sw, 17, sw], 0)
        assert rc == 0 and idx.shape == (5, 0)
        # the handle is still usable: the next batch gives the earlier answers
        rc, idx, res = h.search_batch_topk(queries, 11, 1, sm.flat(), 23, 2, "SW", 20)
        assert rc == 0 and np.array_equal(idx, want_idx) and _rows(res) == want
    finally:
        h.close()


@pytest.fixture(scope="module")
def big():
    sm = matrices.blosum62()
    q = sm.encode(datasets.P18080)
    return sm, q, datasets.config3_db(sm, query=q)


def test_full_size_batch_equals_loop(product, big):
    """BASELINE configs[2] database: 4 queries x top-1000 SW ALIGNMENT with BLOSUM62 11/1, and the 8 x matrix
    (88 / 8, 32-bit re-runs)."""
    sm, q, db = big
    queries = [q] + datasets.config3_queries(sm)[:3]
    h = product.create_db(db, 0)
    try:
        for scale, go, ge in ((1, 11, 1), (8, 88, 8)):
            m = (sm.matrix * scale).ravel().astype(np.int32)
            rc, idx, res = h.search_batch_topk(queries, go, ge, m, 23, 2, "SW", 1000)
            assert rc == 0, product.last_error()
            got = [dump_results(r, digest=True) for r in res]
            for r in res:
                free_alignments(r)
            for s, qq in enumerate(queries):
                rc1, i1, r1 = h.search_topk(qq, go, ge, m, 23, 2, "SW", 1000)
                assert rc1 == 0 and np.array_equal(idx[s], i1), (scale, s)
                assert got[s] == dump_results(r1, digest=True), (scale, s)
                free_alignments(r1)
    finally:
        h.close()
