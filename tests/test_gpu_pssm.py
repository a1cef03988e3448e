"""Searches with a position-specific scoring matrix (opalb200_db_search_pssm and its batch / results / top-k twins) on
the GPU: a PSSM built as S[query] gives exactly the matrix search on every path of the engine (16-bit bulk, 32-bit
re-runs, folded and chained tasks, A = 256, skip masks, tiny queries), and position-specific PSSMs agree with the
oracle's PSSM restatement (tests/oracle_pssm.c) -- score, end, start and operation string."""
import numpy as np
import pytest

from _pssm import matrix_pssm, noisy_pssm, oracle_search_pssm, replay_ok
from _util import MODES, SequenceDB, dump_results, free_alignments
from opal_b200 import datasets, matrices

pytestmark = pytest.mark.gpu

OPAL_ERR_OVERFLOW, OPAL_ERR_INVALID_ARGUMENT = 1, 4


def _db(rng, sm, q, n=400, longest=()):
    seqs = [datasets.random_residues(int(k), rng, sm) for k in rng.integers(1, 420, n)]
    for k, length in enumerate(longest):
        seqs[3 * k + 2] = datasets.random_residues(length, rng, sm)
    seqs[5] = datasets.mutate(q, 0.8, rng, sm)
    seqs[7] = np.zeros(0, dtype=np.uint8)
    return SequenceDB.from_sequences(seqs)


def _same(h, q, m, alen, go, ge, mode, st, skip=None):
    """search_pssm(S[q]) against search(q, S): every array equal.  Returns last_stats() of the PSSM search."""
    rc1, s1, e1, t1, _ = h.search(q, go, ge, m, alen, st, mode, skip=skip)
    rc2, s2, e2, t2, _ = h.search_pssm(matrix_pssm(q, m, alen), go, ge, st, mode, skip=skip, alphabet_length=alen)
    assert rc1 == rc2 == 0, (mode, st)
    assert np.array_equal(s1, s2) and np.array_equal(e1, e2) and np.array_equal(t1, t2), (mode, st)
    return h.last_stats()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_matrix_pssm_equals_matrix_search_on_every_path(product, mode, monkeypatch):
    rng = np.random.default_rng(40 + MODES[mode])
    sm = matrices.blosum62()
    q = datasets.random_residues(200, rng, sm)
    h = product.create_db(_db(rng, sm, q), 0)
    try:
        for st in (0, 1):
            stats = _same(h, q, sm.flat(), 23, 11, 1, mode, st)                      # 16-bit bulk class
            assert stats["kernel_launches"] > 0 and stats["rerun32"] == 0, stats
            skip = (rng.random(h.n) < 0.3).astype(np.uint8)                           # skip mask
            _same(h, q, sm.flat(), 23, 11, 1, mode, st, skip=skip)
            for qq in (q[:0], q[:1]):                                                 # Q = 0, 1
                _same(h, qq, sm.flat(), 23, 11, 1, mode, st)
        m48 = (sm.matrix * 48).ravel().astype(np.int32)                               # 32-bit: re-runs (SW) / large gaps
        go, ge, m = (528, 48, m48) if mode in ("SW", "OV") else (3000, 900, sm.flat())
        for st in (0, 1):
            stats = _same(h, q, m, 23, go, ge, mode, st)
            if mode == "SW":
                assert stats["rerun32"] > 0, stats
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_matrix_pssm_folded_and_chained(product, mode, monkeypatch):
    rng = np.random.default_rng(50 + MODES[mode])
    sm = matrices.blosum62()
    q = datasets.random_residues(513, rng, sm)
    seqs = [datasets.random_residues(int(x), rng, sm) for x in rng.integers(30, 420, 3000)]
    seqs += [datasets.random_residues(int(x), rng, sm) for x in rng.integers(1500, 3500, 70)]
    seqs[3] = datasets.mutate(q, 0.75, rng, sm)
    db = SequenceDB.from_sequences([seqs[i] for i in rng.permutation(len(seqs))])
    monkeypatch.setenv("OPAL_B200_NO_CHAIN", "1")
    h = product.create_db(db, 0)
    try:
        for st in (0, 1):
            assert _same(h, q, sm.flat(), 23, 11, 1, mode, st)["folded"] > 0
    finally:
        h.close()
    monkeypatch.delenv("OPAL_B200_NO_CHAIN")
    monkeypatch.setenv("OPAL_B200_CHAIN", "1")
    q = datasets.random_residues(1600, rng, sm)
    h = product.create_db(_db(rng, sm, q, n=180, longest=(2600, 2300, 1900, 1500, 1200)), 0)
    try:
        for st in (0, 1):
            assert _same(h, q, sm.flat(), 23, 11, 1, mode, st)["chained"] > 0
    finally:
        h.close()


def test_matrix_pssm_alphabet_256_with_code_255(product):
    rng = np.random.default_rng(60)
    m = rng.integers(-5, 6, (256, 256)).astype(np.int32)
    m[np.arange(256), np.arange(256)] = 9
    seqs = [rng.integers(0, 256, int(k), dtype=np.uint8) for k in rng.integers(1, 300, 150)]
    seqs[0][0] = 255
    q = rng.integers(0, 256, 120, dtype=np.uint8)
    q[3] = 255
    h = product.create_db(SequenceDB.from_sequences(seqs), 0)
    try:
        for mode in ("SW", "NW", "HW", "OV"):
            for st in (0, 1):
                _same(h, q, m.ravel(), 256, 7, 2, mode, st)
    finally:
        h.close()


def _check_alignments(product, h, db, q, p, go, ge, mode):
    rc, got = h.search_results_pssm(p, go, ge, 2, mode, query=q)
    assert rc == 0, product.last_error()
    rc, want = oracle_search_pssm(q, p, db, go, ge, 2, MODES[mode])
    assert rc == 0
    g, w = dump_results(got), dump_results(want)
    assert g == w, (mode, [(i, a, b) for i, (a, b) in enumerate(zip(g, w)) if a != b][:3])
    for i in range(len(db)):
        if got["alignmentLength"][i] > 0:
            assert replay_ok(q, p, db.sequence(i), got, i, go, ge)
    free_alignments(got)
    free_alignments(want)


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_position_specific_pssm_alignments_match_the_oracle(product, mode):
    rng = np.random.default_rng(70 + MODES[mode])
    sm = matrices.blosum62()
    q = datasets.random_residues(300, rng, sm)
    db = _db(rng, sm, q, n=250)
    h = product.create_db(db, 0)
    try:
        for go, ge in ((11, 1), (4, 2)):
            _check_alignments(product, h, db, q, noisy_pssm(q, sm.flat(), 23, rng), go, ge, mode)
    finally:
        h.close()


def test_position_specific_pssm_at_configs2_size(product):
    """BASELINE configs[2]'s 570k-sequence database, Q = 1000, all four modes, score + end; the 40 longest targets,
    the 20 best hits and 440 random ones against the oracle's PSSM restatement."""
    sm = matrices.blosum62()
    q = [x for x in datasets.config3_queries(sm) if len(x) == 1000][0]
    db = datasets.config3_db(sm, query=sm.encode(datasets.P18080))
    rng = np.random.default_rng(1000)
    p = noisy_pssm(q, sm.flat(), 23, rng)
    h = product.create_db(db, 0)
    try:
        order = np.argsort(-db.lengths.astype(np.int64), kind="stable")
        for mode in ("SW", "NW", "HW", "OV"):
            rc, sc, eq, et, _ = h.search_pssm(p, 11, 1, 1, mode)
            assert rc == 0, product.last_error()
            sample = np.unique(np.concatenate([order[:40], np.argsort(-sc.astype(np.int64), kind="stable")[:20],
                                               rng.choice(len(db), 440, replace=False)]))
            rc, want = oracle_search_pssm(None, p, db.subset(sample), 11, 1, 1, MODES[mode])
            assert rc == 0
            assert np.array_equal(want["score"], sc[sample]), (mode, sample[want["score"] != sc[sample]][:5])
            ok = want["score"] > 0 if mode == "SW" else np.ones(len(sample), bool)
            assert np.array_equal(want["endLocationQuery"][ok], eq[sample][ok]), mode
            assert np.array_equal(want["endLocationTarget"][ok], et[sample][ok]), mode
    finally:
        h.close()


@pytest.mark.parametrize("mode", ["SW", "OV"])
def test_topk_pssm(product, mode):
    rng = np.random.default_rng(80 + MODES[mode])
    sm = matrices.blosum62()
    q = datasets.random_residues(250, rng, sm)
    db = _db(rng, sm, q, n=600)
    p = noisy_pssm(q, sm.flat(), 23, rng)
    h = product.create_db(db, 0)
    try:
        rc, sc, _, _, _ = h.search_pssm(p, 11, 1, 1, mode)
        assert rc == 0
        top = np.lexsort((np.arange(len(db)), -sc.astype(np.int64)))[:40]
        rc, idx, res = h.search_topk_pssm(p, 11, 1, 2, mode, 40, query=q)
        assert rc == 0, product.last_error()
        assert np.array_equal(idx, top)
        rc, want = oracle_search_pssm(q, p, db.subset(top), 11, 1, 2, MODES[mode])
        assert rc == 0
        assert dump_results(res) == dump_results(want)
        free_alignments(res)
        free_alignments(want)
    finally:
        h.close()


def test_batch_pssm_equals_row_by_row(product):
    rng = np.random.default_rng(90)
    sm = matrices.blosum62()
    qs = [datasets.random_residues(n, rng, sm) for n in (300, 90, 700, 1, 450, 1200)]
    ps = [noisy_pssm(q, sm.flat(), 23, rng) for q in qs]
    modes = ["HW", "SW", "NW", "OV", "SW", "NW"]
    h = product.create_db(_db(rng, sm, qs[0]), 0)
    try:
        for st in (0, 1):
            rows = [h.search_pssm(p, 11, 1, st, m) for p, m in zip(ps, modes)]
            assert all(r[0] == 0 for r in rows)
            for fl in (1, 4):
                rc, S, E, T, _ = h.search_batch_pssm(ps, 11, 1, st, modes, in_flight=fl)
                assert rc == 0, product.last_error()
                for k, r in enumerate(rows):
                    assert np.array_equal(S[k], r[1]) and np.array_equal(E[k], r[2]) and np.array_equal(T[k], r[3]), (st, fl, k)
    finally:
        h.close()


def test_multi_device_pssm_equals_single_device(product):
    """Shards on two devices -- or two shards on one device when there is only one: the same code path (one host thread
    and one set of streams per shard, results scattered by the index map, top-k merged across shards)."""
    rng = np.random.default_rng(100)
    sm = matrices.blosum62()
    q = datasets.random_residues(400, rng, sm)
    db = _db(rng, sm, q, n=500)
    p = noisy_pssm(q, sm.flat(), 23, rng)
    one = product.create_db(db, 0)
    many = product.create_db(db, [0, 1] if product.device_count() >= 2 else [0, 0])
    try:
        assert many.devices() == 2
        for mode in ("SW", "NW", "HW", "OV"):
            a, b = one.search_pssm(p, 11, 1, 1, mode), many.search_pssm(p, 11, 1, 1, mode)
            assert a[0] == b[0] == 0 and all(np.array_equal(x, y) for x, y in zip(a[1:4], b[1:4])), mode
            ra, rb = one.search_results_pssm(p, 11, 1, 2, mode, query=q)[1], many.search_results_pssm(p, 11, 1, 2, mode, query=q)[1]
            assert dump_results(ra) == dump_results(rb), mode
            ka, kb = one.search_topk_pssm(p, 11, 1, 2, mode, 25, query=q), many.search_topk_pssm(p, 11, 1, 2, mode, 25, query=q)
            assert ka[0] == kb[0] == 0 and np.array_equal(ka[1], kb[1]) and dump_results(ka[2]) == dump_results(kb[2]), mode
            bs = many.search_batch_pssm([p, p[:100]], 11, 1, 1, [mode, "SW"], in_flight=2)
            assert bs[0] == 0 and np.array_equal(bs[1][0], a[1])
            for r in (ra, rb, ka[2], kb[2]):
                free_alignments(r)
    finally:
        one.close()
        many.close()


def test_pssm_argument_errors_leave_the_handle_usable(product):
    rng = np.random.default_rng(110)
    sm = matrices.blosum62()
    q = datasets.random_residues(150, rng, sm)
    db = _db(rng, sm, q, n=120)
    p = noisy_pssm(q, sm.flat(), 23, rng)
    h = product.create_db(db, 0)
    try:
        rc0, s0, e0, t0, _ = h.search_pssm(p, 11, 1, 1, "SW")
        assert rc0 == 0
        assert h.search_pssm(None, 11, 1, 1, "SW", query_length=150, alphabet_length=23)[0] == OPAL_ERR_INVALID_ARGUMENT
        assert h.search_results_pssm(p, 11, 1, 2, "SW", query=None)[0] == OPAL_ERR_INVALID_ARGUMENT
        assert h.search_topk_pssm(p, 11, 1, 2, "SW", 5, query=None)[0] == OPAL_ERR_INVALID_ARGUMENT
        big = p.copy()
        big[10, 4] = 2 ** 30
        assert h.search_pssm(big, 11, 1, 1, "SW")[0] == OPAL_ERR_OVERFLOW
        top = int(db.residues.max())  # (random_residues draws the 20 standard amino acids only: codes 0 .. 19)
        assert h.search_pssm(p[:, :top], 11, 1, 1, "SW")[0] == OPAL_ERR_INVALID_ARGUMENT   # database codes >= A
        assert h.search_pssm(p[:, :top + 1], 11, 1, 1, "SW")[0] == 0                       # ... and just enough letters
        assert h.search_pssm(p, -1, 1, 1, "SW")[0] == OPAL_ERR_INVALID_ARGUMENT
        assert h.search_pssm(p, 11, -1, 1, "NW")[0] == OPAL_ERR_INVALID_ARGUMENT
        rc, s, e, t, _ = h.search_pssm(p, 11, 1, 1, "SW")
        assert rc == 0 and np.array_equal(s, s0) and np.array_equal(e, e0) and np.array_equal(t, t0)
    finally:
        h.close()
