"""The oracle's PSSM restatement (tests/oracle_pssm.c), on the CPU: with pssm = S[query] it is the matrix oracle record
for record, operation strings included; on position-specific PSSMs it agrees with an independent numpy Gotoh and every
alignment replays under the PSSM.  Also: include/opal_b200.h, which declares the PSSM entry points, is valid C."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from _pssm import gotoh, matrix_pssm, noisy_pssm, oracle_search_pssm, replay_ok
from _util import MODES, ROOT, SequenceDB, dump_results, free_alignments, search_dump
from opal_b200 import matrices

STYPES = (0, 1, 2)


def _db(rng, alen, n=24, lo=0, hi=70):
    seqs = [rng.integers(0, alen, int(k), dtype=np.uint8) for k in rng.integers(lo, hi, n)]
    seqs[1] = np.zeros(0, dtype=np.uint8)  # an empty target
    return SequenceDB.from_sequences(seqs)


def _matrix(alen, rng):
    if alen == 24:  # BLOSUM62 (23 letters) and a stop letter: -4 against everything, 1 against itself
        m = np.full((24, 24), -4, dtype=np.int32)
        m[:23, :23] = matrices.blosum62().matrix
        m[23, 23] = 1
        return m.ravel()
    m = rng.integers(-4, 5, (alen, alen)).astype(np.int32)
    m[np.arange(alen), np.arange(alen)] = 6
    return m.ravel()


@pytest.mark.parametrize("alen", [4, 24])
@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_matrix_pssm_equals_matrix_oracle(oracle, alen, mode):
    rng = np.random.default_rng(alen * 10 + MODES[mode])
    m = _matrix(alen, rng)
    db = _db(rng, alen)
    top = int(np.argmax(m.reshape(alen, alen).max(axis=1)))  # a letter whose row attains max(S): both bands use one M
    for qlen in (0, 1, 37):
        q = rng.integers(0, alen, qlen, dtype=np.uint8)
        if qlen:
            q[qlen // 2] = top
        p = matrix_pssm(q, m, alen)
        for st in STYPES:
            rc1, want = search_dump(oracle, q, db, 11 if alen == 24 else 5, 1 if alen == 24 else 2, m, alen, st, MODES[mode])
            rc2, res = oracle_search_pssm(q, p, db, 11 if alen == 24 else 5, 1 if alen == 24 else 2, st, MODES[mode])
            got = dump_results(res)
            free_alignments(res)
            assert rc1 == rc2 == 0
            assert got == want, (mode, qlen, st, [(i, g, w) for i, (g, w) in enumerate(zip(got, want)) if g != w][:3])


@pytest.mark.parametrize("mode", ["SW", "NW", "HW", "OV"])
def test_position_specific_pssm_against_numpy_gotoh_and_replay(mode):
    rng = np.random.default_rng(77 + MODES[mode])
    sm = matrices.blosum62()
    db = _db(rng, 23, n=30, hi=45)
    for qlen in (0, 1, 29):
        q = rng.integers(0, 23, qlen, dtype=np.uint8)
        p = noisy_pssm(q, sm.flat(), 23, rng)
        for go, ge in ((11, 1), (3, 3)):
            rc1, ends = oracle_search_pssm(q, p, db, go, ge, 1, MODES[mode])
            rc, res = oracle_search_pssm(q, p, db, go, ge, 2, MODES[mode])
            assert rc1 == rc == 0
            assert (ends["score"] == res["score"]).all()
            for i in range(len(db)):
                t = db.sequence(i)
                want = gotoh(p, t, go, ge, mode)
                got = (int(ends["score"][i]), int(ends["endLocationQuery"][i]), int(ends["endLocationTarget"][i]))
                assert got == want, (mode, qlen, go, ge, i)
                if res["alignmentLength"][i] > 0 or res["startLocationQuery"][i] >= 0:
                    assert replay_ok(q, p, t, res, i, go, ge), (mode, qlen, i)
                else:  # no alignment: SW with score 0, or nothing to align
                    assert (mode == "SW" and got[0] == 0) or qlen == 0 or len(t) == 0, (mode, qlen, i)
            free_alignments(res)


def test_pssm_oracle_argument_rules():
    rng = np.random.default_rng(3)
    db = _db(rng, 4, n=4, lo=1)
    q = rng.integers(0, 4, 5, dtype=np.uint8)
    p = rng.integers(-3, 4, (5, 4)).astype(np.int32)
    assert oracle_search_pssm(q, p, db, 3, 1, 1, 7)[0] == 3                              # invalid mode
    big = p.copy()
    big[2, 1] = 2 ** 30
    assert oracle_search_pssm(q, big, db, 3, 1, 1, 0)[0] == 1                            # entry >= INT_MAX / 2
    assert oracle_search_pssm(q, p, db, -1, 1, 1, 0)[0] == 4                             # negative gap
    assert oracle_search_pssm(q, p[:, :3], db, 3, 1, 1, 0)[0] == 4                       # database codes >= A
    assert oracle_search_pssm(None, p, db, 3, 1, 2, 0)[0] == 4                           # ALIGNMENT without residues
    assert oracle_search_pssm(None, p, db, 3, 1, 1, 0)[0] == 0                           # ... which SCORE_END ignores


def test_opal_b200_header_compiles_as_c():
    cc = shutil.which(os.environ.get("CC", "cc")) or shutil.which("gcc")
    if not cc:
        pytest.skip("no C compiler")
    subprocess.run([cc, "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Werror", os.path.join(ROOT, "include", "opal_b200.h")],
                   check=True)
