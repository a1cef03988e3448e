"""Differential test: oracle/opal_oracle.c against the unmodified reference, CPU only.

The reference's answers come from oracle/_ref/libopal_ref.so when it was built, and otherwise from
tests/golden/oracle_vs_ref.json, which tests/golden/make_golden.py writes by running that library on exactly the
cases below (null where it crashed).  The reference runs in a forked child because its alignment stage can crash on
NW/HW/OV inputs (SURVEY.md section 8c Q8-Q10); where it survives the oracle must agree bit for bit.
"""
import json
import os

import numpy as np
import pytest

from _util import (GOLDEN_DIR, MODES, OPAL_OVERFLOW_BUCKETS, OPAL_OVERFLOW_SIMPLE, REF_SO, OpalCLibrary, SequenceDB,
                   run_forked, search_dump)
from opal_b200 import datasets, matrices

GOLDEN = os.path.join(GOLDEN_DIR, "oracle_vs_ref.json")


def random_case(rng, protein):
    if protein:
        sm = matrices.blosum62() if rng.random() < 0.5 else matrices.blosum50()
        go, ge = (11, 1) if rng.random() < 0.5 else (int(rng.integers(2, 14)), 1)
        q = datasets.random_residues(int(rng.integers(1, 120)), rng, sm)
        seqs = [datasets.random_residues(int(rng.integers(1, 160)), rng, sm) for _ in range(40)]
        for i in range(0, 40, 5):
            seqs[i] = datasets.mutate(q, 0.7, rng, sm)
        return q, SequenceDB.from_sequences(seqs), go, ge, sm.flat(), sm.alphabet_length
    a = int(rng.integers(2, 6))
    match, mism = int(rng.integers(1, 6)), -int(rng.integers(0, 5))
    ge = int(rng.integers(1, 4))
    go = int(rng.integers(2 * ge, 2 * ge + 8))  # keep gapOpen >= 2 gapExt (Q8)
    q = rng.integers(0, a, int(rng.integers(1, 70))).astype(np.uint8)
    seqs = [rng.integers(0, a, int(rng.integers(1, 90))).astype(np.uint8) for _ in range(40)]
    return q, SequenceDB.from_sequences(seqs), go, ge, matrices.simple(a, match, mism).flat(), a


def score_end_args(mode, seed, st):
    q, db, go, ge, m, a = random_case(np.random.default_rng(1000 + seed), protein=seed % 2 == 0)
    return q, db, go, ge, m, a, st, MODES[mode], OPAL_OVERFLOW_BUCKETS


def sw_alignment_args(seed):
    q, db, go, ge, m, a = random_case(np.random.default_rng(2000 + seed), protein=seed % 2 == 0)
    return q, db, go, ge, m, a, 2, MODES["SW"], OPAL_OVERFLOW_SIMPLE


def global_alignment_args(mode, seed):
    """Per-target calls (every 4th target), so that one crashing pair does not hide the others: {target: args}."""
    q, db, go, ge, m, a = random_case(np.random.default_rng(3000 + seed), protein=seed % 2 == 0)
    return {i: (q, db.subset([i]), go, ge, m, a, 2, MODES[mode], OPAL_OVERFLOW_SIMPLE) for i in range(0, len(db), 4)}


def all_cases():
    """(key, search_dump arguments) of every call the tests below compare; the keys of oracle_vs_ref.json."""
    for mode in ("NW", "HW", "OV", "SW"):
        for seed in range(12):
            for st in (0, 1):
                yield f"score_end/{mode}/{seed}/{st}", score_end_args(mode, seed, st)
    for seed in range(12):
        yield f"sw_alignment/{seed}", sw_alignment_args(seed)
    for mode in ("NW", "HW", "OV"):
        for seed in range(8):
            for i, args in global_alignment_args(mode, seed).items():
                yield f"global_alignment/{mode}/{seed}/{i}", args


def run_reference(ref, args):
    """(rc, records) of the reference on `args`, or None if it crashed."""
    return run_forked(lambda: search_dump(ref, *args))


@pytest.fixture(scope="module")
def reference():
    """want(key, args): the reference's (rc, records) for one case, or None where it crashed."""
    if os.path.exists(REF_SO):
        ref = OpalCLibrary(REF_SO)
        return lambda key, args: run_reference(ref, args)
    if os.path.exists(GOLDEN):
        with open(GOLDEN) as f:
            stored = json.load(f)
        return lambda key, args: stored[key]
    pytest.skip("neither oracle/_ref/libopal_ref.so nor tests/golden/oracle_vs_ref.json (make -C oracle && python tests/golden/make_golden.py)")


@pytest.mark.parametrize("seed", range(12))
@pytest.mark.parametrize("mode", ["NW", "HW", "OV", "SW"])
def test_score_end_matches_reference(oracle, reference, mode, seed):
    for st in (0, 1):
        args = score_end_args(mode, seed, st)
        want = reference(f"score_end/{mode}/{seed}/{st}", args)
        assert want is not None
        rc, got = search_dump(oracle, *args)
        assert rc == want[0] == 0
        for i, (g, w) in enumerate(zip(got, want[1])):
            if mode == "SW" and st == 1 and w[1] == 0:
                w = w[:2] + [-1, -1] + w[4:]  # Q2: the reference leaves garbage here
            assert g == w, (mode, st, i)


@pytest.mark.parametrize("seed", range(12))
def test_sw_alignment_matches_reference(oracle, reference, seed):
    args = sw_alignment_args(seed)
    want = reference(f"sw_alignment/{seed}", args)
    assert want is not None
    rc, got = search_dump(oracle, *args)
    assert rc == want[0] == 0
    assert got == want[1]


@pytest.mark.parametrize("seed", range(8))
@pytest.mark.parametrize("mode", ["NW", "HW", "OV"])
def test_global_alignment_matches_reference_where_it_survives(oracle, reference, mode, seed):
    compared = 0
    for i, args in global_alignment_args(mode, seed).items():
        want = reference(f"global_alignment/{mode}/{seed}/{i}", args)
        if want is None:
            continue  # reference crashed (Q8-Q10)
        rc, got = search_dump(oracle, *args)
        assert rc == 0
        assert got == want[1], (mode, i)
        compared += 1
    assert compared > 0
