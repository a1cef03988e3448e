"""Helpers of the PSSM tests: the oracle's PSSM restatement (tests/oracle_pssm.c, compiled on first use into a temporary
directory), an independent numpy Gotoh with the library's end-location key, and the PSSM replay of an alignment."""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile
import threading

import numpy as np

from _util import ROOT, OPAL_SEARCH_ALIGNMENT, get_alignment, new_results
from opal_b200.capi import result_pointers

_lock = threading.Lock()
_lib = None


def pssm_oracle():
    """ctypes handle of tests/oracle_pssm.c (the oracle, plus oracle_search_pssm)."""
    global _lib
    with _lock:
        if _lib is None:
            out = os.path.join(tempfile.mkdtemp(prefix="oracle_pssm_"), "liboracle_pssm.so")
            subprocess.check_call([os.environ.get("CC", "cc"), "-std=c11", "-O2", "-Wall", "-fPIC", "-shared", "-o", out,
                                   os.path.join(ROOT, "tests", "oracle_pssm.c")])
            lib = ctypes.CDLL(out, mode=ctypes.RTLD_LOCAL)
            vp, ci = ctypes.c_void_p, ctypes.c_int
            lib.oracle_search_pssm.argtypes = [vp, vp, ci, vp, ci, vp, ci, ci, ci, vp, ci, ci]
            lib.oracle_search_pssm.restype = ci
            _lib = lib
    return _lib


def oracle_search_pssm(query, pssm, db, go, ge, search_type, mode, results=None):
    """oracle_search_pssm over a SequenceDB. `query` may be None below OPAL_SEARCH_ALIGNMENT. Returns (rc, results)."""
    pssm = np.ascontiguousarray(pssm, dtype=np.int32)
    q_len, alen = pssm.shape
    pbuf = pssm if pssm.size else np.zeros(1, dtype=np.int32)
    qbuf = None if query is None else np.ascontiguousarray(query, dtype=np.uint8)
    if qbuf is not None and not qbuf.size:
        qbuf = np.zeros(1, dtype=np.uint8)
    res = new_results(len(db)) if results is None else results
    rp = result_pointers(res) if len(db) else np.zeros(1, dtype=np.uint64)
    rc = pssm_oracle().oracle_search_pssm(None if qbuf is None else qbuf.ctypes.data, pbuf.ctypes.data, int(q_len),
                                          db.pointers.ctypes.data, len(db), db.lengths.ctypes.data, int(go), int(ge),
                                          int(alen), rp.ctypes.data, int(search_type), int(mode))
    return rc, res


def matrix_pssm(query, matrix, alen):
    """The PSSM that scores exactly like (query, matrix): row r = matrix row of query[r]."""
    m = np.asarray(matrix, dtype=np.int32).reshape(alen, alen)
    return np.ascontiguousarray(m[np.asarray(query, dtype=np.int64)]).reshape(len(query), alen)


def noisy_pssm(query, matrix, alen, rng, noise=3):
    """matrix rows of the query plus independent per-position noise in [-noise, noise]: not expressible as a matrix."""
    p = matrix_pssm(query, matrix, alen).astype(np.int64)
    return (p + rng.integers(-noise, noise + 1, p.shape)).astype(np.int32)


def gotoh(pssm, t, go, ge, mode):
    """Score and end location of one target, straight from the definitions (independent of the oracle): the maximal
    score among the cells `mode` allows an alignment to end in; ties -> smallest target index, then query index."""
    P = np.asarray(pssm, dtype=np.int64)
    Q, T = P.shape[0], len(t)
    NEG = -(1 << 50)
    sw = mode == "SW"
    if Q == 0 or T == 0:
        if mode == "NW":
            sc = 0 if Q == T == 0 else -go - (max(Q, T) - 1) * ge
        elif mode == "HW" and Q > 0:
            sc = -go - (Q - 1) * ge
        else:
            sc = 0
        return (sc, -1, -1) if sw else (sc, Q - 1, T - 1)
    H = np.full((Q + 1, T + 1), NEG, dtype=np.int64)
    E = np.full((Q + 1, T + 1), NEG, dtype=np.int64)
    F = np.full((Q + 1, T + 1), NEG, dtype=np.int64)
    H[0, 0] = 0
    for r in range(1, Q + 1):
        H[r, 0] = 0 if mode in ("SW", "OV") else -go - (r - 1) * ge
    for c in range(1, T + 1):
        H[0, c] = -go - (c - 1) * ge if mode == "NW" else 0
    for c in range(1, T + 1):
        y = int(t[c - 1])
        for r in range(1, Q + 1):
            E[r, c] = max(H[r, c - 1] - go, E[r, c - 1] - ge)
            F[r, c] = max(H[r - 1, c] - go, F[r - 1, c] - ge)
            h = max(E[r, c], F[r, c], H[r - 1, c - 1] + P[r - 1, y])
            H[r, c] = max(h, 0) if sw else h
    if mode == "NW":
        return int(H[Q, T]), Q - 1, T - 1
    if sw:
        cells = [(r, c) for c in range(T) for r in range(Q)]
    elif mode == "HW":
        cells = [(Q - 1, c) for c in range(T)]
    else:
        cells = [(Q - 1, c) for c in range(T)] + [(r, T - 1) for r in range(Q)]
    best = max(cells, key=lambda rc: (H[rc[0] + 1, rc[1] + 1], -rc[1], -rc[0]))
    sc = int(H[best[0] + 1, best[1] + 1])
    if sw and sc == 0:
        return 0, -1, -1
    return sc, best[0], best[1]


def replay_ok(query, pssm, t, res, i, go, ge):
    """Record i's alignment: starts at its start, ends at its end, scores exactly its score under the PSSM, and its
    MATCH / MISMATCH labels agree with `query`."""
    ops = get_alignment(res, i)
    qi, ti = int(res["startLocationQuery"][i]), int(res["startLocationTarget"][i])
    if qi < 0 or ti < 0:
        return False
    sc, prev = 0, -1
    for op in ops:
        op = int(op)
        if op in (0, 3):
            if qi >= len(query) or ti >= len(t) or (query[qi] == t[ti]) != (op == 0):
                return False
            sc += int(pssm[qi][t[ti]])
            qi += 1
            ti += 1
        elif op == 1:
            sc -= ge if prev == 1 else go
            qi += 1
        elif op == 2:
            sc -= ge if prev == 2 else go
            ti += 1
        else:
            return False
        prev = op
    return (qi - 1 == int(res["endLocationQuery"][i]) and ti - 1 == int(res["endLocationTarget"][i])
            and sc == int(res["score"][i]))


__all__ = ["pssm_oracle", "oracle_search_pssm", "matrix_pssm", "noisy_pssm", "gotoh", "replay_ok", "OPAL_SEARCH_ALIGNMENT"]
