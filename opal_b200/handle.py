"""Python mirror of include/opal_b200.h: the resident-database handle of libopal_b200.so.

No CPU implementation exists: constructing :class:`OpalB200` raises if the CUDA library has not
been built, and every search fails loudly (non-zero return code) when no sm_100 device is usable.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

from .capi import MODES, OpalCLibrary, SequenceDB, new_results, result_pointers

LIB_PATH = os.environ.get("OPAL_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libopal_b200.so")


class OpalB200(OpalCLibrary):
    """libopal_b200.so: the opal.h entry points (inherited) plus the opal_b200.h extensions."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build it with `make -C opal_b200/csrc` "
                               "(or __graft_entry__.build()); opal-b200 has no CPU fallback")
        super().__init__(path)
        L, vp, ci = self.lib, ctypes.c_void_p, ctypes.c_int
        L.opalb200_device_count.restype = ci
        L.opalb200_last_error.restype = ctypes.c_char_p
        L.opalb200_db_create.argtypes = [vp, ci, vp, ci]
        L.opalb200_db_create.restype = vp
        L.opalb200_db_create_multi.argtypes = [vp, ci, vp, vp, ci]
        L.opalb200_db_create_multi.restype = vp
        L.opalb200_db_devices.argtypes = [vp]
        L.opalb200_db_devices.restype = ci
        L.opalb200_db_create_sorted.argtypes = [vp, vp, vp, ci, ci]
        L.opalb200_db_create_sorted.restype = vp
        L.opalb200_db_search_batch.argtypes = [vp, ci, vp, vp, ci, ci, vp, ci, ci, ci, vp, vp, vp, ci, vp]
        L.opalb200_db_search_batch.restype = ci
        L.opalb200_db_search_batch_modes.argtypes = [vp, ci, vp, vp, vp, ci, ci, vp, ci, ci, vp, vp, vp, ci, vp]
        L.opalb200_db_search_batch_modes.restype = ci
        L.opalb200_db_search_results.argtypes = [vp, vp, ci, ci, ci, vp, ci, vp, ci, ci]
        L.opalb200_db_search_results.restype = ci
        L.opalb200_db_search_topk.argtypes = [vp, vp, ci, ci, ci, vp, ci, ci, ci, ci, vp, vp, ctypes.POINTER(ci)]
        L.opalb200_db_search_topk.restype = ci
        L.opalb200_db_destroy.argtypes = [vp]
        L.opalb200_db_destroy.restype = None
        L.opalb200_db_length.argtypes = [vp]
        L.opalb200_db_length.restype = ci
        L.opalb200_db_residues.argtypes = [vp]
        L.opalb200_db_residues.restype = ctypes.c_longlong
        L.opalb200_db_search.argtypes = [vp, vp, ci, ci, ci, vp, ci, ci, ci, vp, vp, vp, vp, vp]
        L.opalb200_db_search.restype = ci
        L.opalb200_db_search_pssm.argtypes = [vp, vp, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        L.opalb200_db_search_pssm.restype = ci
        L.opalb200_db_search_batch_pssm.argtypes = [vp, ci, vp, vp, vp, ci, ci, ci, ci, vp, vp, vp, ci, vp]
        L.opalb200_db_search_batch_pssm.restype = ci
        L.opalb200_db_search_results_pssm.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp, ci, ci]
        L.opalb200_db_search_results_pssm.restype = ci
        L.opalb200_db_search_topk_pssm.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp, vp, ctypes.POINTER(ci)]
        L.opalb200_db_search_topk_pssm.restype = ci
        L.opalb200_db_search_batch_topk.argtypes = [vp, ci, vp, vp, vp, ci, ci, vp, ci, ci, ci, vp, vp, ctypes.POINTER(ci), ci]
        L.opalb200_db_search_batch_topk.restype = ci
        L.opalb200_db_search_batch_topk_pssm.argtypes = [vp, ci, vp, vp, vp, vp, ci, ci, ci, ci, ci, vp, vp, ctypes.POINTER(ci), ci]
        L.opalb200_db_search_batch_topk_pssm.restype = ci
        L.opalb200_db_last_stats.argtypes = [vp] + [ctypes.POINTER(ci)] * 7
        L.opalb200_db_last_stats.restype = None
        L.opalb200_db_last_folded.argtypes = [vp]
        L.opalb200_db_last_folded.restype = ci
        L.opalb200_db_last_chained.argtypes = [vp]
        L.opalb200_db_last_chained.restype = ci
        L.opalb200_measure_dpx_peak.argtypes = [ci, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]
        L.opalb200_measure_dpx_peak.restype = ctypes.c_double
        L.opalb200_measure_dpx_peak_mix.argtypes = [ci, ci, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)]
        L.opalb200_measure_dpx_peak_mix.restype = ctypes.c_double
        L.opalb200_trim_cache.argtypes = []
        L.opalb200_trim_cache.restype = None

    def device_count(self):
        return int(self.lib.opalb200_device_count())

    def last_error(self):
        return self.lib.opalb200_last_error().decode()

    def create_db(self, db: SequenceDB, device=0):
        """opalb200_db_create on one device, or -- `device` a list of ordinals -- opalb200_db_create_multi."""
        if isinstance(device, (list, tuple)):
            devs = np.ascontiguousarray(device, dtype=np.int32)
            h = self.lib.opalb200_db_create_multi(db.pointers.ctypes.data, len(db), db.lengths.ctypes.data, devs.ctypes.data, int(devs.size))
        else:
            h = self.lib.opalb200_db_create(db.pointers.ctypes.data, len(db), db.lengths.ctypes.data, int(device))
        if not h:
            raise RuntimeError("opalb200_db_create failed: " + self.last_error())
        return ResidentDb(self, h, len(db))

    def create_db_sorted(self, residues, sorted_lengths, order=None, device=0):
        """opalb200_db_create_sorted: a database that is already packed (longest first, contiguous)."""
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        lens = np.ascontiguousarray(sorted_lengths, dtype=np.int32)
        buf = residues if residues.size else np.zeros(1, dtype=np.uint8)
        order_arr = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
        h = self.lib.opalb200_db_create_sorted(buf.ctypes.data, lens.ctypes.data,
                                               None if order_arr is None else order_arr.ctypes.data, int(lens.size), int(device))
        if not h:
            raise RuntimeError("opalb200_db_create_sorted failed: " + self.last_error())
        return ResidentDb(self, h, int(lens.size))

    def trim_cache(self):
        self.lib.opalb200_trim_cache()

    def measure_dpx_peak(self, device=0, mix=0):
        """(GCUPS the integer pipe can sustain, packed thread-instructions/s, kernel ms); mix 0 = SW, 1 = NW/HW/OV."""
        ips, ms = ctypes.c_double(0), ctypes.c_float(0)
        g = self.lib.opalb200_measure_dpx_peak_mix(int(device), int(mix), ctypes.byref(ips), ctypes.byref(ms))
        if g <= 0:
            raise RuntimeError("DPX probe failed: " + self.last_error())
        return float(g), float(ips.value), float(ms.value)


class ResidentDb:
    """A database packed once into one GPU's HBM (opalb200_db_create)."""

    def __init__(self, eng: OpalB200, handle, n):
        self.eng, self.handle, self.n = eng, handle, n

    def search(self, query, gap_open, gap_ext, score_matrix, alphabet_length, search_type, mode, skip=None):
        """Returns (rc, scores, endQuery, endTarget, device_ms); arrays are in caller order."""
        query = np.ascontiguousarray(query, dtype=np.uint8)
        sm = np.ascontiguousarray(score_matrix, dtype=np.int32).ravel()
        sc = np.zeros(self.n, dtype=np.int32)
        eq = np.full(self.n, -1, dtype=np.int32)
        et = np.full(self.n, -1, dtype=np.int32)
        ms = ctypes.c_float(0)
        if isinstance(mode, str):
            mode = MODES[mode]
        skp = None if skip is None else np.ascontiguousarray(skip, dtype=np.uint8)
        rc = self.eng.lib.opalb200_db_search(
            self.handle, query.ctypes.data, int(query.size), int(gap_open), int(gap_ext), sm.ctypes.data,
            int(alphabet_length), int(search_type), int(mode), None if skp is None else skp.ctypes.data,
            sc.ctypes.data, eq.ctypes.data, et.ctypes.data, ctypes.byref(ms))
        return rc, sc, eq, et, float(ms.value)

    def search_batch(self, queries, gap_open, gap_ext, score_matrix, alphabet_length, search_type, mode, in_flight=3, out=None):
        """opalb200_db_search_batch. Returns (rc, scores[nq, n], endQuery, endTarget, batch_ms); `out` = three
        preallocated int32 [nq, n] arrays to write into (entries that are not computed keep their old values)."""
        qs = [np.ascontiguousarray(q, dtype=np.uint8) for q in queries]
        qs = [q if q.size else np.zeros(1, dtype=np.uint8) for q in qs]
        nq = len(qs)
        ptrs = np.array([q.ctypes.data for q in qs], dtype=np.uint64)
        qlens = np.array([len(q) for q in queries], dtype=np.int32)
        sm = np.ascontiguousarray(score_matrix, dtype=np.int32).ravel()
        if out is not None:
            sc, eq, et = out
            assert all(a.shape == (nq, self.n) and a.dtype == np.int32 and a.flags["C_CONTIGUOUS"] for a in out)
        else:
            sc = np.zeros((nq, self.n), dtype=np.int32)
            eq = np.full((nq, self.n), -1, dtype=np.int32)
            et = np.full((nq, self.n), -1, dtype=np.int32)
        ms = ctypes.c_float(0)
        if isinstance(mode, (list, tuple)):  # one mode per search: opalb200_db_search_batch_modes
            modes = np.array([MODES[m] if isinstance(m, str) else int(m) for m in mode], dtype=np.int32)
            assert len(modes) == nq
            rc = self.eng.lib.opalb200_db_search_batch_modes(
                self.handle, nq, ptrs.ctypes.data, qlens.ctypes.data, modes.ctypes.data, int(gap_open), int(gap_ext), sm.ctypes.data,
                int(alphabet_length), int(search_type), sc.ctypes.data, eq.ctypes.data, et.ctypes.data,
                int(in_flight), ctypes.byref(ms))
            return rc, sc, eq, et, float(ms.value)
        if isinstance(mode, str):
            mode = MODES[mode]
        rc = self.eng.lib.opalb200_db_search_batch(
            self.handle, nq, ptrs.ctypes.data, qlens.ctypes.data, int(gap_open), int(gap_ext), sm.ctypes.data,
            int(alphabet_length), int(search_type), int(mode), sc.ctypes.data, eq.ctypes.data, et.ctypes.data,
            int(in_flight), ctypes.byref(ms))
        return rc, sc, eq, et, float(ms.value)

    def search_results(self, query, gap_open, gap_ext, score_matrix, alphabet_length, search_type, mode, results=None):
        """opalb200_db_search_results: opalSearchDatabase's records against the resident database. Returns (rc, results)."""
        query = np.ascontiguousarray(query, dtype=np.uint8)
        sm = np.ascontiguousarray(score_matrix, dtype=np.int32).ravel()
        if results is None:
            results = new_results(self.n)
        rp = result_pointers(results)
        qbuf = query if query.size else np.zeros(1, dtype=np.uint8)
        if isinstance(mode, str):
            mode = MODES[mode]
        rc = self.eng.lib.opalb200_db_search_results(
            self.handle, qbuf.ctypes.data, int(query.size), int(gap_open), int(gap_ext), sm.ctypes.data,
            int(alphabet_length), rp.ctypes.data, int(search_type), int(mode))
        return rc, results

    def search_topk(self, query, gap_open, gap_ext, score_matrix, alphabet_length, search_type, mode, k):
        """opalb200_db_search_topk. Returns (rc, indices[found], results[found])."""
        query = np.ascontiguousarray(query, dtype=np.uint8)
        sm = np.ascontiguousarray(score_matrix, dtype=np.int32).ravel()
        results = new_results(max(int(k), 1))
        rp = result_pointers(results)
        idx = np.full(max(int(k), 1), -1, dtype=np.int32)
        found = ctypes.c_int(0)
        qbuf = query if query.size else np.zeros(1, dtype=np.uint8)
        if isinstance(mode, str):
            mode = MODES[mode]
        rc = self.eng.lib.opalb200_db_search_topk(
            self.handle, qbuf.ctypes.data, int(query.size), int(gap_open), int(gap_ext), sm.ctypes.data,
            int(alphabet_length), int(search_type), int(mode), int(k), idx.ctypes.data, rp.ctypes.data, ctypes.byref(found))
        return rc, idx[:found.value], results[:found.value]

    # ---- position-specific scoring matrices: `pssm` is an int32 array of shape (Q, A); pssm[r, y] scores query position
    # r against residue code y, and the alphabet length is pssm.shape[1].  pssm=None with `query_length` searches an empty
    # query (or passes NULL, to see the call reject it for query_length > 0).
    @staticmethod
    def _pssm(pssm, query_length=None, alphabet_length=None):
        """(C pointer or None, the array kept alive, Q, A)"""
        if pssm is None:
            return None, None, int(query_length or 0), int(alphabet_length or 1)
        arr = np.ascontiguousarray(pssm, dtype=np.int32)
        if arr.ndim != 2:
            raise ValueError("pssm must have shape (queryLength, alphabetLength)")
        buf = arr if arr.size else np.zeros(1, dtype=np.int32)
        return buf.ctypes.data, buf, int(arr.shape[0]), int(arr.shape[1])

    def search_pssm(self, pssm, gap_open, gap_ext, search_type, mode, skip=None, query_length=None, alphabet_length=None):
        """opalb200_db_search_pssm. Returns (rc, scores, endQuery, endTarget, device_ms) like search()."""
        ptr, keep, Q, A = self._pssm(pssm, query_length, alphabet_length)
        sc = np.zeros(self.n, dtype=np.int32)
        eq = np.full(self.n, -1, dtype=np.int32)
        et = np.full(self.n, -1, dtype=np.int32)
        ms = ctypes.c_float(0)
        if isinstance(mode, str):
            mode = MODES[mode]
        skp = None if skip is None else np.ascontiguousarray(skip, dtype=np.uint8)
        rc = self.eng.lib.opalb200_db_search_pssm(
            self.handle, ptr, Q, A, int(gap_open), int(gap_ext), int(search_type), int(mode),
            None if skp is None else skp.ctypes.data, sc.ctypes.data, eq.ctypes.data, et.ctypes.data, ctypes.byref(ms))
        del keep
        return rc, sc, eq, et, float(ms.value)

    def search_batch_pssm(self, pssms, gap_open, gap_ext, search_type, modes, in_flight=3):
        """opalb200_db_search_batch_pssm: one PSSM and one mode per search (all PSSMs have the same alphabet length).
        Returns (rc, scores[ns, n], endQuery, endTarget, batch_ms)."""
        arrs = [np.ascontiguousarray(x, dtype=np.int32) for x in pssms]
        ns = len(arrs)
        A = int(arrs[0].shape[1]) if ns else 1
        if any(a.ndim != 2 or a.shape[1] != A for a in arrs):
            raise ValueError("every pssm must have shape (queryLength, alphabetLength) with the same alphabetLength")
        bufs = [a if a.size else np.zeros(1, dtype=np.int32) for a in arrs]
        ptrs = np.array([b.ctypes.data for b in bufs], dtype=np.uint64)
        qlens = np.array([a.shape[0] for a in arrs], dtype=np.int32)
        if isinstance(modes, (str, int)):
            modes = [modes] * ns
        md = np.array([MODES[m] if isinstance(m, str) else int(m) for m in modes], dtype=np.int32)
        assert len(md) == ns
        sc = np.zeros((ns, self.n), dtype=np.int32)
        eq = np.full((ns, self.n), -1, dtype=np.int32)
        et = np.full((ns, self.n), -1, dtype=np.int32)
        ms = ctypes.c_float(0)
        rc = self.eng.lib.opalb200_db_search_batch_pssm(
            self.handle, ns, ptrs.ctypes.data, qlens.ctypes.data, md.ctypes.data, A, int(gap_open), int(gap_ext),
            int(search_type), sc.ctypes.data, eq.ctypes.data, et.ctypes.data, int(in_flight), ctypes.byref(ms))
        return rc, sc, eq, et, float(ms.value)

    def search_results_pssm(self, pssm, gap_open, gap_ext, search_type, mode, query=None, results=None, query_length=None,
                            alphabet_length=None):
        """opalb200_db_search_results_pssm; `query` (the residues the PSSM was built for) labels alignment steps
        MATCH / MISMATCH and is required for OPAL_SEARCH_ALIGNMENT. Returns (rc, results)."""
        ptr, keep, Q, A = self._pssm(pssm, query_length, alphabet_length)
        qbuf = None if query is None else np.ascontiguousarray(query, dtype=np.uint8)
        if qbuf is not None and not qbuf.size:
            qbuf = np.zeros(1, dtype=np.uint8)
        if results is None:
            results = new_results(self.n)
        rp = result_pointers(results)
        if isinstance(mode, str):
            mode = MODES[mode]
        rc = self.eng.lib.opalb200_db_search_results_pssm(
            self.handle, None if qbuf is None else qbuf.ctypes.data, ptr, Q, A, int(gap_open), int(gap_ext), rp.ctypes.data,
            int(search_type), int(mode))
        del keep
        return rc, results

    def search_topk_pssm(self, pssm, gap_open, gap_ext, search_type, mode, k, query=None):
        """opalb200_db_search_topk_pssm. Returns (rc, indices[found], results[found])."""
        ptr, keep, Q, A = self._pssm(pssm)
        qbuf = None if query is None else np.ascontiguousarray(query, dtype=np.uint8)
        if qbuf is not None and not qbuf.size:
            qbuf = np.zeros(1, dtype=np.uint8)
        results = new_results(max(int(k), 1))
        rp = result_pointers(results)
        idx = np.full(max(int(k), 1), -1, dtype=np.int32)
        found = ctypes.c_int(0)
        if isinstance(mode, str):
            mode = MODES[mode]
        rc = self.eng.lib.opalb200_db_search_topk_pssm(
            self.handle, None if qbuf is None else qbuf.ctypes.data, ptr, Q, A, int(gap_open), int(gap_ext), int(search_type),
            int(mode), int(k), idx.ctypes.data, rp.ctypes.data, ctypes.byref(found))
        del keep
        return rc, idx[:found.value], results[:found.value]

    @staticmethod
    def _modes(modes, ns):
        if isinstance(modes, (str, int)):
            modes = [modes] * ns
        md = np.array([MODES[m] if isinstance(m, str) else int(m) for m in modes], dtype=np.int32)
        assert len(md) == ns
        return md

    def _batch_topk(self, call, ns, k):
        """Runs call(indices, result pointers, found) over ns x k slots; returns (rc, indices[ns, found], results[ns, found])."""
        k = int(k)
        results = new_results(max(ns * k, 1))
        rp = result_pointers(results)
        idx = np.full(max(ns * k, 1), -1, dtype=np.int32)
        found = ctypes.c_int(0)
        rc = call(idx.ctypes.data, rp.ctypes.data, ctypes.byref(found))
        f = found.value
        rows = idx[:ns * k].reshape(ns, k)[:, :f]
        recs = results[:ns * k].reshape(ns, k)[:, :f]
        return rc, np.ascontiguousarray(rows), np.ascontiguousarray(recs)

    def search_batch_topk(self, queries, gap_open, gap_ext, score_matrix, alphabet_length, search_type, modes, k, in_flight=3):
        """opalb200_db_search_batch_topk: one mode per search (or one mode for all). Returns (rc, indices[ns, found],
        results[ns, found]); row s is what search_topk returns for queries[s] (free_alignments takes one row at a time)."""
        qs = [np.ascontiguousarray(q, dtype=np.uint8) for q in queries]
        bufs = [q if q.size else np.zeros(1, dtype=np.uint8) for q in qs]
        ns = len(qs)
        ptrs = np.array([b.ctypes.data for b in bufs] or [0], dtype=np.uint64)
        qlens = np.array([q.size for q in qs] or [0], dtype=np.int32)
        md = self._modes(modes, ns)
        mdb = md if md.size else np.zeros(1, dtype=np.int32)
        sm = np.ascontiguousarray(score_matrix, dtype=np.int32).ravel()
        return self._batch_topk(lambda idx, rp, found: self.eng.lib.opalb200_db_search_batch_topk(
            self.handle, ns, ptrs.ctypes.data, qlens.ctypes.data, mdb.ctypes.data, int(gap_open), int(gap_ext), sm.ctypes.data,
            int(alphabet_length), int(search_type), int(k), idx, rp, found, int(in_flight)), ns, k)

    def search_batch_topk_pssm(self, pssms, gap_open, gap_ext, search_type, modes, k, queries=None, in_flight=3):
        """opalb200_db_search_batch_topk_pssm: one PSSM (shape (Q, A), the same A for all; None = a NULL PSSM) and one mode
        per search; `queries` (the residues each PSSM was built for) is required for OPAL_SEARCH_ALIGNMENT. Returns
        (rc, indices[ns, found], results[ns, found])."""
        arrs = [None if x is None else np.ascontiguousarray(x, dtype=np.int32) for x in pssms]
        ns = len(arrs)
        shaped = [a for a in arrs if a is not None]
        A = int(shaped[0].shape[1]) if shaped else 1
        if any(a.ndim != 2 or a.shape[1] != A for a in shaped):
            raise ValueError("every pssm must have shape (queryLength, alphabetLength) with the same alphabetLength")
        bufs = [None if a is None else (a if a.size else np.zeros(1, dtype=np.int32)) for a in arrs]
        ptrs = np.array([0 if b is None else b.ctypes.data for b in bufs] or [0], dtype=np.uint64)
        qlens = np.array([1 if a is None else a.shape[0] for a in arrs] or [0], dtype=np.int32)
        qbufs = None
        if queries is not None:
            qbufs = [np.ascontiguousarray(q, dtype=np.uint8) for q in queries]
            qbufs = [q if q.size else np.zeros(1, dtype=np.uint8) for q in qbufs]
            qptrs = np.array([q.ctypes.data for q in qbufs] or [0], dtype=np.uint64)
        md = self._modes(modes, ns)
        mdb = md if md.size else np.zeros(1, dtype=np.int32)
        return self._batch_topk(lambda idx, rp, found: self.eng.lib.opalb200_db_search_batch_topk_pssm(
            self.handle, ns, None if qbufs is None else qptrs.ctypes.data, ptrs.ctypes.data, qlens.ctypes.data, mdb.ctypes.data, A,
            int(gap_open), int(gap_ext), int(search_type), int(k), idx, rp, found, int(in_flight)), ns, k)

    def devices(self):
        return int(self.eng.lib.opalb200_db_devices(self.handle))

    def last_stats(self):
        v = [ctypes.c_int(0) for _ in range(7)]
        self.eng.lib.opalb200_db_last_stats(self.handle, *[ctypes.byref(x) for x in v])
        d = dict(zip(("kernel_launches", "rerun32", "G", "R", "passes", "warps_per_partition", "groups"), (x.value for x in v)))
        d["folded"] = int(self.eng.lib.opalb200_db_last_folded(self.handle))
        d["chained"] = int(self.eng.lib.opalb200_db_last_chained(self.handle))
        return d

    def close(self):
        if self.handle:
            self.eng.lib.opalb200_db_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
