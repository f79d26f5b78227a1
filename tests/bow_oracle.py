"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the BoW database oracle (tests/cpp/bow_oracle.c).

Used by tests/test_bow_database.py and tools/bow_bench.py as the checker and the reported host baseline; never by the
product package.  The C file is compiled into a temporary directory on first use, so the source tree may be read-only.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "bow_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="sfe_bow_oracle_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libbow_oracle.so")
        # -ffp-contract=off: every double operation individually rounded, as in the oracle's own build (oracle/Makefile)
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o", so,
                               _SRC, "-lm"])
        L = C.CDLL(so)
        vp, ci, cd = C.c_void_p, C.c_int, C.c_double
        L.orc_bow_score_l1.restype = cd
        L.orc_bow_score_l1.argtypes = [vp, vp, ci, vp, vp, ci]
        L.orc_bow_query_l1.restype = ci
        L.orc_bow_query_l1.argtypes = [vp, vp, vp, ci, ci, vp, vp, ci, ci, ci, vp, vp, ci, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _bow(v):
    ids, vals = v
    return np.ascontiguousarray(ids, np.int32), np.ascontiguousarray(vals, np.float64)


def bow_score_l1(a, b):
    """L1Scoring::score of two BowVectors given as (ids, values)."""
    (ai, av), (bi, bv) = _bow(a), _bow(b)
    return lib().orc_bow_score_l1(_p(ai), _p(av), len(ai), _p(bi), _p(bv), len(bi))


class BowIfile:
    """A BowVector database as DBoW2 keeps it for queryL1: per word, the entries holding it (ascending) with their values.
    Entry ids are the positions in `vectors`."""

    def __init__(self, vectors, n_words):
        self.n_words, self.n_entries = int(n_words), len(vectors)
        vs = [_bow(v) for v in vectors]
        ids = np.concatenate([i for i, _ in vs] + [np.zeros(0, np.int32)])
        vals = np.concatenate([x for _, x in vs] + [np.zeros(0, np.float64)])
        ent = np.repeat(np.arange(len(vs), dtype=np.int32), [len(i) for i, _ in vs])
        order = np.argsort(ids, kind="stable")  # stable: a word's entries stay in ascending id
        self.entry, self.value = ent[order].copy(), vals[order].copy()
        self.off = np.zeros(self.n_words + 1, np.int64)
        np.cumsum(np.bincount(ids, minlength=self.n_words)[:self.n_words], out=self.off[1:])

    def query(self, v, max_results, max_id=-1, dense=False):
        """TemplatedDatabase::query(v, ret, max_results, max_id) with L1 scoring -> (entries, scores)
        (+ the n_entries dense scores when dense=True)."""
        qi, qv = _bow(v)
        cap = max(self.n_entries, 1)
        ent, sc = np.zeros(cap, np.int32), np.zeros(cap, np.float64)
        d = np.zeros(self.n_entries, np.float64) if dense else None
        n = lib().orc_bow_query_l1(_p(self.off), _p(self.entry), _p(self.value), self.n_words, self.n_entries, _p(qi), _p(qv),
                                   len(qi), int(max_id), int(max_results), _p(ent), _p(sc), cap, _p(d))
        return (ent[:n].copy(), sc[:n].copy()) + ((d,) if dense else ())
