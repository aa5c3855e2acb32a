"""Test infrastructure: ctypes wrapper of tests/track_oracle.c, the CPU oracle's normcounts with the callable-base track
(runs of hm_callable_run, abi.RUN_DTYPE).  The library is compiled on first use into a temporary directory (the tree
may be read-only), with the oracle's flags (oracle/Makefile)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from himut_b200 import abi
from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "track_oracle.c"), os.path.join(_ROOT, "oracle", "himut_oracle.c"),
            os.path.join(_ROOT, "include", "himut_b200.h")]
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256()
        for s in _SOURCES:
            with open(s, "rb") as f:
                h.update(f.read())
        path = os.path.join(tempfile.gettempdir(), "himut_track_oracle_%d_%s.so" % (os.getuid(), h.hexdigest()[:16]))
        if not os.path.exists(path):
            tmp = "%s.%d.tmp" % (path, os.getpid())
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-std=c11", "-shared",
                                   "-o", tmp, _SOURCES[0], "-lm"])
            os.replace(tmp, path)
        _LIB = C.CDLL(path)
    return _LIB


def normcounts_chunks_track(params, batch, refseq, chunks, common=None, pon=None, phase=None, alt_order=None, qseen=None):
    """oracle.normcounts_chunks with the callable-base track -> (ccs_tri[33], ref_tri[33], log[14], n_alt_tie,
    runs: abi.RUN_DTYPE in chunk order, then position order)"""
    _p = oracle._p
    common = np.zeros(0, np.uint64) if common is None else np.ascontiguousarray(common, np.uint64)
    pon = np.zeros(0, np.uint64) if pon is None else np.ascontiguousarray(pon, np.uint64)
    chunks = np.ascontiguousarray(chunks, dtype=abi.CHUNK_DTYPE)
    ph, keep = oracle._phase_struct(phase)
    ref = np.frombuffer(refseq, dtype=np.uint8)
    ao = None if alt_order is None else np.ascontiguousarray(alt_order, np.uint8)
    cap = 4096
    while True:
        ccs = np.zeros(abi.TRI_BINS, np.int64)
        rt = np.zeros(abi.TRI_BINS, np.int64)
        log = np.zeros(abi.NORM_LOG_LEN, np.int64)
        ties = C.c_int64(0)
        runs = np.zeros(cap, abi.RUN_DTYPE)
        n = C.c_size_t(0)
        rc = lib().trk_normcounts_chunks_track(
            C.byref(params), C.byref(batch.as_struct()), _p(ref), C.c_size_t(ref.size), _p(chunks),
            C.c_size_t(len(chunks)), _p(common), C.c_size_t(common.size), _p(pon), C.c_size_t(pon.size),
            C.byref(ph) if ph is not None else None, _p(ao), _p(ccs), _p(rt), _p(log), C.byref(ties),
            None if qseen is None else _p(qseen), C.c_size_t(0 if qseen is None else qseen.size),
            _p(runs), C.c_size_t(cap), C.byref(n))
        if rc == abi.HM_ERR_CAPACITY:
            cap = int(n.value)
            continue
        if rc != 0:
            raise RuntimeError("trk_normcounts_chunks_track failed: %d" % rc)
        return ccs, rt, log, ties.value, runs[: n.value].copy()
