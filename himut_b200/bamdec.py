"""ctypes binding of the native BAM region decoder (include/himut_io.h, csrc/bamdec.c).

The GPU workers read their regions through this module: BGZF inflate on a pthread pool, record
parse and cs -> op stream in C, straight into the packed batch the C ABI takes.  It replaces
pysam's fetch + bamlib.BAM.__init__ + cslib.cs2tuple of the reference
(src/himut/caller.py:299, bamlib.py:15-32, cslib.py:7-44).  bamio.py / pack.py remain the
readable specification of the same rules (tests/test_bamdec.py compares the two byte for byte)
and provide the BAM writer used by the tests and tools.
"""
import ctypes as C
import os

import numpy as np

from . import abi, bamio, pack

_LIB = None
EXPORTS = ["hm_bam_open", "hm_bam_close", "hm_bam_error", "hm_bam_header_text", "hm_bam_n_refs", "hm_bam_ref_name",
           "hm_bam_ref_len", "hm_bam_read_batch", "hm_bam_set_option", "hm_bam_last_compact", "hm_bam_qnames_blob", "hm_bam_n_qnames", "hm_bam_qname", "hm_bam_window_qlens", "hm_bam_write_batch", "hm_bam_write_batch_tags", "hm_bam_write_batch_index", "hm_bq_compact_build",
           "hm_bq_compact_free", "hm_bam_region_plan", "hm_bam_intern_qnames", "hm_bam_set_reference", "hm_bam_index_kind"]


def lib_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libhimut_io.so")


def load():
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise RuntimeError("%s is missing: run `python __graft_entry__.py` to build it" % path)
        lib = C.CDLL(path)
        vp = C.c_void_p
        lib.hm_bam_open.argtypes = [C.c_char_p, C.POINTER(vp)]
        lib.hm_bam_close.argtypes = [vp]
        lib.hm_bam_close.restype = None
        lib.hm_bam_error.argtypes = [vp]
        lib.hm_bam_error.restype = C.c_char_p
        lib.hm_bam_header_text.argtypes = [vp]
        lib.hm_bam_header_text.restype = C.c_char_p
        lib.hm_bam_n_refs.argtypes = [vp]
        lib.hm_bam_ref_name.argtypes = [vp, C.c_int]
        lib.hm_bam_ref_name.restype = C.c_char_p
        lib.hm_bam_ref_len.argtypes = [vp, C.c_int]
        lib.hm_bam_read_batch.argtypes = [vp, C.c_int, C.c_int32, C.c_int32, C.c_int, C.POINTER(abi.hm_read_batch)]
        lib.hm_bam_set_option.argtypes = [vp, C.c_int, C.c_int]
        lib.hm_bam_last_compact.argtypes = [vp, C.POINTER(abi.hm_bq_compact)]
        lib.hm_bam_window_qlens.argtypes = [vp, C.c_int, C.c_int32, C.c_int32, C.c_int, vp, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.hm_bam_write_batch.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, C.c_char_p, C.POINTER(abi.hm_read_batch), C.c_int, C.c_int]
        lib.hm_bam_write_batch_tags.argtypes = lib.hm_bam_write_batch.argtypes + [C.c_int]
        lib.hm_bam_write_batch_index.argtypes = lib.hm_bam_write_batch_tags.argtypes + [C.c_int, C.c_int]
        lib.hm_bam_index_kind.argtypes = [vp]
        lib.hm_bq_compact_build.argtypes = [C.POINTER(abi.hm_read_batch), C.c_int, vp, vp, C.POINTER(vp), C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)]
        lib.hm_bq_compact_free.argtypes = [vp]
        lib.hm_bq_compact_free.restype = None
        lib.hm_bam_qnames_blob.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.hm_bam_n_qnames.argtypes = [vp]
        lib.hm_bam_n_qnames.restype = C.c_uint32
        lib.hm_bam_qname.argtypes = [vp, C.c_uint32]
        lib.hm_bam_qname.restype = C.c_char_p
        lib.hm_bam_region_plan.argtypes = [vp, C.c_int, C.c_int32, C.c_int32, C.POINTER(abi.hm_bgzf_plan)]
        lib.hm_bam_intern_qnames.argtypes = [vp, vp, vp, C.c_size_t, vp]
        lib.hm_bam_set_reference.argtypes = [vp, C.c_int, C.c_char_p, C.c_size_t]
        _LIB = lib
    return _LIB


def default_threads():
    t = os.environ.get("HIMUT_B200_DECODE_THREADS")
    if t:
        return max(1, int(t))
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def _view(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype)
    dt = np.dtype(dtype)
    buf = (C.c_char * (n * dt.itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dt, count=n)


def write_batch_bam(path, chrom, contig_len, batch, sample="synth", level=1, threads=None, tags="cs", index="bai", min_shift=14,
                    depth=None):
    """ReadBatch -> coordinate-sorted BAM + BAI, natively (same content as bamio.write_batch_bam, tags alike).
    index="csi" writes <path>.csi instead, with min_shift and depth (None: the smallest that holds the contig)."""
    if tags not in bamio.TAGS:
        raise ValueError("tags must be one of %s" % (bamio.TAGS,))
    if index not in ("bai", "csi"):
        raise ValueError("index must be 'bai' or 'csi'")
    if index == "bai" and contig_len > bamio.BAI_MAX_LEN:
        raise ValueError("a BAI cannot index a contig longer than 2^29 (%d): use index='csi'" % contig_len)
    rc = load().hm_bam_write_batch_index(os.fsencode(path), chrom.encode(), int(contig_len), sample.encode(), C.byref(batch.as_struct()),
                                         int(level), int(threads or default_threads()), bamio.TAGS.index(tags),
                                         int(min_shift) if index == "csi" else 0, int(depth or 0))
    if rc != 0:
        raise IOError("cannot write %s" % path)


def compact_bq(batch, threads=None):
    """abi.BqCompact of a batch: bitmap of the modal quality + exceptions (lossless; expanded on the device)"""
    L = load()
    mask = np.zeros(batch.bq.size // 8, np.uint8)
    exc_off = np.zeros(batch.n_reads + 1, np.uint64)
    exc_p, exc_n, modal = C.c_void_p(), C.c_uint64(0), C.c_uint8(0)
    rc = L.hm_bq_compact_build(C.byref(batch.as_struct()), int(threads or default_threads()), mask.ctypes.data_as(C.c_void_p),
                               exc_off.ctypes.data_as(C.c_void_p), C.byref(exc_p), C.byref(exc_n), C.byref(modal))
    if rc != 0:
        raise RuntimeError("hm_bq_compact_build failed: %d" % rc)
    n = int(exc_n.value)
    exc = np.zeros((n + 31) & ~15, np.uint8)
    if n:
        exc[:n] = _view(exc_p.value, n, np.uint8)
    L.hm_bq_compact_free(exc_p)
    return abi.BqCompact(mask, exc, exc_off, int(modal.value), n)


def _pos32(pos):
    """a region bound as the C ABI's int32: past 2^31 - 1 (the longest contig a BAM holds) it reads as the contig's end"""
    return int(min(pos, 2**31 - 1))


class NativeBam:
    """one open BAM (+ its BAI or CSI); read_batch() returns an abi.ReadBatch copied out of the handle"""

    def __init__(self, path, threads=None):
        self.lib = load()
        self.h = C.c_void_p()
        rc = self.lib.hm_bam_open(os.fsencode(path), C.byref(self.h))
        if rc != 0:
            why = self.lib.hm_bam_error(None)
            raise IOError("cannot open %s as BAM%s" % (path, ": " + why.decode() if why else ""))
        self.threads = threads or default_threads()
        self.references = [self.lib.hm_bam_ref_name(self.h, i).decode() for i in range(self.lib.hm_bam_n_refs(self.h))]
        self.lengths = [self.lib.hm_bam_ref_len(self.h, i) for i in range(len(self.references))]
        self.header_text = self.lib.hm_bam_header_text(self.h).decode()
        self.index_kind = ("none", "bai", "csi")[self.lib.hm_bam_index_kind(self.h)]
        self.has_index = self.index_kind != "none"

    def read_batch(self, chrom, start, end, copy=True, seq=True, compact=False, buffer_set=0):
        """seq=False: the batch comes without its 2-bit base stream (HM_BAM_OPT_NO_SEQ), as `call` and the phase
        edges want it; the decoder still checks the bases against the cs tag.
        compact=True: the qualities come as modal bitmap + exceptions, written by the record-parse pass itself
        (HM_BAM_OPT_COMPACT_BQ); returns (batch, abi.BqCompact) for Context.upload_compact — no one-byte-per-base
        stream exists on the host then (batch.bq is empty).
        buffer_set (copy=False): which of the handle's two buffer sets receives the batch; a batch stays valid until
        the next one decoded into the same set, so one can be uploaded while the next is decoded."""
        if chrom not in self.references:
            raise KeyError(chrom)
        for opt, val in ((1, 0 if seq else 1), (2, 1 if compact else 0), (3, int(buffer_set))):
            if self.lib.hm_bam_set_option(self.h, opt, val) != 0:
                raise RuntimeError(self.lib.hm_bam_error(self.h).decode())
        s = abi.hm_read_batch()
        rc = self.lib.hm_bam_read_batch(self.h, self.references.index(chrom), _pos32(max(start, 0)), _pos32(end), self.threads, C.byref(s))
        if rc != 0:
            raise pack.BatchFormatError(self.lib.hm_bam_error(self.h).decode())
        n = int(s.n_reads)
        cp = (lambda a: a.copy()) if copy else (lambda a: a)
        sizes = {"seq": int(s.seq_bytes), "bq": 0 if compact else int(s.bq_bytes), "ops": int(s.n_ops_total)}
        arrays = {}
        for name, dt in abi.ReadBatch._FIELDS:
            arrays[name] = cp(_view(getattr(s, name), sizes.get(name, n), dt))
        batch = abi.ReadBatch(keepalive=None if copy else self, **arrays)
        if not compact:
            return batch
        batch.bq_bytes_expanded = int(s.bq_bytes)
        q = abi.hm_bq_compact()
        if self.lib.hm_bam_last_compact(self.h, C.byref(q)) != 0:
            raise RuntimeError(self.lib.hm_bam_error(self.h).decode())
        n_exc = int(q.exc_bytes)
        mask = cp(_view(q.mask, int(q.mask_bytes), np.uint8))
        exc = cp(_view(q.exc, (n_exc + 31) & ~15, np.uint8))  # the decoder keeps 32 readable bytes past the last exception
        exc_off = cp(_view(q.exc_off, n + 1, np.uint64))
        return batch, abi.BqCompact(mask, exc, exc_off, int(q.modal), n_exc)

    def set_reference(self, chrom, seq):
        """the sequence of `chrom` (bytes or str, the whole contig: its length must be the @SQ LN), for its records with
        neither cs:Z nor MD:Z, which read_batch then decodes from CIGAR + reference (pack.parse_ref); None clears it.
        The handle keeps a reference to the bytes it reads."""
        if chrom not in self.references:
            raise KeyError(chrom)
        seq = seq.encode() if isinstance(seq, str) else (None if seq is None else bytes(seq))
        rc = self.lib.hm_bam_set_reference(self.h, self.references.index(chrom), seq, 0 if seq is None else len(seq))
        if rc != 0:
            self._ref = None
            raise pack.BatchFormatError(self.lib.hm_bam_error(self.h).decode())
        self._ref = seq

    def plan(self, chrom, start, end):
        """abi.hm_bgzf_plan of the records read_batch(chrom, start, end) visits, for Context.decode_region: the
        compressed blocks and the record starts the index knows, nothing inflated.  Valid until the next plan()."""
        if chrom not in self.references:
            raise KeyError(chrom)
        p = abi.hm_bgzf_plan()
        if self.lib.hm_bam_region_plan(self.h, self.references.index(chrom), _pos32(max(start, 0)), _pos32(end), C.byref(p)) != 0:
            raise pack.BatchFormatError(self.lib.hm_bam_error(self.h).decode())
        return p

    def intern_qnames(self, blob, off, n):
        """query-name ids (the ones read_batch gives) of n NUL-terminated names, name i at blob + off[i]"""
        ids = np.zeros(n, np.uint32)
        off = np.ascontiguousarray(off, np.uint64)
        blob_p = blob if isinstance(blob, int) else blob.ctypes.data
        if n and self.lib.hm_bam_intern_qnames(self.h, C.c_void_p(blob_p), off.ctypes.data_as(C.c_void_p), n, ids.ctypes.data_as(C.c_void_p)) != 0:
            raise RuntimeError(self.lib.hm_bam_error(self.h).decode())
        return ids

    def window_qlens(self, chrom, start, end):
        """len(query_sequence) of the records overlapping [start, end) with MAPQ > 0 and tp:A:P, fetch order
        (the list bamlib.get_thresholds builds per window, src/himut/bamlib.py:156-164)"""
        rid = self.references.index(chrom)
        cap = 4096
        while True:
            out = np.empty(cap, np.int32)
            n = C.c_size_t(0)
            rc = self.lib.hm_bam_window_qlens(self.h, rid, _pos32(max(start, 0)), _pos32(end), self.threads, out.ctypes.data_as(C.c_void_p), cap, C.byref(n))
            if rc == 3:  # HM_ERR_CAPACITY
                cap = int(n.value)
                continue
            if rc != 0:
                raise pack.BatchFormatError(self.lib.hm_bam_error(self.h).decode())
            return out[: int(n.value)]

    def n_qnames(self):
        return int(self.lib.hm_bam_n_qnames(self.h))

    def qname(self, i):
        v = self.lib.hm_bam_qname(self.h, i)
        return None if v is None else v.decode()

    def qnames_blob(self, flags):
        """b"name\\n..." of the ids whose flag is set (flags: uint8 per qname id, as Context.qname_seen / QnameTally keep them)"""
        flags = np.ascontiguousarray(flags, np.uint8)
        need = C.c_size_t(0)
        self.lib.hm_bam_qnames_blob(self.h, flags.ctypes.data_as(C.c_void_p), flags.size, None, 0, C.byref(need))
        buf = C.create_string_buffer(max(int(need.value), 1))
        rc = self.lib.hm_bam_qnames_blob(self.h, flags.ctypes.data_as(C.c_void_p), flags.size, buf, int(need.value), C.byref(need))
        if rc != 0 and need.value:
            raise RuntimeError("hm_bam_qnames_blob failed: %d" % rc)
        return buf.raw[: int(need.value)]

    def close(self):
        if self.h:
            self.lib.hm_bam_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
