"""ctypes binding of libhimut_b200.so (include/himut_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is usable the
calls raise.  Build with `python -c "import __graft_entry__ as g; g.build()"`.
"""
import ctypes as C
import os

import numpy as np

from . import abi, pack

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HIMUT_B200_LIB") or os.path.join(_HERE, "libhimut_b200.so")  # override: instrumented builds
_LIB = None

# every symbol include/himut_b200.h declares (tests/test_abi.py checks the export table)
EXPORTS = [
    "hm_abi_version", "hm_create", "hm_destroy", "hm_last_error", "hm_set_params", "hm_set_site_sets",
    "hm_set_phase_sets", "hm_upload_batch", "hm_call_chunks", "hm_call_batch", "hm_normcounts_chunks",
    "hm_read_stats", "hm_last_timing", "hm_last_kernel_times", "hm_set_stream", "hm_host_register",
    "hm_host_unregister", "hm_abi_sizeof", "hm_last_records", "hm_qname_seen", "hm_set_reference", "hm_ref_tricounts", "hm_last_norm_exact_sites",
    "hm_phase_edges_begin", "hm_phase_edges_add", "hm_phase_edges_end", "hm_upload_batch_compact", "hm_call_batch_compact", "hm_call_chunks_async", "hm_records_wait", "hm_set_option", "hm_last_call_path", "hm_call_chunks_submit", "hm_call_chunks_collect", "hm_device_count", "hm_upload_batch_compact_begin", "hm_upload_wait",
    "hm_decode_bam_begin", "hm_decode_bam_names", "hm_decode_bam_end", "hm_batch_read_back", "hm_inflate_device_test",
    "hm_decode_bam_begin_opts", "hm_batch_read_back_seq",
]


class HimutError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("himut_b200 error %d: %s" % (code, msg))
        self.code = code


def load():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing (no CPU fallback exists): build it with "
                               "`python -c 'import __graft_entry__ as g; g.build()'`" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        vp, sz = C.c_void_p, C.c_size_t
        lib.hm_abi_version.restype = C.c_int
        lib.hm_device_count.restype = C.c_int
        lib.hm_abi_sizeof.restype = sz
        lib.hm_abi_sizeof.argtypes = [C.c_int]
        lib.hm_create.argtypes = [C.c_int, C.POINTER(vp)]
        lib.hm_destroy.argtypes = [vp]
        lib.hm_destroy.restype = None
        lib.hm_last_error.argtypes = [vp]
        lib.hm_last_error.restype = C.c_char_p
        lib.hm_set_params.argtypes = [vp, C.POINTER(abi.hm_params)]
        lib.hm_set_site_sets.argtypes = [vp, vp, sz, vp, sz]
        lib.hm_set_phase_sets.argtypes = [vp, vp, vp, vp, vp, sz, vp, sz]
        lib.hm_upload_batch.argtypes = [vp, C.POINTER(abi.hm_read_batch)]
        lib.hm_call_chunks.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz), vp]
        lib.hm_call_chunks_async.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz), vp]
        lib.hm_call_batch.argtypes = [vp, C.POINTER(abi.hm_read_batch), vp, sz, vp, sz, C.POINTER(sz), vp]
        lib.hm_upload_batch_compact.argtypes = [vp, C.POINTER(abi.hm_read_batch), C.POINTER(abi.hm_bq_compact)]
        lib.hm_upload_batch_compact_begin.argtypes = [vp, C.POINTER(abi.hm_read_batch), C.POINTER(abi.hm_bq_compact)]
        lib.hm_upload_wait.argtypes = [vp]
        lib.hm_call_batch_compact.argtypes = [vp, C.POINTER(abi.hm_read_batch), C.POINTER(abi.hm_bq_compact), vp, sz, vp, sz,
                                              C.POINTER(sz), vp]
        lib.hm_normcounts_chunks.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp, C.POINTER(C.c_int64)]
        lib.hm_read_stats.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        lib.hm_last_timing.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        lib.hm_last_kernel_times.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
        lib.hm_last_records.argtypes = [vp, vp, sz, C.POINTER(sz)]
        lib.hm_records_wait.argtypes = [vp]
        lib.hm_call_chunks_submit.argtypes = [vp, vp, sz]
        lib.hm_call_chunks_collect.argtypes = [vp, vp, sz, C.POINTER(sz), vp]
        lib.hm_set_option.argtypes = [vp, C.c_int, C.c_int]
        lib.hm_qname_seen.argtypes = [vp, vp, sz, C.POINTER(sz)]
        lib.hm_set_reference.argtypes = [vp, vp, sz]
        lib.hm_ref_tricounts.argtypes = [vp, vp, sz, vp]
        lib.hm_last_norm_exact_sites.argtypes = [vp, C.POINTER(C.c_uint64)]
        lib.hm_phase_edges_begin.argtypes = [vp, vp, vp, sz, C.c_uint32]
        lib.hm_phase_edges_add.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_uint32)]
        lib.hm_phase_edges_end.argtypes = [vp, vp, sz]
        lib.hm_set_stream.argtypes = [vp, vp]
        lib.hm_last_call_path.argtypes = [vp]
        lib.hm_last_call_path.restype = C.c_int
        lib.hm_host_register.argtypes = [vp, vp, sz]
        lib.hm_host_unregister.argtypes = [vp, vp]
        lib.hm_decode_bam_begin.argtypes = [vp, C.POINTER(abi.hm_bgzf_plan), C.c_int, C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]
        lib.hm_decode_bam_begin_opts.argtypes = [vp, C.POINTER(abi.hm_bgzf_plan), C.c_int, C.c_int32, C.c_int32, C.c_uint32,
                                                 C.POINTER(C.c_uint64)]
        lib.hm_decode_bam_names.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_uint64)]
        lib.hm_decode_bam_end.argtypes = [vp, vp]
        lib.hm_batch_read_back.argtypes = [vp, C.POINTER(abi.hm_read_batch)] + [vp] * 11
        lib.hm_batch_read_back_seq.argtypes = [vp, vp, vp, C.POINTER(C.c_uint64)]
        lib.hm_inflate_device_test.argtypes = [vp, C.c_char_p, sz, vp, sz, C.c_uint32]
        _LIB = lib
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def device_count():
    """cudaGetDeviceCount through the library (0 when no driver / device)"""
    return int(load().hm_device_count())


class DecodedRegion:
    """what Context.decode_region leaves on the host: the per-read coordinates the chunk table needs"""

    chunk_table = abi.ReadBatch.chunk_table

    def __init__(self, tstart, tend):
        self.n_reads, self.tstart, self.tend = int(tstart.size), tstart, tend


class Context:
    """one hm_ctx: single-threaded, bound to one GPU; create it inside the worker process"""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.hm_create(int(device), C.byref(h))
        if rc != 0:
            raise HimutError(rc, "hm_create(device=%d) failed: no usable CUDA device (there is no CPU fallback)" % device)
        self.h = h
        self.device = int(device)
        self._keep = {}

    def close(self):
        if getattr(self, "h", None):
            for buf in getattr(self, "_outs", None) or ():  # the two page-locked record buffers
                if buf is not None:
                    self.lib.hm_records_wait(self.h)
                    self.lib.hm_host_unregister(self.h, _p(buf))
            self._outs = None
            for a in list(self._keep.values()):
                self.lib.hm_host_unregister(self.h, _p(a))
            self._keep = {}
            self.lib.hm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown: the driver reclaims the context
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _chk(self, rc):
        if rc != 0:
            raise HimutError(rc, self.lib.hm_last_error(self.h).decode())

    # ---- configuration ----------------------------------------------------------------
    def set_params(self, params):
        self._chk(self.lib.hm_set_params(self.h, C.byref(params)))

    def set_site_sets(self, common=None, pon=None):
        common = np.zeros(0, np.uint64) if common is None else np.ascontiguousarray(common, np.uint64)
        pon = np.zeros(0, np.uint64) if pon is None else np.ascontiguousarray(pon, np.uint64)
        self._chk(self.lib.hm_set_site_sets(self.h, _p(common), common.size, _p(pon), pon.size))

    def set_phase_sets(self, phase):
        k = {n: np.ascontiguousarray(phase[n], dt) for n, dt in
             (("hpos", np.int32), ("href", np.uint8), ("halt", np.uint8), ("hbit", np.uint8), ("set_off", np.uint64))}
        self._chk(self.lib.hm_set_phase_sets(self.h, _p(k["hpos"]), _p(k["href"]), _p(k["halt"]), _p(k["hbit"]),
                                             k["hpos"].size, _p(k["set_off"]), max(k["set_off"].size - 1, 0)))

    def set_stream(self, cuda_stream):
        self._chk(self.lib.hm_set_stream(self.h, C.c_void_p(cuda_stream)))

    def pin(self, batch):
        """page-lock the batch's big arrays so uploads run at PCIe speed"""
        for name in ("seq", "bq", "ops"):
            a = getattr(batch, name)
            if a.size:
                self._chk(self.lib.hm_host_register(self.h, _p(a), a.nbytes))
                self._keep[id(a)] = a

    def unpin(self, batch):
        for name in ("seq", "bq", "ops"):
            a = getattr(batch, name)
            if id(a) in self._keep:
                self.lib.hm_host_unregister(self.h, _p(a))
                del self._keep[id(a)]

    # ---- work -------------------------------------------------------------------------
    def upload(self, batch):
        self._chk(self.lib.hm_upload_batch(self.h, C.byref(batch.as_struct())))

    def upload_compact(self, batch, cq, wait=True):
        """upload with the quality stream as modal bitmap + exceptions (abi.BqCompact); expanded on the device.
        wait=False: returns as soon as the copies are enqueued — the arrays of `batch` and `cq` must stay untouched until
        upload_wait() (calls may be submitted meanwhile: they run behind the copies)"""
        if wait:
            self._chk(self.lib.hm_upload_batch_compact(self.h, C.byref(batch.as_struct()), C.byref(cq.struct)))
        else:
            self._uploading = (batch, cq)  # alive until the copies are done
            self._chk(self.lib.hm_upload_batch_compact_begin(self.h, C.byref(batch.as_struct()), C.byref(cq.struct)))

    def decode_region(self, reader, chrom, start, end, seq=False):
        """the records reader.read_batch(chrom, start, end, seq=seq) returns, decoded on the device from the
        compressed file (reader: bamdec.NativeBam) and left resident as upload() would leave that batch: seq=True
        with the 2-bit base stream normcounts reads, seq=False without it (`call`, phase edges).  Query-name ids come
        from the reader's table.  Rejected input raises pack.BatchFormatError with the host decoder's text.
        -> DecodedRegion (n_reads, tstart, tend, chunk_table)"""
        rid = reader.references.index(chrom)
        start, end = int(max(start, 0)), int(min(end, reader.lengths[rid]))
        plan = reader.plan(chrom, start, end)
        n = C.c_uint64(0)
        if seq:
            rc = self.lib.hm_decode_bam_begin_opts(self.h, C.byref(plan), rid, start, end, abi.HM_DECODE_SEQ, C.byref(n))
        else:
            rc = self.lib.hm_decode_bam_begin(self.h, C.byref(plan), rid, start, end, C.byref(n))
        if rc == abi.HM_ERR_ARG:
            raise pack.BatchFormatError(self.lib.hm_last_error(self.h).decode())
        self._chk(rc)
        self.last_decode_times = self.last_kernel_times()
        names, off, ts, te = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._chk(self.lib.hm_decode_bam_names(self.h, C.byref(names), C.byref(off), C.byref(ts), C.byref(te), C.byref(n)))
        nr = int(n.value)
        view = lambda p, dt: np.ctypeslib.as_array(C.cast(p, C.POINTER(dt)), (nr,)) if nr else np.zeros(0, dt)
        ids = reader.intern_qnames(names.value or 0, view(off, C.c_uint64), nr)
        self._chk(self.lib.hm_decode_bam_end(self.h, _p(ids)))
        return DecodedRegion(view(ts, C.c_int32).copy(), view(te, C.c_int32).copy())

    def read_back(self, seq=False):
        """diagnostics (tests): the resident batch as an abi.ReadBatch (mapq, qname_id, qualities, ops included; flags
        as uploaded by a decoder: 0); seq=True also brings back seq_off / seq (empty when the batch has no base
        stream), seq=False leaves them empty"""
        s = abi.hm_read_batch()
        self._chk(self.lib.hm_batch_read_back(self.h, C.byref(s), *([None] * 11)))
        n, nbq, nops = int(s.n_reads), int(s.bq_bytes), int(s.n_ops_total)
        a = dict(tstart=np.zeros(n, np.int32), tend=np.zeros(n, np.int32), qstart=np.zeros(n, np.int32), qlen=np.zeros(n, np.int32),
                 mapq=np.zeros(n, np.uint8), qname_id=np.zeros(n, np.uint32), bq_off=np.zeros(n, np.uint64), op_off=np.zeros(n, np.uint64),
                 n_ops=np.zeros(n, np.uint32), bq=np.zeros(nbq, np.uint8), ops=np.zeros(nops, np.uint32))
        order = ("tstart", "tend", "qstart", "qlen", "mapq", "qname_id", "bq_off", "op_off", "n_ops", "bq", "ops")
        self._chk(self.lib.hm_batch_read_back(self.h, C.byref(s), *[_p(a[k]) for k in order]))
        seq_off, seq_b = np.zeros(0, np.uint64), np.zeros(0, np.uint8)
        if seq:
            nseq = C.c_uint64(0)
            self._chk(self.lib.hm_batch_read_back_seq(self.h, None, None, C.byref(nseq)))
            if nseq.value:
                seq_off, seq_b = np.zeros(n, np.uint64), np.zeros(int(nseq.value), np.uint8)
                self._chk(self.lib.hm_batch_read_back_seq(self.h, _p(seq_off), _p(seq_b), C.byref(nseq)))
        return abi.ReadBatch(flags=np.zeros(n, np.uint8), seq_off=seq_off, seq=seq_b, **a)

    def inflate_test(self, comp, n, crc):
        """tests: the device decoder of k_bgzf_inflate on one raw DEFLATE stream -> (rc, bytes)"""
        out = np.zeros(max(n, 1), np.uint8)
        rc = self.lib.hm_inflate_device_test(self.h, bytes(comp), len(comp), _p(out), n, crc & 0xffffffff)
        if rc == abi.HM_ERR_CUDA:
            self._chk(rc)
        return rc, out[:n].tobytes()

    def upload_wait(self):
        """the copies of the last upload_compact(..., wait=False) are done: its arrays may be reused"""
        self._chk(self.lib.hm_upload_wait(self.h))
        self._uploading = None

    def call_batch_compact(self, batch, cq, chunks, cap=None, view=False):
        """call_batch with the compact quality stream: fewer bytes over PCIe, identical records"""
        return self._call(self.lib.hm_call_batch_compact, (C.byref(batch.as_struct()), C.byref(cq.struct)), chunks, cap, view)

    def pin_arrays(self, arrays):
        for a in arrays:
            if a.size and id(a) not in self._keep:
                self._chk(self.lib.hm_host_register(self.h, _p(a), a.nbytes))
                self._keep[id(a)] = a

    def unpin_arrays(self, arrays):
        for a in arrays:
            if id(a) in self._keep:
                self.lib.hm_host_unregister(self.h, _p(a))
                del self._keep[id(a)]

    def _out_buffer(self, cap):
        """persistent page-locked record buffers (records are copied device -> here directly); two of them,
        used alternately, so that an asynchronous call's records stay valid while the next call runs"""
        bufs = getattr(self, "_outs", None)
        if bufs is None:
            bufs = self._outs = [None, None]
            self._out_i = 0
        self._out_i ^= 1
        buf = bufs[self._out_i]
        if buf is None or buf.shape[0] < cap:
            self._chk(self.lib.hm_records_wait(self.h))
            if buf is not None:
                self.lib.hm_host_unregister(self.h, _p(buf))
            buf = np.empty(cap, dtype=abi.SITE_DTYPE)
            self._chk(self.lib.hm_host_register(self.h, _p(buf), buf.nbytes))
            bufs[self._out_i] = buf
        return buf

    def _call(self, fn, head, chunks, cap, view):
        chunks = np.ascontiguousarray(chunks, dtype=abi.CHUNK_DTYPE)
        out = self._out_buffer(int(cap or getattr(self, "_cap", 65536)))
        n = C.c_size_t(0)
        log = np.zeros(abi.CALL_LOG_LEN, np.int64)
        rc = fn(self.h, *head, _p(chunks), len(chunks), _p(out), out.shape[0], C.byref(n), _p(log))
        if rc == abi.HM_ERR_CAPACITY:  # results are kept by the library: fetch, do not recompute
            self._cap = int(n.value) + int(n.value) // 4 + 1024
            out = self._out_buffer(self._cap)
            rc = self.lib.hm_last_records(self.h, _p(out), out.shape[0], C.byref(n))
        self._chk(rc)
        res = out[: n.value]
        return (res if view else res.copy()), log

    def call_chunks(self, chunks, cap=None, view=False, wait=True):
        """`himut call` over the resident batch -> (records, log[15]).
        view=True returns a view of one of the context's two pinned buffers, valid until the second next call.
        wait=False (needs view=True): the records may still be on their way when this returns — the copy overlaps
        the next call's kernels; records_wait() completes them."""
        if not wait and not view:
            raise ValueError("wait=False needs view=True")
        return self._call(self.lib.hm_call_chunks if wait else self.lib.hm_call_chunks_async, (), chunks, cap, view)

    def call_chunks_submit(self, chunks):
        """enqueue the device path of a call and return at once (call_chunks_collect finishes it): several contexts
        on one GPU are submitted back to back so the device never waits for the host between them"""
        chunks = np.ascontiguousarray(chunks, dtype=abi.CHUNK_DTYPE)
        self._chk(self.lib.hm_call_chunks_submit(self.h, _p(chunks), len(chunks)))

    def call_chunks_collect(self, cap=None, view=True):
        """-> (records, log[15]) of the submitted call; view=True: a view of one of the two pinned buffers whose copy
        may still be in flight (records_wait)"""
        out = self._out_buffer(int(cap or getattr(self, "_cap", 65536)))
        n = C.c_size_t(0)
        log = np.zeros(abi.CALL_LOG_LEN, np.int64)
        rc = self.lib.hm_call_chunks_collect(self.h, _p(out), out.shape[0], C.byref(n), _p(log))
        if rc == abi.HM_ERR_CAPACITY:
            self._cap = int(n.value) + int(n.value) // 4 + 1024
            out = self._out_buffer(self._cap)
            rc = self.lib.hm_last_records(self.h, _p(out), out.shape[0], C.byref(n))
        self._chk(rc)
        if not view:  # the record copy of a collected call may still be in flight: a private copy needs it finished
            self.records_wait()
        res = out[: n.value]
        return (res if view else res.copy()), log

    def omit_restatements(self, on=True):
        """records of germline restatements (never emitted by the reference) stay on the device; counters unchanged"""
        self._chk(self.lib.hm_set_option(self.h, 1, 1 if on else 0))

    def kernel_timing(self, on=True):
        """CUDA events around the kernels of a call (last_kernel_times); off saves a dozen driver calls per call"""
        self._chk(self.lib.hm_set_option(self.h, 2, 1 if on else 0))

    def records_wait(self):
        self._chk(self.lib.hm_records_wait(self.h))

    def call_batch(self, batch, chunks, cap=None, view=False):
        """upload + call (host buffers in, records out): the end-to-end path"""
        return self._call(self.lib.hm_call_batch, (C.byref(batch.as_struct()),), chunks, cap, view)

    def normcounts_chunks(self, refseq, chunks):
        """callable-base half of `himut normcounts` -> (ccs_tri[33], ref_tri[33], log[14], n_alt_tie)"""
        chunks = np.ascontiguousarray(chunks, dtype=abi.CHUNK_DTYPE)
        if refseq is not getattr(self, "_ref_obj", None):  # upload a contig's reference once
            ref = np.frombuffer(refseq, dtype=np.uint8)
            self._chk(self.lib.hm_set_reference(self.h, _p(ref), ref.size))
            self._ref_obj = refseq
        ref = np.zeros(0, np.uint8)
        ccs = np.zeros(abi.TRI_BINS, np.int64)
        rt = np.zeros(abi.TRI_BINS, np.int64)
        log = np.zeros(abi.NORM_LOG_LEN, np.int64)
        ties = C.c_int64(0)
        self._chk(self.lib.hm_normcounts_chunks(self.h, _p(ref), ref.size, _p(chunks), len(chunks), _p(ccs), _p(rt),
                                                _p(log), C.byref(ties)))
        return ccs, rt, log, int(ties.value)

    def read_stats(self, batch):
        """per-read statistics of the resident batch (must be `batch`) from k_read_scan"""
        n = batch.n_reads
        out = dict(bq_total=np.zeros(n, np.int64), n_match=np.zeros(n, np.int32), n_sub=np.zeros(n, np.int32),
                   ins_len=np.zeros(n, np.int32), del_len=np.zeros(n, np.int32), n_mismatch=np.zeros(n, np.int32))
        self._chk(self.lib.hm_read_stats(self.h, *[_p(out[k]) for k in
                                                   ("bq_total", "n_match", "n_sub", "ins_len", "del_len", "n_mismatch")]))
        return out

    def ref_tricounts(self, refseq):
        """reference trinucleotide counts of one contig -> int64[33] (reflib.get_chrom_tricount)"""
        ref = np.frombuffer(refseq, dtype=np.uint8)
        out = np.zeros(abi.TRI_BINS, np.int64)
        self._chk(self.lib.hm_ref_tricounts(self.h, _p(ref), ref.size, _p(out)))
        self._ref_obj = None
        return out

    def phase_edges_begin(self, hpos, href, band):
        self._edge_hpos = np.ascontiguousarray(hpos, np.int32)
        self._edge_href = np.ascontiguousarray(href, np.uint8)
        self._edge_band = int(band)
        self._chk(self.lib.hm_phase_edges_begin(self.h, _p(self._edge_hpos), _p(self._edge_href), self._edge_hpos.size, self._edge_band))

    def phase_edges_add(self, min_bq, min_mapq, min_tstart=-2**31):
        """accumulate the resident batch; -> 0, or the band a retry needs (nothing usable was added then)"""
        need = C.c_uint32(0)
        rc = self.lib.hm_phase_edges_add(self.h, int(min_bq), int(min_mapq), int(max(min_tstart, -2**31)), C.byref(need))
        if rc == abi.HM_ERR_CAPACITY and need.value != 0xFFFFFFFF:
            return int(need.value)
        self._chk(rc)
        return 0

    def phase_edges_end(self):
        """-> uint32[n_hetsnp, band, 4]"""
        out = np.zeros((self._edge_hpos.size, self._edge_band, 4), np.uint32)
        self._chk(self.lib.hm_phase_edges_end(self.h, _p(out), out.size))
        return out

    def last_norm_exact_sites(self):
        """positions the last normcounts call evaluated exactly (the rest: certified integer pass)"""
        n = C.c_uint64(0)
        self._chk(self.lib.hm_last_norm_exact_sites(self.h, C.byref(n)))
        return int(n.value)

    def qname_seen(self):
        """flags per qname_id of the last call: which query names passed the read gates"""
        n = C.c_size_t(0)
        self.lib.hm_qname_seen(self.h, None, 0, C.byref(n))
        out = np.zeros(n.value, np.uint8)
        self._chk(self.lib.hm_qname_seen(self.h, _p(out), out.size, C.byref(n)))
        return out

    def last_call_path(self):
        """2: the last call_chunks ran the fused device path, 1: the first version, 0: none yet"""
        return int(self.lib.hm_last_call_path(self.h))

    def last_timing(self):
        ms, n = C.c_float(0), C.c_int(0)
        self._chk(self.lib.hm_last_timing(self.h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def last_kernel_times(self):
        cap = 64
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        n = C.c_size_t(0)
        self._chk(self.lib.hm_last_kernel_times(self.h, C.cast(names, C.c_void_p), C.cast(ms, C.c_void_p), cap, C.byref(n)))
        return [(names[i].decode(), float(ms[i])) for i in range(n.value)]
