"""ctypes mirror of include/himut_b200.h (structs, constants) and the packed read batch.

The layouts here must match the header byte for byte; tests/test_abi.py checks the sizes
against the built library (hm_abi_sizeof).
"""
import ctypes as C

import numpy as np

HM_OK, HM_ERR_ARG, HM_ERR_CUDA, HM_ERR_CAPACITY, HM_ERR_BQ_ZERO, HM_ERR_NO_DEVICE, HM_ERR_STATE = range(7)
HM_DECODE_SEQ = 1  # hm_decode_bam_begin_opts: decode the 2-bit base stream too
HM_DECODE_REF = 2  # hm_decode_bam_begin_opts: records with neither cs:Z nor MD:Z decode against the resident reference

OP_MATCH, OP_SUB, OP_INS, OP_DEL = 0, 1, 2, 3
BASE_N = 4
READ_SECONDARY = 1

# reference util.base2idx (src/himut/util.py:14-20)
BASE2CODE = {"A": 0, "T": 1, "G": 2, "C": 3}
CODE2BASE = "ATGC"

CALL_LOG_LEN = 15
NORM_LOG_LEN = 14
TRI_BINS = 33

ST_PASS, ST_GERM_HET, ST_GERM_HETALT, ST_GERM_HOMALT, ST_GERM_HOMREF, ST_HET_SITE, \
    ST_HETALT_SITE, ST_HOMALT_SITE, ST_INDEL_SITE, ST_LOW_GQ, ST_LOW_BQ, ST_PON, ST_COMSNP, \
    ST_LOW_DEPTH, ST_HIGH_DEPTH, ST_UNPHASED = range(16)
# status strings of the emitted rows (reference caller.py:349-621); germline restatements
# are counted but never emitted
STATUS_NAME = {
    ST_PASS: "PASS", ST_HET_SITE: "HetSite", ST_HETALT_SITE: "HetAltSite",
    ST_HOMALT_SITE: "HomAltSite", ST_INDEL_SITE: "IndelSite", ST_LOW_GQ: "LowGQ",
    ST_LOW_BQ: "LowBQ", ST_PON: "PanelOfNormal", ST_COMSNP: "ComSnp",
    ST_LOW_DEPTH: "LowDepth", ST_HIGH_DEPTH: "HighDepth", ST_UNPHASED: "Unphased",
}
SITE_PL_TIE = 1


class hm_read_batch(C.Structure):
    _fields_ = [
        ("n_reads", C.c_uint64),
        ("tstart", C.c_void_p), ("tend", C.c_void_p), ("qstart", C.c_void_p), ("qlen", C.c_void_p),
        ("mapq", C.c_void_p), ("flags", C.c_void_p), ("qname_id", C.c_void_p),
        ("seq_off", C.c_void_p), ("bq_off", C.c_void_p), ("op_off", C.c_void_p), ("n_ops", C.c_void_p),
        ("seq", C.c_void_p), ("seq_bytes", C.c_uint64),
        ("bq", C.c_void_p), ("bq_bytes", C.c_uint64),
        ("ops", C.c_void_p), ("n_ops_total", C.c_uint64),
    ]


class hm_bq_compact(C.Structure):
    _fields_ = [("mask", C.c_void_p), ("mask_bytes", C.c_uint64), ("exc", C.c_void_p), ("exc_bytes", C.c_uint64),
                ("exc_off", C.c_void_p), ("modal", C.c_uint8), ("reserved", C.c_uint8 * 7)]


class BqCompact:
    """numpy-backed hm_bq_compact: the quality stream of a ReadBatch as modal-value bitmap + exceptions"""

    def __init__(self, mask, exc, exc_off, modal, n_exc):
        self.mask, self.exc, self.exc_off, self.modal, self.n_exc = mask, exc, exc_off, modal, n_exc
        s = hm_bq_compact()
        s.mask, s.mask_bytes = _ptr(mask), mask.size
        s.exc, s.exc_bytes = _ptr(exc), n_exc
        s.exc_off, s.modal = _ptr(exc_off), modal
        self.struct = s

    def nbytes(self):
        return self.mask.nbytes + self.n_exc + self.exc_off.nbytes


class hm_bgzf_plan(C.Structure):
    """a BAM region planned for the device decoder (include/himut_b200.h)"""
    _fields_ = [("comp", C.c_void_p), ("comp_bytes", C.c_uint64), ("n_blocks", C.c_uint64),
                ("blk_coff", C.c_void_p), ("blk_csize", C.c_void_p), ("blk_isize", C.c_void_p), ("blk_uoff", C.c_void_p),
                ("blk_crc", C.c_void_p), ("entry", C.c_void_p), ("n_entry", C.c_uint64), ("walk_end", C.c_uint64),
                ("path", C.c_char_p)]


class hm_chunk(C.Structure):
    _fields_ = [("start", C.c_int32), ("end", C.c_int32), ("read_lo", C.c_uint32),
                ("read_hi", C.c_uint32), ("phase_set", C.c_int32), ("reserved", C.c_int32)]


class hm_params(C.Structure):
    _fields_ = [
        ("min_qv", C.c_int32), ("min_mapq", C.c_int32),
        ("qlen_lower_limit", C.c_int32), ("qlen_upper_limit", C.c_int32),
        ("min_gq", C.c_int32), ("min_bq", C.c_int32),
        ("max_mismatch_count", C.c_int32), ("mismatch_window", C.c_int32),
        ("min_ref_count", C.c_int32), ("min_alt_count", C.c_int32), ("min_hap_count", C.c_int32),
        ("phase", C.c_int32), ("non_human_sample", C.c_int32), ("create_panel_of_normals", C.c_int32),
        ("min_sequence_identity", C.c_double), ("min_trim", C.c_double), ("md_threshold", C.c_double),
        ("log10_prior", C.c_double * 4),
        ("lut_hom", C.c_double * 256), ("lut_het", C.c_double * 256), ("lut_err", C.c_double * 256),
    ]


class hm_site_record(C.Structure):
    _fields_ = [
        ("tpos", C.c_int32),
        ("ref", C.c_uint8), ("alt", C.c_uint8), ("status", C.c_uint8), ("flags", C.c_uint8),
        ("chunk", C.c_int32), ("gq", C.c_int32),
        ("germ_gt", C.c_uint8 * 2), ("germ_state", C.c_uint8), ("pad0", C.c_uint8),
        ("counts", C.c_int32 * 6), ("bq_sum", C.c_int32 * 4),
        ("hap_count", C.c_int32 * 2), ("som_hap_mask", C.c_int32), ("phase_set", C.c_int32),
    ]


SITE_DTYPE = np.dtype([
    ("tpos", "<i4"), ("ref", "u1"), ("alt", "u1"), ("status", "u1"), ("flags", "u1"),
    ("chunk", "<i4"), ("gq", "<i4"), ("germ_gt", "u1", (2,)), ("germ_state", "u1"), ("pad0", "u1"),
    ("counts", "<i4", (6,)), ("bq_sum", "<i4", (4,)), ("hap_count", "<i4", (2,)),
    ("som_hap_mask", "<i4"), ("phase_set", "<i4"),
])
assert SITE_DTYPE.itemsize == C.sizeof(hm_site_record)

class hm_callable_run(C.Structure):
    _fields_ = [("chunk", C.c_uint32), ("start", C.c_int32), ("end", C.c_int32), ("value", C.c_uint32)]


# runs of the callable-base track (hm_last_callable_runs): positions [start, end) of chunk `chunk`, each counted with
# `value` callable read bases
RUN_DTYPE = np.dtype([("chunk", "<u4"), ("start", "<i4"), ("end", "<i4"), ("value", "<u4")])
assert RUN_DTYPE.itemsize == C.sizeof(hm_callable_run)

CHUNK_DTYPE = np.dtype([("start", "<i4"), ("end", "<i4"), ("read_lo", "<u4"), ("read_hi", "<u4"),
                        ("phase_set", "<i4"), ("reserved", "<i4")])
assert CHUNK_DTYPE.itemsize == C.sizeof(hm_chunk)


def make_op(kind, value):
    return (kind | (value << 2)) & 0xFFFFFFFF


def make_sub(ref_code, alt_code):
    return make_op(OP_SUB, ref_code | (alt_code << 3))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class ReadBatch:
    """Packed structure-of-arrays read batch of one contig (hm_read_batch), numpy backed.

    Replaces the per-record attribute pulls of the reference's bamlib.BAM.__init__
    (src/himut/bamlib.py:15-32): tstart/tend/qstart/qlen/mapq/flags/qname_id per read,
    2-bit bases, one BQ byte per base and the cs op stream.
    """

    _FIELDS = [("tstart", np.int32), ("tend", np.int32), ("qstart", np.int32), ("qlen", np.int32),
               ("mapq", np.uint8), ("flags", np.uint8), ("qname_id", np.uint32),
               ("seq_off", np.uint64), ("bq_off", np.uint64), ("op_off", np.uint64),
               ("n_ops", np.uint32), ("seq", np.uint8), ("bq", np.uint8), ("ops", np.uint32)]

    def __init__(self, **arrays):
        for name, dt in self._FIELDS:
            a = np.ascontiguousarray(arrays[name], dtype=dt)
            setattr(self, name, a)
        self.n_reads = int(self.tstart.shape[0])
        self.keepalive = arrays.get("keepalive")
        if self.seq.size % 16 or self.bq.size % 16:
            raise ValueError("seq / bq buffers must be padded to a multiple of 16 bytes")
        self._struct = None

    @property
    def aligned_bases(self):
        """sum of query_alignment_end - query_alignment_start (the bench metric's unit)"""
        kind = self.ops & 3
        val = (self.ops >> 2).astype(np.int64)
        qspan = np.where(kind == OP_MATCH, val, 0) + np.where(kind == OP_SUB, 1, 0) + np.where(kind == OP_INS, val, 0)
        return int(qspan.sum())

    def as_struct(self):
        if self._struct is None:
            s = hm_read_batch()
            s.n_reads = self.n_reads
            for name, _ in self._FIELDS:
                setattr(s, name, _ptr(getattr(self, name)))
            if self.n_reads and not self.seq.size:  # no base stream (see without_seq)
                s.seq, s.seq_off = None, None
            s.seq_bytes = self.seq.size
            s.bq_bytes = self.bq.size
            if not self.bq.size and getattr(self, "bq_bytes_expanded", 0):
                # the qualities travel in compact form (BqCompact): no one-byte-per-base stream on the host;
                # bq_off / bq_bytes describe the layout the device expands to
                s.bq, s.bq_bytes = None, int(self.bq_bytes_expanded)
            s.n_ops_total = self.ops.size
            self._struct = s
        return self._struct

    def nbytes(self):
        return sum(getattr(self, n).nbytes for n, _ in self._FIELDS)

    def without_seq(self):
        """the same batch (arrays shared) without its base stream: hm_read_batch.seq = NULL.  `call` and the phase
        edges take the bases of match runs from the site's reference allele then — which is what a cs match says
        (src/himut/cslib.py:22-29) — so a worker need neither unpack nor upload them."""
        kw = {name: getattr(self, name) for name, _ in self._FIELDS}
        kw["seq"], kw["seq_off"] = np.zeros(0, np.uint8), np.zeros(0, np.uint64)
        return ReadBatch(keepalive=(self, self.keepalive), **kw)

    # ---- chunk -> read index range --------------------------------------------------
    def chunk_table(self, chunkloci, phase_sets=None):
        """hm_chunk[] for a list of (start, end) fetch windows.

        read_hi = first read with tstart >= end; read_lo = first read whose running maximum
        of tend exceeds start — the smallest file-order range holding every record
        pysam's fetch(chrom, start, end) returns (src/himut/caller.py:299).
        """
        out = np.zeros(len(chunkloci), dtype=CHUNK_DTYPE)
        if self.n_reads:
            pmax = np.maximum.accumulate(self.tend)
        for i, (s, e) in enumerate(chunkloci):
            out["start"][i], out["end"][i] = s, e
            if self.n_reads:
                out["read_hi"][i] = np.searchsorted(self.tstart, e, side="left")
                out["read_lo"][i] = min(np.searchsorted(pmax, s, side="right"), out["read_hi"][i])
            out["phase_set"][i] = -1 if phase_sets is None else phase_sets[i]
        return out

    def select(self, idx):
        """sub-batch of the given read indices (repacks seq / bq / ops)"""
        idx = np.asarray(idx, dtype=np.int64)
        seq_parts, bq_parts, op_parts = [], [], []
        seq_off, bq_off, op_off = [], [], []
        so = bo = oo = 0
        for r in idx:
            ql = int(self.qlen[r])
            sb = (ql + 3) // 4
            s0, b0, o0 = int(self.seq_off[r]), int(self.bq_off[r]), int(self.op_off[r])
            seq_parts.append(np.pad(self.seq[s0:s0 + sb], (0, (-sb) % 16)))
            bq_parts.append(np.pad(self.bq[b0:b0 + ql], (0, (-ql) % 16)))
            op_parts.append(self.ops[o0:o0 + int(self.n_ops[r])])
            seq_off.append(so); bq_off.append(bo); op_off.append(oo)
            so += seq_parts[-1].size; bo += bq_parts[-1].size; oo += op_parts[-1].size
        cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
        return ReadBatch(
            tstart=self.tstart[idx], tend=self.tend[idx], qstart=self.qstart[idx], qlen=self.qlen[idx],
            mapq=self.mapq[idx], flags=self.flags[idx], qname_id=self.qname_id[idx],
            seq_off=np.array(seq_off, np.uint64), bq_off=np.array(bq_off, np.uint64),
            op_off=np.array(op_off, np.uint64), n_ops=self.n_ops[idx],
            seq=cat(seq_parts, np.uint8), bq=cat(bq_parts, np.uint8), ops=cat(op_parts, np.uint32))
