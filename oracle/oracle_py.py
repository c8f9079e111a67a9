"""ctypes binding of oracle/liburmap_oracle.so -- TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs.
The product package (urmap_b200/) must never import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liburmap_oracle.so")
REF_BIN = os.path.join(HERE, "_ref", "urmap")

RESULT_DTYPE = np.dtype([
    ("db_pos", "<u4"), ("path_off", "<u4"), ("path_runs", "<u2"), ("score", "<i2"), ("best", "<i2"),
    ("second", "<i2"), ("mapq", "u1"), ("flags", "u1"), ("hit_count", "u1"), ("hsp_count", "u1"),
])
assert RESULT_DTYPE.itemsize == 20

STATS_FIELDS = ["reads", "probes", "row_calls", "row_hops", "extend_calls", "compare_bytes", "slot_hashes",
                "dp_calls", "dp_cells", "scan_calls", "tb_poison_reads", "compare_bytes_rows", "row_hops_long",
                "compare_bytes_rows_long", "dp_cells_scan"]


class Params(C.Structure):
    _fields_ = [("method", C.c_int32), ("pe_method", C.c_int32), ("band_radius", C.c_int32), ("minq", C.c_int32)]


def build(ref: bool = True, quiet: bool = True):
    """Compile the restatement and (when /root/reference exists) the reference binary."""
    out = subprocess.DEVNULL if quiet else None
    subprocess.check_call(["make", "-C", HERE, "port"], stdout=out, stderr=out)
    if ref and os.path.isdir("/root/reference/src") and not os.path.exists(REF_BIN):
        subprocess.check_call(["make", "-C", HERE, "-j8", "ref"], stdout=out, stderr=out)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build(ref=False)
        L = C.CDLL(LIB_PATH)
        L.uo_index_open.restype = C.c_void_p
        L.uo_index_open.argtypes = [C.c_char_p]
        L.uo_index_close.argtypes = [C.c_void_p]
        for nm, rt in (("uo_index_slot_count", C.c_uint64), ("uo_index_seq_size", C.c_uint32),
                       ("uo_index_word_length", C.c_uint32), ("uo_index_max_ix", C.c_uint32),
                       ("uo_index_contig_count", C.c_uint32), ("uo_index_blob", C.c_void_p),
                       ("uo_index_seq", C.c_void_p)):
            getattr(L, nm).restype = rt
            getattr(L, nm).argtypes = [C.c_void_p]
        vp = C.c_void_p
        L.uo_map_se.restype = C.c_int
        L.uo_map_se.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_uint32, vp, vp, C.c_uint32, vp, vp, C.c_int]
        L.uo_map_pe.restype = C.c_int
        L.uo_map_pe.argtypes = [vp, C.POINTER(Params), vp, vp, vp, vp, C.c_uint32, vp, vp, vp, C.c_uint32, vp, vp,
                                C.c_int]
        L.uo_sam_header.restype = vp
        L.uo_sam_header.argtypes = [vp, C.c_char_p, C.c_char_p, vp]
        L.uo_sam_se.restype = vp
        L.uo_sam_se.argtypes = [vp, C.c_uint32] + [vp] * 7 + [vp]
        L.uo_sam_pe.restype = vp
        L.uo_sam_pe.argtypes = [vp, C.c_uint32] + [vp] * 13 + [vp]
        L.uo_free.argtypes = [vp]
        L.uo_slots.argtypes = [vp, vp, C.c_uint32, vp, vp]
        L.uo_revcomp.argtypes = [vp, C.c_uint32, vp]
        L.uo_viterbi.restype = C.c_float
        L.uo_viterbi.argtypes = [C.POINTER(Params), vp, C.c_uint32, vp, C.c_uint32, C.c_int, C.c_int, C.c_char_p]
        L.uo_viterbi_ex.restype = C.c_float
        L.uo_viterbi_ex.argtypes = [C.POINTER(Params), vp, C.c_uint32, vp, C.c_uint32, C.c_int, C.c_int, C.c_char_p, vp]
        L.uo_path_to_cigar.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p]
        L.uo_index_functional_diff.restype = C.c_uint64
        L.uo_index_functional_diff.argtypes = [vp, vp, vp]
        L.uo_get_prime.restype = C.c_uint64
        L.uo_get_prime.argtypes = [C.c_uint64]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class ReadBatch:
    """Concatenated reads: seqs/quals/labels uint8 arrays + uint32 offsets."""

    def __init__(self, seqs, offs, quals=None, labels=None, label_offs=None):
        self.seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        self.offs = np.ascontiguousarray(offs, dtype=np.uint32)
        self.quals = None if quals is None else np.ascontiguousarray(quals, dtype=np.uint8)
        self.n = len(self.offs) - 1
        if labels is None:
            labs = [b"r%d" % i for i in range(self.n)]
            labels = np.frombuffer(b"".join(labs), dtype=np.uint8)
            label_offs = np.concatenate([[0], np.cumsum([len(x) for x in labs])])
        self.labels = np.ascontiguousarray(labels, dtype=np.uint8)
        self.label_offs = np.ascontiguousarray(label_offs, dtype=np.uint32)

    @staticmethod
    def from_arrays(reads2d, names=None, qual=b"I"):
        n, L = reads2d.shape
        offs = np.arange(n + 1, dtype=np.uint32) * L
        quals = np.full(n * L, qual[0], dtype=np.uint8)
        if names is None:
            return ReadBatch(reads2d.reshape(-1), offs, quals)
        labels = np.frombuffer(b"".join(names), dtype=np.uint8)
        lo = np.concatenate([[0], np.cumsum([len(x) for x in names])])
        return ReadBatch(reads2d.reshape(-1), offs, quals, labels, lo)

    @staticmethod
    def from_fastq(path):
        """Minimal FASTQ reader with the reference's conventions (fastqseqsource.cpp:9-116):
        label = whole header line after '@', CR stripped."""
        data = open(path, "rb").read().replace(b"\r", b"")
        lines = data.split(b"\n")
        while lines and lines[-1] == b"":
            lines.pop()
        assert len(lines) % 4 == 0, "truncated FASTQ"
        labs = [l[1:] for l in lines[0::4]]
        seqs = lines[1::4]
        quals = lines[3::4]
        offs = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.uint32)
        lo = np.concatenate([[0], np.cumsum([len(s) for s in labs])]).astype(np.uint32)
        return ReadBatch(np.frombuffer(b"".join(seqs), dtype=np.uint8), offs,
                         np.frombuffer(b"".join(quals), dtype=np.uint8),
                         np.frombuffer(b"".join(labs), dtype=np.uint8), lo)


class Index:
    def __init__(self, path):
        self.h = lib().uo_index_open(path.encode())
        if not self.h:
            raise IOError(f"cannot open UFI {path}")
        self.path = path
        L = lib()
        self.slot_count = L.uo_index_slot_count(self.h)
        self.seq_size = L.uo_index_seq_size(self.h)
        self.word_length = L.uo_index_word_length(self.h)
        self.max_ix = L.uo_index_max_ix(self.h)
        self.contig_count = L.uo_index_contig_count(self.h)

    def close(self):
        if self.h:
            lib().uo_index_close(self.h)
            self.h = None

    def blob(self):
        p = lib().uo_index_blob(self.h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(5 * self.slot_count,))

    def seq(self):
        p = lib().uo_index_seq(self.h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(self.seq_size,))


def _stats_dict(arr):
    return dict(zip(STATS_FIELDS, (int(x) for x in arr)))


def map_se(ix: Index, batch: ReadBatch, method=6, band_radius=-1, threads=1, want_stats=False):
    p = Params(method, 4, band_radius, 10)
    res = np.zeros(batch.n, dtype=RESULT_DTYPE)
    cap = max(1024, 64 * batch.n)
    runs = np.zeros(cap, dtype=np.uint16)
    used = C.c_uint32(0)
    st = np.zeros(len(STATS_FIELDS), dtype=np.uint64)
    rc = lib().uo_map_se(ix.h, C.byref(p), _p(batch.seqs), _p(batch.offs), batch.n, _p(res), _p(runs), cap,
                         C.addressof(used), _p(st) if want_stats else None, threads)
    assert rc == 0, rc
    out = (res, runs[:used.value].copy())
    return out + (_stats_dict(st),) if want_stats else out


def map_pe(ix: Index, b1: ReadBatch, b2: ReadBatch, pe_method=4, band_radius=-1, threads=1, want_stats=False):
    assert b1.n == b2.n
    if pe_method == 5 and band_radius < 0:
        band_radius = 4  # map2.cpp:17-21
    p = Params(6, pe_method, band_radius, 10)
    r1 = np.zeros(b1.n, dtype=RESULT_DTYPE)
    r2 = np.zeros(b1.n, dtype=RESULT_DTYPE)
    cap = max(1024, 128 * b1.n)
    runs = np.zeros(cap, dtype=np.uint16)
    used = C.c_uint32(0)
    st = np.zeros(len(STATS_FIELDS), dtype=np.uint64)
    rc = lib().uo_map_pe(ix.h, C.byref(p), _p(b1.seqs), _p(b1.offs), _p(b2.seqs), _p(b2.offs), b1.n, _p(r1), _p(r2),
                         _p(runs), cap, C.addressof(used), _p(st) if want_stats else None, threads)
    assert rc == 0, rc
    out = (r1, r2, runs[:used.value].copy())
    return out + (_stats_dict(st),) if want_stats else out


def _take(ptr, n):
    s = C.string_at(ptr, n)
    lib().uo_free(ptr)
    return s


def sam_header(ix: Index, version="1.0.1441", cmdline=""):
    n = C.c_size_t(0)
    p = lib().uo_sam_header(ix.h, version.encode(), cmdline.encode(), C.addressof(n))
    return _take(p, n.value)


def sam_se(ix: Index, b: ReadBatch, res, runs):
    n = C.c_size_t(0)
    runs = np.ascontiguousarray(runs if len(runs) else np.zeros(1, np.uint16))
    p = lib().uo_sam_se(ix.h, b.n, _p(b.seqs), _p(b.offs), _p(b.quals), _p(b.labels), _p(b.label_offs), _p(res),
                        _p(runs), C.addressof(n))
    return _take(p, n.value)


def sam_pe(ix: Index, b1: ReadBatch, b2: ReadBatch, r1, r2, runs):
    n = C.c_size_t(0)
    runs = np.ascontiguousarray(runs if len(runs) else np.zeros(1, np.uint16))
    p = lib().uo_sam_pe(ix.h, b1.n, _p(b1.seqs), _p(b1.offs), _p(b1.quals), _p(b1.labels), _p(b1.label_offs),
                        _p(b2.seqs), _p(b2.offs), _p(b2.quals), _p(b2.labels), _p(b2.label_offs), _p(r1), _p(r2),
                        _p(runs), C.addressof(n))
    return _take(p, n.value)


def slots(ix: Index, seq: bytes):
    a = np.frombuffer(seq, dtype=np.uint8)
    n = max(0, len(a) - ix.word_length + 1)
    plus = np.zeros(max(n, 1), dtype=np.uint64)
    minus = np.zeros(max(n, 1), dtype=np.uint64)
    lib().uo_slots(ix.h, _p(a), len(a), _p(plus), _p(minus))
    return plus[:n], minus[:n]


def viterbi(A: bytes, B: bytes, left: bool, right: bool, method=6, band_radius=-1):
    p = Params(method, 4, band_radius, 10)
    buf = C.create_string_buffer(len(A) + len(B) + 4)
    a = np.frombuffer(A, dtype=np.uint8)
    b = np.frombuffer(B, dtype=np.uint8)
    sc = lib().uo_viterbi(C.byref(p), _p(a) if len(a) else None, len(a), _p(b) if len(b) else None, len(b),
                          int(left), int(right), buf)
    return float(sc), buf.value.decode()


def viterbi_ex(A: bytes, B: bytes, left: bool, right: bool, method=6, band_radius=-1):
    """viterbi() plus the number of traceback reads of cells the call never wrote (the result is undefined when it is
    not zero): (score, path, poison reads)."""
    p = Params(method, 4, band_radius, 10)
    buf = C.create_string_buffer(len(A) + len(B) + 4)
    a = np.frombuffer(A, dtype=np.uint8)
    b = np.frombuffer(B, dtype=np.uint8)
    n = C.c_uint64(0)
    sc = lib().uo_viterbi_ex(C.byref(p), _p(a) if len(a) else None, len(a), _p(b) if len(b) else None, len(b),
                             int(left), int(right), buf, C.addressof(n))
    return float(sc), buf.value.decode(), int(n.value)


def path_to_cigar(path: str, ql: int):
    buf = C.create_string_buffer(12 * len(path) + 32)
    lib().uo_path_to_cigar(path.encode(), ql, buf)
    return buf.value.decode()


def index_functional_diff(a: Index, b: Index):
    first = C.c_uint64(0)
    n = lib().uo_index_functional_diff(a.h, b.h, C.addressof(first))
    return int(n), int(first.value)


def get_prime(n: int) -> int:
    return int(lib().uo_get_prime(n))


def run_reference(args, quiet=True):
    """Run the unmodified reference binary (oracle/_ref/urmap)."""
    if not os.path.exists(REF_BIN):
        raise FileNotFoundError(REF_BIN)
    r = subprocess.run([REF_BIN] + list(args), capture_output=True)
    if r.returncode != 0:
        raise RuntimeError(f"reference failed rc={r.returncode}: {r.stderr[-2000:].decode(errors='replace')}")
    return r
