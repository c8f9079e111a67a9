"""ctypes binding of liburmb.so (include/urmb.h) -- the host-side mirror of the reference's worker loop.

The reference drives the hot path as (map.cpp:11-25, map2.cpp:11-37)::

    State1 UD; UD.SetUFI(UFI); for each read: UD.Search(Query); UD.Output1();
    State2 UD; UD.SetUFI(UFI); for each pair: UD.Search(Query1, Query2);

Here a :class:`Context` plays the role of the per-thread State1/State2 (but for one GPU, and whole batches at a
time), :class:`HostIndex` of ``UFIndex::FromFile``.  There is no CPU mapping path: if ``liburmb.so`` is missing
or no CUDA device is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liburmb.so")

URMB_SLOTS = 8
URMB_SEQ_PAD = 4096
URMB_BLOB_PAD = 16
URMB_E_OVERFLOW = -5

RESULT_DTYPE = np.dtype([
    ("db_pos", "<u4"), ("path_off", "<u4"), ("path_runs", "<u2"), ("score", "<i2"), ("best", "<i2"),
    ("second", "<i2"), ("mapq", "u1"), ("flags", "u1"), ("hit_count", "u1"), ("hsp_count", "u1"),
])
assert RESULT_DTYPE.itemsize == 20


class UrmbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"urmb error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    _fields_ = [("method", C.c_int32), ("pe_method", C.c_int32), ("band_radius", C.c_int32), ("minq", C.c_int32),
                ("want_second", C.c_int32)]


SECOND_DTYPE = np.dtype([("db_pos", "<u4"), ("score", "<i2"), ("flags", "u1"), ("pad", "u1")])


class Batch(C.Structure):
    _fields_ = [("n", C.c_uint32), ("seqs", C.c_void_p), ("offs", C.c_void_p)]


class IndexDesc(C.Structure):
    _fields_ = [("word_length", C.c_uint32), ("max_ix", C.c_uint32), ("seq_data_size", C.c_uint32),
                ("reserved", C.c_uint32), ("slot_count", C.c_uint64), ("d_blob", C.c_void_p), ("d_seq", C.c_void_p)]


class Contig(C.Structure):
    _fields_ = [("length", C.c_uint32), ("offset", C.c_uint32), ("label", C.c_char_p)]


class Timing(C.Structure):
    _fields_ = [("probe_ms", C.c_float), ("search_ms", C.c_float), ("h2d_ms", C.c_float), ("d2h_ms", C.c_float),
                ("rescue_ms", C.c_float), ("kernel_ms", C.c_float * 12), ("kernel_launches", C.c_uint32 * 12)]


KERNEL_CLASSES = ("probe", "pair", "align_a", "rows", "align_c", "finish", "rescue", "rows_long", "rescue_dp",
                  "rescue_legacy", "rescue_last", "k11")


EXPORTS = [
    "urmb_index_load_host", "urmb_index_free_host", "urmb_index_info", "urmb_index_contig", "urmb_ctx_create",
    "urmb_ctx_destroy", "urmb_last_error", "urmb_index_upload", "urmb_index_attach", "urmb_index_broadcast",
    "urmb_index_device_desc", "urmb_map_se", "urmb_map_pe", "urmb_submit", "urmb_wait", "urmb_upload",
    "urmb_launch", "urmb_download", "urmb_timing_last", "urmb_launch_count", "urmb_mark", "urmb_mark_elapsed",
    "urmb_build_index_device", "urmb_build_last_error", "urmb_peak_gather", "urmb_peak_alu",
    "urmb_host_alloc", "urmb_host_free", "urmb_reserve", "urmb_second_hits", "urmb_overflow_count",
    "urmb_unsupported_count", "urmb_first_look_count", "urmb_index_from_fasta", "urmb_index_dropped",
    "urmb_index_fasta_times",
]

_lib = None


def lib():
    """Load liburmb.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C urmap_b200/csrc`")
        L = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        L.urmb_index_load_host.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.urmb_index_free_host.argtypes = [vp]
        L.urmb_index_info.argtypes = [vp, C.POINTER(IndexDesc), C.POINTER(C.c_uint32)]
        L.urmb_index_contig.argtypes = [vp, C.c_uint32, C.POINTER(Contig)]
        L.urmb_ctx_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(vp)]
        L.urmb_ctx_destroy.argtypes = [vp]
        L.urmb_last_error.restype = C.c_char_p
        L.urmb_last_error.argtypes = [vp]
        L.urmb_index_upload.argtypes = [vp, vp]
        L.urmb_index_attach.argtypes = [vp, C.POINTER(IndexDesc)]
        L.urmb_index_broadcast.argtypes = [C.POINTER(vp), C.c_int, vp]
        L.urmb_index_device_desc.argtypes = [vp, C.POINTER(IndexDesc)]
        L.urmb_map_se.argtypes = [vp, C.POINTER(Batch), vp, vp, C.c_uint32, C.POINTER(C.c_uint32)]
        L.urmb_map_pe.argtypes = [vp, C.POINTER(Batch), C.POINTER(Batch), vp, vp, vp, C.c_uint32, C.POINTER(C.c_uint32)]
        L.urmb_submit.argtypes = [vp, C.c_int, C.POINTER(Batch), C.POINTER(Batch)]
        L.urmb_upload.argtypes = [vp, C.c_int, C.POINTER(Batch), C.POINTER(Batch)]
        L.urmb_launch.argtypes = [vp, C.c_int]
        L.urmb_download.argtypes = [vp, C.c_int]
        L.urmb_wait.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_uint32)]
        L.urmb_timing_last.argtypes = [vp, C.c_int, C.POINTER(Timing)]
        L.urmb_launch_count.restype = C.c_uint64
        L.urmb_launch_count.argtypes = [vp]
        L.urmb_mark.argtypes = [vp, C.c_int]
        L.urmb_mark_elapsed.argtypes = [vp, C.POINTER(C.c_float)]
        L.urmb_peak_gather.argtypes = [vp, C.c_uint64, C.c_uint32, C.c_uint64, C.POINTER(C.c_float)]
        L.urmb_peak_alu.argtypes = [C.c_uint64, C.POINTER(C.c_float), C.POINTER(C.c_double)]
        L.urmb_reserve.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32]
        L.urmb_second_hits.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp)]
        L.urmb_overflow_count.argtypes = [vp, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
        L.urmb_first_look_count.argtypes = [vp, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
        L.urmb_unsupported_count.argtypes = [vp, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
        L.urmb_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
        L.urmb_host_free.argtypes = [vp]
        L.urmb_host_free.restype = None
        L.urmb_index_from_fasta.argtypes = [C.POINTER(vp), C.c_int, vp, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64,
                                            C.POINTER(vp)]
        L.urmb_index_dropped.argtypes = [vp, C.c_uint32, C.POINTER(C.c_char_p)]
        L.urmb_index_fasta_times.argtypes = [vp, C.POINTER(C.c_double)]
        for nm in EXPORTS:
            if nm not in ("urmb_last_error", "urmb_launch_count", "urmb_index_free_host", "urmb_ctx_destroy",
                          "urmb_build_last_error", "urmb_host_free"):
                getattr(L, nm).restype = C.c_int
        _lib = L
    return _lib


def _check(rc, ctx=None, allow=()):
    if rc != 0 and rc not in allow:
        msg = lib().urmb_last_error(ctx).decode(errors="replace") if True else ""
        raise UrmbError(rc, msg)
    return rc


def peak_gather(d_ptr: int, n_bytes: int, access_bytes: int = 8, n_access: int = 1 << 28) -> dict:
    """Random sector-aligned reads over a device buffer (current device): the measured denominator of the gather
    roofline (SURVEY.md §8d).  Returns accesses/s and GB/s counted at 32 B (one sector) per access."""
    ms = C.c_float(0)
    _check(lib().urmb_peak_gather(C.c_void_p(d_ptr), n_bytes, access_bytes, n_access, C.byref(ms)))
    s = ms.value / 1e3
    return {"access_bytes": access_bytes, "accesses": n_access, "ms": ms.value, "gaccess_per_s": n_access / s / 1e9,
            "sector_gbs": 32.0 * n_access / s / 1e9}


def peak_alu(ops_per_thread: int = 1 << 22) -> dict:
    """Measured 32-bit integer ALU rate (independent LOP3/IADD chains on every SM): the DP / extension denominator."""
    ms = C.c_float(0)
    ops = C.c_double(0)
    _check(lib().urmb_peak_alu(ops_per_thread, C.byref(ms), C.byref(ops)))
    return {"ms": ms.value, "ops": ops.value, "tops_per_s": ops.value / (ms.value / 1e3) / 1e12}


class HostIndex:
    """Parsed UFI file (UFIndex::FromFile, ufindexio.cpp:60-115); mmap-backed, host only."""

    def __init__(self, path: str):
        self.h = C.c_void_p()
        _check(lib().urmb_index_load_host(os.fsencode(path), C.byref(self.h)))
        d = IndexDesc()
        n = C.c_uint32()
        _check(lib().urmb_index_info(self.h, C.byref(d), C.byref(n)))
        self.word_length, self.max_ix = d.word_length, d.max_ix
        self.seq_data_size, self.slot_count = d.seq_data_size, d.slot_count
        self._blob_ptr, self._seq_ptr = d.d_blob, d.d_seq
        self.contigs = []
        for i in range(n.value):
            c = Contig()
            _check(lib().urmb_index_contig(self.h, i, C.byref(c)))
            self.contigs.append((c.label.decode(), c.length, c.offset))

    def blob(self) -> np.ndarray:
        return np.ctypeslib.as_array(C.cast(self._blob_ptr, C.POINTER(C.c_uint8)), shape=(5 * self.slot_count,))

    def seq(self) -> np.ndarray:
        return np.ctypeslib.as_array(C.cast(self._seq_ptr, C.POINTER(C.c_uint8)), shape=(self.seq_data_size,))

    def close(self):
        if self.h:
            lib().urmb_index_free_host(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _as_batch(seqs: np.ndarray, offs: np.ndarray) -> Batch:
    assert seqs.dtype == np.uint8 and offs.dtype == np.uint32 and seqs.flags.c_contiguous and offs.flags.c_contiguous
    return Batch(len(offs) - 1, seqs.ctypes.data, offs.ctypes.data)


class Context:
    """One GPU's mapping context (replaces the per-thread State1 / State2 of map.cpp:13, map2.cpp:14)."""

    def __init__(self, device: int = 0, method: int = 6, pe_method: int = 4, band_radius: int = -1, minq: int = 10,
                 want_second: bool = False):
        self.c = C.c_void_p()
        p = Params(method, pe_method, band_radius, minq, 1 if want_second else 0)
        _check(lib().urmb_ctx_create(device, C.byref(p), C.byref(self.c)))
        self.device = device
        self._keep = []

    # -- State1::SetUFI ---------------------------------------------------------------
    def set_index(self, hix: HostIndex):
        _check(lib().urmb_index_upload(self.c, hix.h), self.c)

    def attach_index(self, word_length, max_ix, seq_data_size, slot_count, d_blob_ptr, d_seq_ptr, keepalive=()):
        """Use device buffers owned by the caller (e.g. torch tensors that arrived through an NCCL broadcast)."""
        d = IndexDesc(word_length, max_ix, seq_data_size, 0, slot_count, d_blob_ptr, d_seq_ptr)
        _check(lib().urmb_index_attach(self.c, C.byref(d)), self.c)
        self._keep = list(keepalive)

    def index_from_fasta(self, path: str, word_length: int = 24, max_ix: int = 32, slot_count: int | None = None,
                         load_factor: float = 0.6):
        """Build the index of a FASTA file (plain or gzip) on this GPU: the table `-make_ufi` writes for the same options,
        without a file.  slot_count defaults to -make_ufi's: the first table prime >= file size / load_factor.  Returns the
        contig list in the form of HostIndex.contigs; self.dropped lists the labels of the records without sequence."""
        import gzip
        from .index_build import get_prime
        if slot_count is None:
            slot_count = get_prime(int(os.path.getsize(path) / load_factor))
        with open(path, "rb") as f:
            data = f.read()
        if data[:2] == b"\x1f\x8b":
            data = gzip.decompress(data)
        buf = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, dtype=np.uint8)
        ctxs = (C.c_void_p * 1)(self.c)
        h = C.c_void_p()
        _check(lib().urmb_index_from_fasta(ctxs, 1, buf.ctypes.data, len(data), word_length, max_ix, slot_count, C.byref(h)),
               self.c)
        try:
            n = C.c_uint32()
            _check(lib().urmb_index_info(h, None, C.byref(n)))
            contigs = []
            for i in range(n.value):
                c = Contig()
                _check(lib().urmb_index_contig(h, i, C.byref(c)))
                contigs.append((c.label.decode(), c.length, c.offset))
            self.dropped = []
            lab = C.c_char_p()
            while lib().urmb_index_dropped(h, len(self.dropped), C.byref(lab)) == 0:
                self.dropped.append(lab.value.decode())
            t = (C.c_double * 5)()
            _check(lib().urmb_index_fasta_times(h, t))
            self.fasta_times = dict(zip(("upload_s", "parse_s", "build_s", "pack_s", "parse_kernel_s"), list(t)))
        finally:
            lib().urmb_index_free_host(h)
        self._keep = []
        return contigs

    def device_index(self) -> IndexDesc:
        """Description of the index the context maps against (device pointers)."""
        d = IndexDesc()
        _check(lib().urmb_index_device_desc(self.c, C.byref(d)), self.c)
        return d

    # -- State1::Search / State2::Search over a whole batch -----------------------------
    def map_se(self, seqs, offs):
        n = len(offs) - 1
        res = np.zeros(n, dtype=RESULT_DTYPE)
        cap = 32 * n + 4096
        runs = np.zeros(cap, dtype=np.uint16)
        used = C.c_uint32()
        b = _as_batch(seqs, offs)
        rc = lib().urmb_map_se(self.c, C.byref(b), res.ctypes.data, runs.ctypes.data, cap, C.byref(used))
        _check(rc, self.c)
        return res, runs[:used.value]

    def map_pe(self, seqs1, offs1, seqs2, offs2):
        n = len(offs1) - 1
        r1 = np.zeros(n, dtype=RESULT_DTYPE)
        r2 = np.zeros(n, dtype=RESULT_DTYPE)
        cap = 64 * n + 4096
        runs = np.zeros(cap, dtype=np.uint16)
        used = C.c_uint32()
        b1, b2 = _as_batch(seqs1, offs1), _as_batch(seqs2, offs2)
        rc = lib().urmb_map_pe(self.c, C.byref(b1), C.byref(b2), r1.ctypes.data, r2.ctypes.data, runs.ctypes.data, cap,
                               C.byref(used))
        _check(rc, self.c)
        return r1, r2, runs[:used.value]

    # -- pipelined interface -----------------------------------------------------------------
    def upload(self, slot, seqs1, offs1, seqs2=None, offs2=None):
        b1 = _as_batch(seqs1, offs1)
        b2 = _as_batch(seqs2, offs2) if seqs2 is not None else None
        _check(lib().urmb_upload(self.c, slot, C.byref(b1), C.byref(b2) if b2 is not None else None), self.c)

    def submit(self, slot, seqs1, offs1, seqs2=None, offs2=None):
        b1 = _as_batch(seqs1, offs1)
        b2 = _as_batch(seqs2, offs2) if seqs2 is not None else None
        _check(lib().urmb_submit(self.c, slot, C.byref(b1), C.byref(b2) if b2 is not None else None), self.c)

    def launch(self, slot):
        _check(lib().urmb_launch(self.c, slot), self.c)

    def download(self, slot):
        _check(lib().urmb_download(self.c, slot), self.c)

    def wait(self, slot, n, paired):
        """Returns (res1, res2|None, runs) as numpy views of the slot's pinned buffers (valid until restaged)."""
        p1, p2, pr = C.c_void_p(), C.c_void_p(), C.c_void_p()
        used = C.c_uint32()
        _check(lib().urmb_wait(self.c, slot, C.byref(p1), C.byref(p2), C.byref(pr), C.byref(used)), self.c)

        def view(p, count, dt):
            if not p or count == 0:
                return np.zeros(0, dtype=dt)
            buf = (C.c_uint8 * (count * np.dtype(dt).itemsize)).from_address(p)
            return np.frombuffer(buf, dtype=dt, count=count)

        r1 = view(p1.value, n, RESULT_DTYPE)
        r2 = view(p2.value, n, RESULT_DTYPE) if paired else None
        return r1, r2, view(pr.value, used.value, np.uint16)

    def second_hits(self, slot, n):
        """State2's second pair per mate (contexts created with want_second; after wait() on a paired-end slot)."""
        p1, p2 = C.c_void_p(), C.c_void_p()
        _check(lib().urmb_second_hits(self.c, slot, C.byref(p1), C.byref(p2)), self.c)
        mk = lambda p: np.frombuffer((C.c_uint8 * (n * SECOND_DTYPE.itemsize)).from_address(p.value), dtype=SECOND_DTYPE, count=n)
        return mk(p1), mk(p2)

    def timing(self, slot):
        t = Timing()
        _check(lib().urmb_timing_last(self.c, slot, C.byref(t)), self.c)
        return {"probe_ms": t.probe_ms, "search_ms": t.search_ms, "h2d_ms": t.h2d_ms, "d2h_ms": t.d2h_ms,
                "rescue_ms": t.rescue_ms,
                "kernel_ms": {k: float(t.kernel_ms[i]) for i, k in enumerate(KERNEL_CLASSES)},
                "kernel_launches": {k: int(t.kernel_launches[i]) for i, k in enumerate(KERNEL_CLASSES)}}

    def mark(self, which):
        """Context-wide time mark (0 = start, 1 = end) after all work submitted so far."""
        _check(lib().urmb_mark(self.c, which), self.c)

    def mark_elapsed(self):
        """Device milliseconds between mark 0 and mark 1 (synchronises)."""
        ms = C.c_float()
        _check(lib().urmb_mark_elapsed(self.c, C.byref(ms)), self.c)
        return float(ms.value)

    def overflow_count(self, slot=0):
        """(reads of the slot's last batch, reads over all batches) that exceeded a per-read capacity (flags bit 7)."""
        last, total = C.c_uint32(), C.c_uint64()
        _check(lib().urmb_overflow_count(self.c, slot, C.byref(last), C.byref(total)), self.c)
        return int(last.value), int(total.value)

    def unsupported_count(self, slot=0):
        """(reads of the slot's last batch, reads over all batches) not searched: longer than URMB_MAX_READ_LEN (flags bit 6)."""
        last, total = C.c_uint32(), C.c_uint64()
        _check(lib().urmb_unsupported_count(self.c, slot, C.byref(last), C.byref(total)), self.c)
        return int(last.value), int(total.value)

    def first_look_count(self, slot=0):
        """(pairs of the slot's last batch, pairs over all batches) finished by the probe kernel's first look."""
        last, total = C.c_uint32(), C.c_uint64()
        _check(lib().urmb_first_look_count(self.c, slot, C.byref(last), C.byref(total)), self.c)
        return int(last.value), int(total.value)

    def launch_count(self):
        return int(lib().urmb_launch_count(self.c))

    def close(self):
        if self.c:
            lib().urmb_ctx_destroy(self.c)
            self.c = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
