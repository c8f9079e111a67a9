"""ctypes wrapper of the FASTA parse kernels under the debugging emulator (tests/emu/libemu_fasta.so). Test infrastructure
only."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(HERE, "libemu_fasta.so")
        src = [os.path.join(HERE, f) for f in ("emu_fasta.cpp", "emu.cpp", "cuda_runtime.h")] + [
            os.path.join(HERE, "../../urmap_b200/csrc", f) for f in ("urmb_fasta.cu", "urmb_build.cu", "urmb_kernels.cu", "urmb_internal.h")] + [
            os.path.join(HERE, "../kunit/kunit_cases.cuh")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
            subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-I.", "-o", so, "emu_fasta.cpp",
                                   "-Wno-unused-function"], cwd=HERE)
        _lib = C.CDLL(so)
    return _lib


def emu_parse_fasta(data: bytes):
    """The FASTA parse kernels (urmb_fasta.cu) under emulation.  Returns (rc, seq, records, dropped, error): seq = SeqData
    with the URMB_SEQ_PAD zero bytes cut off, records = [(label bytes, length, offset)], dropped = [label bytes]."""
    L = lib()
    L.emu_parse_fasta.restype = C.c_int
    L.emu_fasta_seq.restype = C.c_uint64
    L.emu_fasta_n_records.restype = C.c_uint32
    L.emu_fasta_n_dropped.restype = C.c_uint32
    L.emu_fasta_record.restype = C.c_void_p
    L.emu_fasta_dropped.restype = C.c_void_p
    L.emu_fasta_error.restype = C.c_char_p
    buf = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
    rc = L.emu_parse_fasta(buf.ctypes.data_as(C.c_void_p), C.c_uint64(len(data)))
    if rc != 0:
        return rc, b"", [], [], L.emu_fasta_error().decode(errors="replace")
    p = C.c_void_p()
    n = L.emu_fasta_seq(C.byref(p))
    seq = C.string_at(p.value, n - 4096) if n > 4096 else b""
    assert C.string_at(p.value + n - 4096, 4096) == bytes(4096)
    recs, dropped = [], []
    ll, ln, off = C.c_uint32(), C.c_uint32(), C.c_uint32()
    for i in range(L.emu_fasta_n_records()):
        q = L.emu_fasta_record(i, C.byref(ll), C.byref(ln), C.byref(off))
        recs.append((C.string_at(q, ll.value) if ll.value else b"", ln.value, off.value))
    for i in range(L.emu_fasta_n_dropped()):
        q = L.emu_fasta_dropped(i, C.byref(ll))
        dropped.append(C.string_at(q, ll.value) if ll.value else b"")
    return 0, seq, recs, dropped, ""
