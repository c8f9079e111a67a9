"""ctypes wrapper of the debugging emulator (tests/emu/libemu.so). Test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


class Params(C.Structure):
    _fields_ = [("method", C.c_int32), ("pe_method", C.c_int32), ("band_radius", C.c_int32), ("minq", C.c_int32),
                ("want_second", C.c_int32)]


SECOND_DTYPE = np.dtype([("db_pos", "<u4"), ("score", "<i2"), ("flags", "u1"), ("pad", "u1")])


_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(HERE, "libemu.so")
        src = [os.path.join(HERE, "emu.cpp"), os.path.join(HERE, "cuda_runtime.h"),
               os.path.join(HERE, "../../urmap_b200/csrc/urmb_kernels.cu"),
               os.path.join(HERE, "../../urmap_b200/csrc/urmb_internal.h"), os.path.join(HERE, "../kunit/kunit_cases.cuh")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
            subprocess.check_call([os.path.join(HERE, "build.sh")])
        _lib = C.CDLL(so)
        _lib.emu_map.restype = C.c_int
    return _lib


def emu_map(oix, res_dtype, seqs, offs, n_units, paired, method=6, pe_method=4, band_radius=-1, second=None):
    """oix: oracle_py.Index (only used as a UFI parser that exposes blob/seq pointers)."""
    L = lib()
    seq = np.zeros(oix.seq_size + 4096, dtype=np.uint8)
    seq[:oix.seq_size] = oix.seq()
    blob = oix.blob()
    nreads = 2 * n_units if paired else n_units
    res = np.zeros(nreads, dtype=res_dtype)
    cap = 64 * nreads + 1024
    runs = np.zeros(cap, dtype=np.uint16)
    counters = np.zeros(8, dtype=np.uint32)
    p = Params(method, pe_method, band_radius, 10, 0)
    L.emu_set_second(second.ctypes.data_as(C.c_void_p) if second is not None else None)
    seqs = np.concatenate([np.asarray(seqs, dtype=np.uint8), np.zeros(64, dtype=np.uint8)])   # padded like the device buffer
    offs = np.ascontiguousarray(offs, dtype=np.uint32)
    vp = C.c_void_p
    rc = L.emu_map(blob.ctypes.data_as(vp), seq.ctypes.data_as(vp), C.c_uint32(oix.seq_size), C.c_uint64(oix.slot_count),
                   C.c_uint32(oix.word_length), C.c_uint32(oix.max_ix), C.byref(p), seqs.ctypes.data_as(vp),
                   offs.ctypes.data_as(vp), C.c_uint32(n_units), C.c_int(1 if paired else 0), res.ctypes.data_as(vp),
                   runs.ctypes.data_as(vp), C.c_uint32(cap), counters.ctypes.data_as(vp))
    assert rc == 0, rc
    return res, runs, counters


def emu_first_look() -> int:
    """Pairs the probe kernel's first look finished in the last emu_map call."""
    L = lib()
    L.emu_first_look.restype = C.c_uint32
    return int(L.emu_first_look())


def emu_build_index(seq: np.ndarray, slot_count: int, word_len: int = 24, max_ix: int = 32):
    """Runs the device index-builder kernels under emulation; returns (blob uint8[5*slot_count], stats)."""
    L = lib()
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    pad = np.zeros(len(seq) + 64, dtype=np.uint8)
    pad[:len(seq)] = seq
    blob = np.zeros(5 * slot_count + 16, dtype=np.uint8)
    stats = np.zeros(3, dtype=np.uint64)
    vp = C.c_void_p
    rc = L.emu_build_index(pad.ctypes.data_as(vp), C.c_uint64(len(seq)), C.c_uint64(slot_count), C.c_uint32(word_len),
                           C.c_uint32(max_ix), blob.ctypes.data_as(vp), stats.ctypes.data_as(vp))
    assert rc == 0
    return blob[:5 * slot_count], stats


def emu_flank_dp(A: bytes, B: bytes, left: bool, right: bool, method=6, band_radius=-1):
    """One flank DP of the kernels (flank_viterbi) under emulation: (score, path string, overflowed)."""
    L = lib()
    L.emu_flank_dp.restype = C.c_float
    p = Params(method, 4, band_radius, 10, 0)
    a = np.frombuffer(A, dtype=np.uint8).copy()
    b = np.concatenate([np.frombuffer(B, dtype=np.uint8), np.zeros(64, dtype=np.uint8)])
    buf = C.create_string_buffer(len(A) + len(B) + 8)
    ovf = C.c_int(0)
    vp = C.c_void_p
    sc = L.emu_flank_dp(C.byref(p), a.ctypes.data_as(vp), C.c_uint32(len(A)), b.ctypes.data_as(vp), C.c_uint32(len(B)),
                        C.c_int(int(left)), C.c_int(int(right)), buf, C.byref(ovf))
    return float(sc), buf.value.decode(), bool(ovf.value)
