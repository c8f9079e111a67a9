"""One Python API over the single-case runners of tests/kunit/kunit_cases.cuh.  Test infrastructure only.

Two back ends run the same runners on the product's device functions: "emu" (tests/emu/libemu.so, the lock-step warp
emulator, any machine) and "gpu" (tests/kunit/libkunit.so and libkunit_big.so, nvcc for sm_100a with the flags of
urmap_b200/csrc/Makefile; needs a CUDA device to run).  Libraries are rebuilt when a source is newer."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "urmap_b200", "csrc")
SOURCES = [os.path.join(HERE, "kunit_cases.cuh"), os.path.join(HERE, "kunit.cu"), os.path.join(CSRC, "urmb_kernels.cu"),
           os.path.join(CSRC, "urmb_internal.h"), os.path.join(ROOT, "include", "urmb.h")]
vp = C.c_void_p


def nvflags():
    """NVFLAGS of urmap_b200/csrc/Makefile with $(ARCH) expanded: the kernels are tested as the product compiles them."""
    mk = open(os.path.join(CSRC, "Makefile")).read()
    var = dict(re.findall(r"^(\w+)\s*:=\s*(.*)$", mk, re.M))
    return var["NVFLAGS"].replace("$(ARCH)", var["ARCH"]).split()


def _build_gpu(so, extra):
    srcs = SOURCES + [os.path.join(CSRC, "Makefile")]
    if os.path.exists(so) and all(os.path.getmtime(s) <= os.path.getmtime(so) for s in srcs):
        return None
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tmp = f"{so}.{os.getpid()}.tmp"
    cmd = [nvcc] + nvflags() + extra + ["-shared", "-o", tmp, os.path.join(HERE, "kunit.cu")]
    return so, tmp, subprocess.Popen(cmd)


def build_gpu():
    """libkunit.so and libkunit_big.so (-DURMB_BIG), compiled side by side."""
    jobs = [j for j in (_build_gpu(os.path.join(HERE, "libkunit.so"), []),
                        _build_gpu(os.path.join(HERE, "libkunit_big.so"), ["-DURMB_BIG"])) if j]
    for so, tmp, p in jobs:
        if p.wait() != 0:
            raise RuntimeError(f"nvcc failed building {so}")
        os.replace(tmp, so)


def _bind(L):
    L.ku_run_cap.restype = C.c_int
    L.ku_dp.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_uint32] + [vp] * 10
    L.ku_slots.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp, C.c_uint32, vp, vp]
    L.ku_mod.argtypes = [C.c_uint32, vp, vp, vp]
    L.ku_compchar.argtypes = [vp]
    L.ku_packed_words.restype = C.c_size_t
    L.ku_packed_words.argtypes = [C.c_size_t]
    L.ku_coarse_words.restype = C.c_size_t
    L.ku_coarse_words.argtypes = [C.c_size_t]
    L.ku_pack.argtypes = [vp, C.c_size_t, vp, vp, vp]
    L.ku_ext.argtypes = [C.c_int, C.c_uint32, C.c_uint32, vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, C.c_uint32, vp,
                         vp, vp]
    L.ku_mapq.argtypes = [C.c_uint32, vp, vp]
    return L


def _p(a):
    return a.ctypes.data_as(vp)


def _concat(seqs, pad):
    """bytes objects -> (concatenated uint8 array with `pad` zero bytes after the last, uint32 offsets)."""
    offs = np.zeros(len(seqs) + 1, dtype=np.uint32)
    offs[1:] = np.cumsum([len(s) for s in seqs])
    buf = np.zeros(int(offs[-1]) + pad, dtype=np.uint8)
    buf[:offs[-1]] = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    return buf, offs


def _seqcap(maxlen):
    return (max(maxlen, 32) + 31) & ~31


class Backend:
    def __init__(self, name):
        self.name = name
        if name == "emu":
            sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
            import emu_py
            self.lib = self.big = _bind(emu_py.lib())
        else:
            build_gpu()
            self.lib = _bind(C.CDLL(os.path.join(HERE, "libkunit.so")))
            self.big = _bind(C.CDLL(os.path.join(HERE, "libkunit_big.so")))

    def run_cap(self, big=False):
        return (self.big if big else self.lib).ku_run_cap()

    def dp(self, cases, kind=0, method=6, pe_method=4, band_radius=-1, seqcap=256, big=False):
        """cases: (A, B, left, right) tuples.  kind 0 = flank_viterbi, 1 = viterbi_full.  Returns per case (score, forward
        path string, ovf, guard bits); the path is None when ovf is set (the stored runs are truncated then)."""
        L = self.big if big else self.lib
        n = len(cases)
        A, aoff = _concat([c[0] for c in cases], 1)
        B, boff = _concat([c[1] for c in cases], 64)
        lr = np.array([int(c[2]) | (int(c[3]) << 1) for c in cases], dtype=np.uint8)
        nro = L.ku_run_cap() + 8
        score = np.zeros(n, np.float32)
        nrev = np.zeros(n, np.int32)
        ovf = np.zeros(n, np.int32)
        runs = np.zeros((n, nro), np.uint16)
        guard = np.zeros(n, np.uint32)
        rc = L.ku_dp(method, pe_method, band_radius, seqcap, kind, n, _p(A), _p(aoff), _p(B), _p(boff), _p(lr), _p(score),
                     _p(nrev), _p(ovf), _p(runs), _p(guard))
        assert rc == 0, f"ku_dp: {rc}"
        out = []
        for k in range(n):
            path = None
            if not ovf[k]:
                path = "".join("MDI"[r & 3] * (int(r) >> 2) for r in runs[k, :nrev[k]][::-1])
            out.append((float(score[k]), path, bool(ovf[k]), int(guard[k])))
        return out

    def slots(self, reads, slot_count, word_len):
        """slot_of for every k-mer of both strands of each read (stage_read first): [(plus, minus, hasbad, slow)]."""
        seqs, offs = _concat(reads, 64)
        nq = [max(len(r) - word_len + 1, 0) for r in reads]
        outoff = np.zeros(len(reads), np.uint32)
        outoff[1:] = np.cumsum([2 * q for q in nq])[:-1]
        nout = 2 * sum(nq)
        slots = np.zeros(max(nout, 1), np.uint64)
        flags = np.zeros(len(reads), np.uint8)
        rc = self.lib.ku_slots(slot_count, word_len, _seqcap(max(len(r) for r in reads)), len(reads), _p(seqs), _p(offs),
                               _p(outoff), nout, _p(slots), _p(flags))
        assert rc == 0, f"ku_slots: {rc}"
        out = []
        for r, q in enumerate(nq):
            o = int(outoff[r])
            out.append((slots[o:o + q], slots[o + q:o + 2 * q], bool(flags[r] & 1), bool(flags[r] & 2)))
        return out

    def mod(self, h, p):
        h = np.ascontiguousarray(h, np.uint64)
        p = np.ascontiguousarray(p, np.uint64)
        r = np.zeros(len(h), np.uint64)
        assert self.lib.ku_mod(len(h), _p(h), _p(p), _p(r)) == 0
        return r

    def compchar(self):
        out = np.zeros(256, np.uint8)
        assert self.lib.ku_compchar(_p(out)) == 0
        return out

    def pack(self, seq):
        seq = np.ascontiguousarray(np.frombuffer(seq, np.uint8) if isinstance(seq, bytes) else seq, np.uint8)
        nw, nc = self.lib.ku_packed_words(len(seq)), self.lib.ku_coarse_words(len(seq))
        seq2 = np.zeros(nw, np.uint64)
        seqx = np.zeros(nw, np.uint32)
        seqc = np.zeros(nc, np.uint32)
        assert self.lib.ku_pack(_p(seq), len(seq), _p(seq2), _p(seqx), _p(seqc)) == 0
        return seq2, seqx, seqc

    def ext(self, genome, reads, cases, word_len, method=6, flags=0):
        """cases: (read index, plus, SeedPosQ, SeedPosDB, LeftCountsPen, PenBound).  Returns uint32 [n, 3]: pure_ext_t<false>,
        pure_ext_t<true>, pure_ext_bytes (packed as ext_pack)."""
        g = np.frombuffer(genome, np.uint8)
        seqs, offs = _concat(reads, 64)
        cs = np.array([c[:5] for c in cases], dtype=np.uint32).reshape(-1, 5)
        pen = np.array([c[5] for c in cases], dtype=np.int32)
        out = np.zeros((len(cases), 3), np.uint32)
        rc = self.lib.ku_ext(method, flags, word_len, _p(g), len(g), _seqcap(max(len(r) for r in reads)), len(reads),
                             _p(seqs), _p(offs), len(cases), _p(cs), _p(pen), _p(out))
        assert rc == 0, f"ku_ext: {rc}"
        return out

    def mapq(self, ql, best, second, hitcount):
        a = np.ascontiguousarray(np.stack([ql, best, second, hitcount], axis=1), np.int32)
        out = np.zeros(len(a), np.uint32)
        assert self.lib.ku_mapq(len(a), _p(a), _p(out)) == 0
        return out
