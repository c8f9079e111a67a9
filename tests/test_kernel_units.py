"""The kernels' device functions, one case at a time, against exact references (tests/kunit).

Each test runs under the warp emulator (a seeded sample of its case list, any machine) and on the GPU (the full list,
marked gpu).  Every comparison is exact:
  flank DP (flank_viterbi: viterbi_band / viterbi_warp<true>) and rescue DP (viterbi_full) against the oracle's Viterbi:
      same score and forward path unless the oracle's traceback read a cell it never wrote (its result is undefined
      there: such cases are counted per shape class and excluded); ovf set iff the path has more than kRunCap runs;
      the canaries after the DP's shared-memory areas and after runs_a unchanged;
  gapless extension (pure_ext_t<false>, pure_ext_t<true>, pure_ext_bytes) against the walks of extendpen.cpp:29-78;
  stage_read + slot_of against the oracle's SetSlotsVec and a big-integer restatement, mod_slots, compchar_of;
  pack_genome_kernel against numpy; calc_mapq6 against binary64 arithmetic in the order of search1m6.cpp:9-33.
"""
import ctypes as C
import os
import random
import sys
import time

import numpy as np
import pytest

from conftest import CLI, ROOT, have_gpu, make_ufi

sys.path.insert(0, os.path.join(ROOT, "tests", "kunit"))
import kunit_py  # noqa: E402

EMU_SAMPLE = {"dp": 350, "rescue": 12, "ext": 1500, "slots": 60, "mapq": 4000}
M64 = (1 << 64) - 1
# (method, pe_method, band radius): -map (R 12), -map -veryfast (R 8), -map2 -veryfast (R 4)
DP_PARAMS = [(6, 4, 12), (7, 4, 8), (6, 5, 4)]
MM = {6: -3, 7: -4}
XDROP = {6: 9, 7: 12}


@pytest.fixture(scope="module", params=["emu", pytest.param("gpu", marks=pytest.mark.gpu)])
def be(request):
    if request.param == "gpu" and not have_gpu():
        pytest.skip("no CUDA device")
    return kunit_py.Backend(request.param)


def sample(be, cases, key, seed=0):
    """All cases on the GPU, a seeded sample under the emulator."""
    if be.name == "gpu" or len(cases) <= EMU_SAMPLE[key]:
        return cases
    return random.Random(seed).sample(cases, EMU_SAMPLE[key])


def rseq(rng, n, alpha=b"ACGT"):
    return bytes(rng.choice(alpha) for _ in range(n))


def runs_of(path):
    return sum(1 for k in range(len(path)) if k == 0 or path[k] != path[k - 1])


# ---------------------------------------------------------------------------------------------------------------------
# flank DP
# ---------------------------------------------------------------------------------------------------------------------
def derive(rng, B, LA, cls, R, at_end):
    """A read part of length LA for window B (aligned to B's end for a left flank, to its start for a right flank)."""
    if cls == "random" or len(B) == 0:
        return rseq(rng, LA)
    if cls == "homopolymer":
        return b"A" * LA
    if cls == "dinucleotide":
        return (b"AC" * LA)[:LA]
    src = bytearray(B[-LA:] if at_end and len(B) >= LA else B[:LA])
    src += rseq(rng, LA - len(src))
    offs = [o for o in (0, 1, LA // 2, LA - 1) if o < LA]
    if cls == "sub":
        o = rng.choice(offs)
        src[o] = ord(rng.choice([c for c in "ACGT" if ord(c) != src[o]]))
    elif cls in ("ins", "del"):
        o, g = rng.choice(offs), rng.choice([max(R - 1, 1), R, R + 1, 2 * R])
        if cls == "ins":
            src[o:o] = rseq(rng, g)
        else:
            del src[o:o + g]
        src = (src + bytearray(rseq(rng, LA)))[:LA]
    elif cls == "letters":
        for _ in range(max(1, LA // 10)):
            src[rng.randrange(LA)] = ord(rng.choice("NRYKMnacgt"))
    elif cls == "alternating":   # a base in, a base out, every few bases: many short runs
        out, k, step = bytearray(), 0, rng.choice([5, 6, 8])
        while k < len(src):
            out += src[k:k + step]
            out += rseq(rng, 1) if (k // step) % 2 == 0 else b""
            k += step + ((k // step) % 2)
        src = out[:LA] + bytearray(rseq(rng, max(0, LA - len(out))))
    return bytes(src)


CLASSES = ["equal", "sub", "ins", "del", "random", "homopolymer", "dinucleotide", "letters", "alternating"]


def flank_cases(rng, R, max_la=232):
    """(shape class, A, B, Left, Right) for the shapes align_hsp produces and the dispatch borders.  align_hsp's windows:
    left flank LB = LA + 2R (LeftTL = LeftQL + BRN R), right flank LB = LA + 2R + 1 (RightTHi = RightTLo + RightQL + BRN R,
    inclusive), clipped to 1 ... LA + 2R at the end of the genome."""
    out = []
    for LA in range(1, max_la + 1):
        cls = CLASSES[LA % len(CLASSES)]
        B = rseq(rng, LA + 2 * R + 1)
        out.append(("left", derive(rng, B[:-1], LA, cls, R, True), B[:-1], True, False))
        for LB in range(1, LA + 2 * R + 2):
            c = CLASSES[(LA + LB) % len(CLASSES)]
            Bc = B[:LB]
            if c in ("homopolymer", "dinucleotide"):
                Bc = derive(rng, b"", LB, c, R, False)
            out.append(("right" if LB == LA + 2 * R + 1 else "right-clipped", derive(rng, Bc, LA, c, R, False), Bc, False,
                        True))
    for LA in (R + 1, 40, 100, 150, 200):   # band width dhi - dlo + 1 = 63 / 64 / 65, window longer and shorter than A
        for bw in (63, 64, 65):
            for LB in (LA + bw - 1 - 2 * R, LA - (bw - 1 - 2 * R)):
                if LB >= 1:
                    B = rseq(rng, LB)
                    for lr in ((True, False), (False, True)):
                        out.append(("band-width", derive(rng, B, LA, rng.choice(CLASSES), R, lr[0]), B, *lr))
    for LA in (1, 5, 100):
        out.append(("degenerate", b"", rseq(rng, LA), True, False))
        out.append(("degenerate", rseq(rng, LA), b"", False, True))
    out.append(("degenerate", b"", b"", True, False))
    return out


def tb_rows_cases(rng, R, seqcap):
    """LA + 1 at and just above tb_rows = seqcap + 2: band in shared memory, then the row-block fallback."""
    out = []
    for LA in (seqcap, seqcap + 1, seqcap + 2):
        for lr in ((True, False), (False, True)):
            B = rseq(rng, LA + 2 * R)
            out.append(("tb-rows", derive(rng, B, LA, rng.choice(["equal", "sub", "ins", "del"]), R, lr[0]), B, *lr))
    return out


def row_block(LA, LB, R, seqcap):
    """flank_viterbi's dispatch: the row-block fallback viterbi_warp<true> instead of the band across the lanes."""
    lo = min(LA, LB) - R if min(LA, LB) > R else 1
    hi = min(max(LA, LB) + R, LA + LB - 1)
    return LA == 0 or LB == 0 or hi - lo + 1 > 64 or LA + 1 > seqcap + 2


GAP = {6: (-5, -1), 7: (-6, -2)}   # GO, GE


MAX_PENALTY = 130   # State1::m_MaxPenalty never exceeds max(MAXPEN, 130): MAXPEN is 100 / 75, Scan sets 130 (scan.cpp)


def known_row_block_difference(method, R, seqcap, A, B, sc, osc):
    """The difference of viterbi_warp<true> from the reference that DESIGN.md §7 describes, on a flank the row-block
    fallback takes: either a shape align_hsp never cuts (a window longer than LA + 2R + 1, or LA + 1 > tb_rows: a flank is
    shorter than its read), or a flank whose penalty alone, LA - max(score, AllGapScore), exceeds every penalty bound with
    either score, so that align_hsp drops the hit in both."""
    LA, LB = len(A), len(B)
    if not row_block(LA, LB, R, seqcap) or min(LA, LB) == 0:
        return False
    if LB > LA + 2 * R + 1 or LA + 1 > seqcap + 2:
        return True
    go, ge = GAP[method]
    allgap = go + (LA - 1) * ge
    return LA - max(sc, allgap) > MAX_PENALTY and LA - max(osc, allgap) > MAX_PENALTY


def check_dp(be, cases, kind, method, pe_method, R, seqcap, oracle, big=False, tolerate=False):
    """Runs the cases; returns {shape class: [cases, poison-excluded cases]}.  With `tolerate`, the known difference of the
    row-block fallback (known_row_block_difference) is counted under (class, "differs") instead of failing."""
    got = be.dp([c[1:] for c in cases], kind=kind, method=method, pe_method=pe_method, seqcap=seqcap, big=big)
    cap = be.run_cap(big)
    counts, bad = {}, []
    for (cls, A, B, left, right), (sc, path, ovf, guard) in zip(cases, got):
        if kind == 0 and row_block(len(A), len(B), R, seqcap):
            cls += "/row-block"
        n = counts.setdefault(cls, [0, 0])
        n[0] += 1
        osc, opath, poison = oracle.viterbi_ex(A, B, left, right, method=method, band_radius=R)
        if guard:
            bad.append((cls, len(A), len(B), left, right, "guard", guard))
        if poison:
            n[1] += 1
            continue
        want_ovf = runs_of(opath) > cap
        if sc != osc or ovf != want_ovf or (not ovf and path != opath):
            if tolerate and known_row_block_difference(method, R, seqcap, A, B, sc, osc):
                counts.setdefault((cls, "differs"), [0, 0])[0] += 1
                continue
            bad.append((cls, len(A), len(B), left, right, A, B, (sc, osc), (ovf, want_ovf), path, opath))
    assert not bad, f"{len(bad)} of {len(cases)} cases differ, first: {bad[:3]}"
    return counts


@pytest.mark.parametrize("method,pe_method,R", DP_PARAMS)
def test_flank_dp(be, oracle, method, pe_method, R):
    rng = random.Random(1000 + R)
    t0 = time.time()
    counts = {}
    for seqcap in (160, 256):   # read parts up to seqcap - 1 bases (a flank is shorter than the read)
        cases = flank_cases(rng, R, min(232, seqcap - 1)) + tb_rows_cases(rng, R, seqcap)
        cases = sample(be, cases, "dp", seed=seqcap + R)
        for cls, n in check_dp(be, cases, 0, method, pe_method, R, seqcap, oracle, tolerate=True).items():
            counts.setdefault(cls, [0, 0])
            counts[cls] = [counts[cls][0] + n[0], counts[cls][1] + n[1]]
    print(f"\n[{be.name}] flank DP R={R}: {sum(v[0] for k, v in counts.items() if isinstance(k, str))} cases in {time.time() - t0:.1f} s; "
          f"(cases, excluded for traceback reads of unwritten cells) by shape: {counts}")
    # the shapes align_hsp produces (left flank LB = LA + 2R, right flank LB <= LA + 2R + 1) are always comparable
    for cls, n in counts.items():
        if isinstance(cls, str) and cls.split("/")[0] in ("left", "right", "right-clipped"):
            assert n[1] == 0, (cls, n)


# Cases of row_block_cases whose score or path differs from the reference (every one a known_row_block_difference).
ROW_BLOCK_DIFFERS = {12: [5, 51, 78, 96, 104, 141, 159], 8: [14, 41, 42, 113, 194, 213], 4: [32, 69, 104, 123, 132, 140, 167, 185, 186]}


def row_block_cases(R, n=240):
    """Right flanks that flank_viterbi sends to the row-block fallback viterbi_warp<true>: windows clipped at the end of
    the genome so far that the band is wider than 64 (the read part overhangs the window by 64 - 2R bases or more)."""
    rng, out = random.Random(1500 + R), []
    while len(out) < n:
        LA = rng.randrange(64 - 2 * R + 1, 130)
        LB = rng.randrange(1, LA - (64 - 2 * R) + 1)
        if row_block(LA, LB, R, 256):
            B = rseq(rng, LB)
            out.append((derive(rng, B, LA, CLASSES[len(out) % len(CLASSES)], R, False), B, False, True))
    return out


@pytest.mark.parametrize("method,pe_method,R", DP_PARAMS)
def test_flank_dp_row_block(be, oracle, method, pe_method, R):
    """viterbi_warp<true> differs from State1::Viterbi on a few per cent of the shapes it takes (DESIGN.md §7).  Pinned: the
    differing cases of a fixed list are exactly ROW_BLOCK_DIFFERS, and each is a known_row_block_difference.
    A fix of the fallback, or a difference of another kind, fails here."""
    cases = row_block_cases(R)
    got = be.dp(cases, method=method, pe_method=pe_method, seqcap=256)
    differs = []
    for k, ((A, B, left, right), (sc, path, ovf, guard)) in enumerate(zip(cases, got)):
        osc, opath, poison = oracle.viterbi_ex(A, B, left, right, method=method, band_radius=R)
        assert guard == 0 and poison == 0, (k, guard, poison)
        if sc != osc or path != opath:
            differs.append(k)
            assert known_row_block_difference(method, R, 256, A, B, sc, osc), (k, len(A), len(B), sc, osc)
    assert differs == ROW_BLOCK_DIFFERS[R]


@pytest.mark.gpu
def test_flank_dp_big(be, oracle):
    """The build that maps reads over a capacity again (-DURMB_BIG, kRunCap 192): same DP, a larger run cap."""
    if be.name != "gpu":
        pytest.skip("the big-capacity build is a GPU build")
    assert be.run_cap(big=True) == 192
    rng = random.Random(77)
    for method, pe_method, R in DP_PARAMS:
        cases = [c for c in flank_cases(rng, R) if c[0] != "right-clipped" or len(c[1]) % 7 == 0]
        cases += [("alt", derive(rng, B, 232, "alternating", R, False), B, False, True)
                  for B in (rseq(rng, 232 + 2 * R) for _ in range(40))]
        check_dp(be, cases, 0, method, pe_method, R, 256, oracle, big=True, tolerate=True)


# ---------------------------------------------------------------------------------------------------------------------
# rescue DP (State1::Scan: Left = Right = true, LA = mate length, LB = 1024 or 1024 + 2 QL of the other mate)
# ---------------------------------------------------------------------------------------------------------------------
RESCUE_LA = [1, 31, 32, 33, 63, 64, 65, 150, 255, 256]


def rescue_cases(rng, R, seqcap):
    out = []
    las = [la for la in RESCUE_LA if la <= seqcap]
    lbs = {1024, 1024 + 2 * 1, 1024 + 2 * 100, 1024 + 2 * 256}
    if seqcap == 32:   # tb_rows 34: windows of up to 34 * 32 - 4 = 1084 bases sit in shared memory, longer ones stay global
        lbs |= {1083, 1084, 1085, 1088}
    for LA in las:
        for LB in sorted(lbs):
            B = rseq(rng, LB)
            o = rng.randrange(0, LB - LA + 1)
            A = bytearray(B[o:o + LA])
            cls = rng.choice(["equal", "sub", "indel", "random"])
            if cls == "sub":
                for _ in range(1 + LA // 20):
                    A[rng.randrange(LA)] = ord(rng.choice("ACGT"))
            elif cls == "indel" and LA > 4:
                k = rng.randrange(1, LA - 1)
                A = (A[:k] + (rseq(rng, R) if rng.random() < 0.5 else b"") + A[k + rng.choice([0, 1, R]):])[:LA]
                A += rseq(rng, LA - len(A))
            elif cls == "random":
                A = bytearray(rseq(rng, LA))
            out.append((f"scan-{'global' if seqcap == 32 and LB > 1084 else 'shared'}", bytes(A), B, True, True))
    return out


@pytest.mark.parametrize("method,pe_method,R", DP_PARAMS)
def test_rescue_dp(be, oracle, method, pe_method, R):
    rng = random.Random(2000 + R)
    for seqcap in (32, 160, 256):
        cases = rescue_cases(rng, R, seqcap)
        if be.name == "emu":   # the emulator takes seconds per full window: short reads only
            cases = random.Random(seqcap).sample([c for c in cases if len(c[1]) <= 65], min(EMU_SAMPLE["rescue"], 20))
        counts = check_dp(be, cases, 1, method, pe_method, R, seqcap, oracle)
        print(f"\n[{be.name}] rescue DP R={R} seqcap={seqcap}: {counts}")


# ---------------------------------------------------------------------------------------------------------------------
# gapless extension
# ---------------------------------------------------------------------------------------------------------------------
def ext_ref(Q, T, sq, W, mm, xd, lcp):
    """ExtendPen's walks without the penalty bound (extendpen.cpp:29-78): Best, Start, End, visited mismatches.
    T[p] is the genome byte under read position p."""
    QL = len(Q)
    score, best, nmis, end = W, 0, 0, sq + W - 1
    for p in range(end + 1, QL):
        if Q[p] == T[p]:
            score += 1
            if score > best:
                best, end = score, p
        else:
            nmis += 1
            score += mm
            if best - score > xd:
                break
    start = sq
    for p in range(sq - 1, -1, -1):
        if Q[p] == T[p]:
            score += 1
            if score > best:
                best, start = score, p
        else:
            nmis += lcp
            score += mm
            if best - score > xd:
                break
    return best, start, end, nmis


def unpack(x):
    return x & 511, (x >> 9) & 255, (x >> 17) & 255, x >> 25


COMP = bytes.maketrans(b"ACGT", b"TGCA")
EXT_QL = [24, 25, 31, 32, 33, 47, 48, 159, 160, 161, 176, 255, 256]


def ext_cases(rng, W, method, n_blocks=260):
    """Genome with exception sites, reads and candidates: [(read, plus, SeedPosQ, SeedPosDB, LeftCountsPen, PenBound)]."""
    mm = MM[method]
    G = bytearray(rseq(rng, 2048 * n_blocks))
    reads, cases = [], []

    def add(read, plus, sq, dblo, lcp=None, pen=None):
        reads.append(bytes(read) if plus else bytes(read).translate(COMP)[::-1])
        maxmis = rng.choice([0, 1, 2, 5, 125, 126, 127, 300])
        pen = maxmis * -mm + rng.randrange(-mm) if pen is None else pen
        cases.append((len(reads) - 1, int(plus), sq, dblo + sq, int(rng.random() < 0.7) if lcp is None else lcp, pen))

    def window(dblo, QL):
        w = bytearray(G[dblo:dblo + QL])
        return w + bytearray(rseq(rng, QL - len(w)))

    def mutate(w, sq, extra=()):
        QL = len(w)
        spots = [sq + W, QL - 1] + [16 * k + d for k in range(1, QL // 16 + 1) for d in (-1, 0)] + list(extra)
        for p in rng.sample(spots, min(len(spots), rng.choice([0, 1, 2, 3, 4]))):
            if 0 <= p < QL:
                w[p] = ord(rng.choice([c for c in "ACGT" if ord(c) != w[p]]))
        if rng.random() < 0.4:   # a run of 3 or 4 mismatches: Best - Score reaches XD or XD + 1 (method 6; 2-3 for method 7)
            k = rng.choice([3, 4])
            p = rng.randrange(QL)
            for q in range(p, min(QL, p + k)):
                w[q] = ord(rng.choice([c for c in "ACGT" if ord(c) != w[q]]))
        if rng.random() < 0.3:   # many mismatches: the maxmis cap
            for _ in range(rng.randrange(QL)):
                p = rng.randrange(QL)
                w[p] = ord(rng.choice("ACGT"))
        return w

    def seedpos(QL):
        return rng.choice([0, 1, max(QL - W - 1, 0), QL - W, rng.randrange(QL - W + 1)])

    # clean windows: every QL, every DBLo residue mod 32, both strands
    for QL in EXT_QL:
        for res in range(32):
            dblo = 2048 * rng.randrange(1, n_blocks - 1) + 300 + res - (300 % 32)
            sq = seedpos(QL)
            add(mutate(window(dblo, QL), sq), rng.random() < 0.5, sq, dblo)
    # exception bytes in the genome: first / last byte of the window, one byte outside, only in the second 1024-base block
    blk = 1
    for QL in EXT_QL:
        for where in ("first", "last", "before", "after", "cb1"):
            for _ in range(3):
                base = 2048 * blk
                blk += 1
                if where == "cb1":   # window crosses the block border at base + 1024, the exception lies past it
                    dblo = base + 1024 - rng.randrange(1, QL) if QL > 1 else base + 1023
                    site = rng.randrange(base + 1024, dblo + QL) if dblo + QL > base + 1024 else base + 1024
                else:
                    dblo = base + 512 + rng.randrange(32)
                    site = {"first": dblo, "last": dblo + QL - 1, "before": dblo - 1, "after": dblo + QL}[where]
                G[site] = ord(rng.choice("NRY-"))
                sq = seedpos(QL)
                w = mutate(window(dblo, QL), sq)
                if dblo <= site < dblo + QL:
                    w[site - dblo] = ord("A")   # what the 2-bit code of a non-ACGT byte reads as
                add(w, True, sq, dblo)
    # windows running into the zero padding after the genome; reads with lower-case / IUPAC letters; EXT_NONE
    for QL in EXT_QL:
        for _ in range(4):
            d = rng.randrange(1, QL - W + 1) if QL > W else 0
            dblo = len(G) - QL + d
            add(mutate(window(dblo, QL), 0), True, 0, dblo)
            dblo = 2048 * rng.randrange(1, n_blocks - 1) + rng.randrange(1024)
            sq = seedpos(QL)
            w = mutate(window(dblo, QL), sq)
            for _ in range(rng.randrange(1, 4)):
                w[rng.randrange(QL)] = ord(rng.choice("acgtNRn"))
            add(w, True, sq, dblo, lcp=rng.choice([0, 1]))
        sq = rng.randrange(1, QL - W + 1) if QL > W else 0
        if sq:
            add(window(0, QL), True, sq, -rng.randrange(1, sq + 1))
    assert blk < n_blocks
    return bytes(G), reads, cases


@pytest.mark.parametrize("method", [6, 7])
@pytest.mark.parametrize("flags", [0, 32])
def test_gapless_extension(be, method, flags):
    W = 24
    rng = random.Random(3000 + method + flags)
    G, reads, cases = ext_cases(rng, W, method)
    cases = sample(be, cases, "ext", seed=method + flags)
    t0 = time.time()
    out = be.ext(G, reads, cases, W, method=method, flags=flags)
    bad = []
    mm, xd = MM[method], XDROP[method]
    for (r, plus, sq, sdb, lcp, pen), x in zip(cases, out):
        Q = reads[r] if plus else reads[r].translate(COMP)[::-1]
        if sdb < sq:
            if not (x == 0xFFFFFFFF).all():
                bad.append(("EXT_NONE", r, sq, sdb, x))
            continue
        dblo = sdb - sq
        T = (G + bytes(4096))[dblo:dblo + len(Q)]
        ref = ext_ref(Q, T, sq, W, mm, xd, lcp)
        maxmis = min(pen // -mm, 126)
        if unpack(int(x[2])) != ref[:3] + (min(ref[3], 127),):
            bad.append(("bytes", len(Q), sq, dblo, lcp, unpack(int(x[2])), ref))
        for k in (0, 1):
            u = unpack(int(x[k]))
            if (u[3] > maxmis) != (ref[3] > maxmis) or (ref[3] <= maxmis and u != ref):
                bad.append((f"pure_ext_t<{bool(k)}>", len(Q), sq, dblo, lcp, pen, u, ref))
    print(f"\n[{be.name}] gapless extension method {method} flags {flags}: {len(cases)} cases in {time.time() - t0:.1f} s")
    assert not bad, f"{len(bad)} of {len(cases)} differ, first: {bad[:4]}"


# ---------------------------------------------------------------------------------------------------------------------
# hashing
# ---------------------------------------------------------------------------------------------------------------------
LETTER = {ord(c): i for i, c in enumerate("ACGT")}
LETTER.update({ord(c): i for i, c in enumerate("acgt")})
LETTER.update({ord("U"): 3, ord("u"): 3})


def murmur64(h):
    h ^= h >> 33
    h = (h * 0xff51afd7ed558ccd) & M64
    h ^= h >> 33
    h = (h * 0xc4ceb9fe1a85ec53) & M64
    h ^= h >> 33
    return h


def slots_ref(seq, W, p):
    """SetSlotsVec restated with Python integers: 2-bit word of each k-mer, murmur64, % slot count; 2^64 - 1 where a letter
    is not ACGTU."""
    out = []
    for q in range(len(seq) - W + 1):
        k = seq[q:q + W]
        if any(c not in LETTER for c in k):
            out.append(M64)
            continue
        word = 0
        for c in k:
            word = (word << 2) | LETTER[c]
        out.append(murmur64(word & ((1 << 2 * W) - 1)) % p)
    return out


def revcomp(oracle, seq):
    a = np.frombuffer(seq, np.uint8)
    out = np.zeros(max(len(a), 1), np.uint8)
    oracle.lib().uo_revcomp(a.ctypes.data_as(C.c_void_p), len(a), out.ctypes.data_as(C.c_void_p))
    return out[:len(a)].tobytes()


def hash_reads(rng, genome, W):
    reads = []
    for L in range(1, 257):
        o = rng.randrange(len(genome) - L)
        r = bytearray(genome[o:o + L])
        kind = L % 4
        if kind == 1:   # invalid letters at the first, last, a word-border position and a random one
            for p in {0, L - 1, min(L - 1, 31), min(L - 1, 32), rng.randrange(L)}:
                r[p] = ord(rng.choice("NRYn.-"))
        elif kind == 2:
            for _ in range(1 + L // 16):
                r[rng.randrange(L)] = ord(rng.choice("acgtuU"))
        reads.append(bytes(r))
    return reads


def test_slots_golden_index(be, oracle, golden_oix):
    ix = golden_oix
    rng = random.Random(4000)
    genome = ix.seq().tobytes()
    reads = hash_reads(rng, genome, ix.word_length)
    reads = sample(be, reads, "slots", seed=1)
    got = be.slots(reads, ix.slot_count, ix.word_length)
    for r, (p, m, _, _) in zip(reads, got):
        op, om = oracle.slots(ix, r)
        assert (p == op).all() and (m == om).all(), (r, np.nonzero(p != op)[0], np.nonzero(m != om)[0])


@pytest.mark.parametrize("W", [20, 32])
def test_slots_built_index(be, oracle, built_lib, tmp_path, W):
    """Indexes built with -wordlength 20 (the reference's file, pinned by its digest as in test_index_build) and 32, the
    longest word the mapper accepts: slot_of against the oracle's SetSlotsVec."""
    import subprocess
    from urmap_b200 import synth
    g = synth.make_genome(400_000, n_contigs=3, seed=31, repeat_frac=0.15, n_runs=[(1, 0.3, 900)], tandem=15, segdup=4)
    fa, ufi = str(tmp_path / "r.fa"), str(tmp_path / "r.ufi")
    g.write_fasta(fa)
    if W == 20:
        make_ufi("r_400kb_seed31_maxix_5_wordlength_20", fa, ufi, ["-maxix", "5", "-wordlength", "20"])
    else:
        subprocess.run([CLI, "-make_ufi", fa, "-output", ufi, "-wordlength", str(W), "-quiet"], check=True)
    ix = oracle.Index(ufi)
    assert ix.word_length == W
    reads = sample(be, hash_reads(random.Random(4100 + W), ix.seq().tobytes(), W), "slots", seed=W)
    for r, (p, m, _, _) in zip(reads, be.slots(reads, ix.slot_count, W)):
        op, om = oracle.slots(ix, r)
        assert (p == op).all() and (m == om).all(), (W, r, np.nonzero(p != op)[0], np.nonzero(m != om)[0])
    ix.close()


# slot counts: small primes, 2^31 - 1, the primes just below and above 2^32, the human-scale count (above 2^32)
SLOT_COUNTS = [2, 3, 7, 65521, 2147483647, 4294967291, 4294967311, 5392814809]


@pytest.mark.parametrize("W", [20, 24, 32])
def test_slots_restatement(be, oracle, W):
    rng = random.Random(5000 + W)
    genome = rseq(rng, 20000)
    reads = hash_reads(rng, genome, W)
    for p in SLOT_COUNTS:
        rs = sample(be, reads, "slots", seed=p)
        got = be.slots(rs, p, W)
        for r, (gp, gm, _, _) in zip(rs, got):
            assert gp.tolist() == slots_ref(r, W, p), (p, r)
            assert gm.tolist() == slots_ref(revcomp(oracle, r), W, p), (p, r)


def test_mod_slots(be):
    h, p = [], []
    for P in SLOT_COUNTS + [(1 << 62) - 57, 1000003]:
        K = M64 // P
        for k in (K, K - 1, K - 2, 1, 2, 12345):
            for d in (-1, 0, 1):
                v = k * P + d
                if 0 <= v <= M64:
                    h.append(v)
                    p.append(P)
        h.append(M64)
        p.append(P)
        h += [random.Random(P).getrandbits(64) for _ in range(50)]
        p += [P] * 50
    got = be.mod(np.array(h, dtype=np.uint64), np.array(p, dtype=np.uint64))
    want = [a % b for a, b in zip(h, p)]
    bad = [(a, b, int(g), w) for a, b, g, w in zip(h, p, got, want) if int(g) != w]
    assert not bad, bad[:5]


def test_compchar(be, oracle):
    allb = bytes(range(256))
    want = revcomp(oracle, allb)[::-1]
    got = be.compchar().tobytes()
    assert got == want, [(c, got[c], want[c]) for c in range(256) if got[c] != want[c]]


# ---------------------------------------------------------------------------------------------------------------------
# genome packing
# ---------------------------------------------------------------------------------------------------------------------
def pack_ref(seq, nw, nc):
    a = np.zeros(nw * 32, np.uint8)
    a[:len(seq)] = np.frombuffer(seq, np.uint8)
    code = np.zeros(len(a), np.uint64)
    for i, c in enumerate(b"ACGT"):
        code[a == c] = i
    exc = ~np.isin(a, np.frombuffer(b"ACGT", np.uint8))
    sh = (62 - 2 * np.arange(32, dtype=np.uint64)).astype(np.uint64)
    seq2 = np.bitwise_or.reduce(code.reshape(nw, 32) << sh, axis=1)
    seqx = np.bitwise_or.reduce(exc.reshape(nw, 32).astype(np.uint32) << np.arange(32, dtype=np.uint32), axis=1)
    seqc = np.zeros(nc, np.uint32)
    for b in np.unique(np.nonzero(seqx)[0] * 32 >> 10):
        seqc[b >> 5] |= np.uint32(1 << (b & 31))
    return seq2, seqx, seqc


@pytest.mark.parametrize("n", [1, 31, 33, 1023, 1025, 5000 + 7, 40000 + 3])
def test_pack_genome(be, n):
    rng = random.Random(6000 + n)
    seqs = [rseq(rng, n), bytes(rng.randrange(256) for _ in range(n))]
    for offs in ((31,), (32,), (1023,), (1024,), (n - 1,), (31, 1024, n - 1)):
        s = bytearray(rseq(rng, n))
        for o in offs:
            if o < n:
                s[o] = ord(rng.choice("NRn-a")) if rng.random() < 0.8 else 0
        seqs.append(bytes(s))
    if n >= 256:
        seqs.append((bytes(range(256)) * (n // 256 + 1))[:n])
    for s in seqs:
        got = be.pack(s)
        want = pack_ref(s, len(got[0]), len(got[2]))
        for name, g, w in zip(("seq2", "seqx", "seqc"), got, want):
            assert (g == w).all(), (name, n, np.nonzero(g != w)[0][:5])


# ---------------------------------------------------------------------------------------------------------------------
# CalcMAPQ6
# ---------------------------------------------------------------------------------------------------------------------
def mapq_ref(ql, best, second, hc):
    """search1m6.cpp:9-33 in binary64, same operation order."""
    bp = ql.astype(np.float64)
    s = second.astype(np.float64)
    low = s < bp / 2.0
    s = np.where(low, bp / 2.0, s)
    b = best.astype(np.float64)
    zero = (hc == 0) | (best <= 0) | (low & (b <= s))
    fract = b / bp
    drop = np.minimum(b - s, 40.0)
    v = (drop * fract) * fract
    m = np.minimum(np.trunc(np.where(zero, 0.0, v)), 40).astype(np.uint32)
    return np.where(zero, 0, m).astype(np.uint32)


def test_calc_mapq6(be):
    ql, best, second = [], [], []
    for q in range(1, 257):   # Best <= QL, Second from -50 to Best
        for b in range(-2, q + 1):
            s = np.arange(-50, b + 1)
            ql.append(np.full(len(s), q))
            best.append(np.full(len(s), b))
            second.append(s)
    ql, best, second = (np.concatenate(x).astype(np.int32) for x in (ql, best, second))
    n = len(ql)
    ql, best, second = np.tile(ql, 2), np.tile(best, 2), np.tile(second, 2)
    hc = np.repeat(np.array([0, 1], np.int32), n)
    if be.name == "emu":
        sel = np.random.default_rng(7).choice(len(ql), EMU_SAMPLE["mapq"], replace=False)
        sel = np.concatenate([sel, np.nonzero((hc == 1) & (2 * second == ql) & (best >= second))[0][::97]])
        ql, best, second, hc = ql[sel], best[sel], second[sel], hc[sel]
    t0 = time.time()
    got = be.mapq(ql, best, second, hc)
    want = mapq_ref(ql, best, second, hc)
    print(f"\n[{be.name}] calc_mapq6: {len(ql)} cases in {time.time() - t0:.1f} s")
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, [(ql[i], best[i], second[i], hc[i], got[i], want[i]) for i in bad[:5]]
