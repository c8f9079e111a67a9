// oracle/urmap_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// Scalar CPU restatement of URMAP's mapping hot path, written from the semantics in
// SURVEY.md §8a; every function cites the reference file:line it follows (paths are under
// /root/reference/src).  It exists so that tests can (1) check themselves against the
// unmodified reference binary (oracle/_ref/urmap) at the SAM level and (2) check the CUDA
// path field by field at the C-ABI result level.  The product never links this file.
//
// Parity status: PINNED (see urmap_oracle.h).
//
// Deliberate, documented deviations from the reference's undefined behaviour:
//  * genome bytes at offsets >= SeqDataSize read as 0 (the reference reads past its malloc
//    in extendpen.cpp:31, scan.cpp:28, scanslots.cpp:16);
//  * traceback cells the current Viterbi call never wrote read as 0 (the reference reads
//    stale bytes of earlier calls, xdpmem.h:79; SURVEY.md quirk 12 shows this never changes
//    SAM output; `tb_poison_reads` counts how often it happens here).
#include "urmap_oracle.h"

#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <string>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <vector>

#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

typedef uint8_t byte;
typedef uint32_t uint32;
typedef uint64_t uint64;
typedef int64_t int64;

// ---- tally encoding, ufindex.h:23-36 ---------------------------------------------------
const byte T_FREE = 0, T_END = 127, T_MY_BIT = 128, T_PLUS1 = 254, T_BOTH1 = 255;
const byte T_NEXT_MASK = 127, T_LONG_MINE = 253, T_LONG_OTHER = 125;
inline bool TallyMine(byte t) { return (t & T_MY_BIT) != 0; }   // ufindex.h:72
inline bool TallyOther(byte t) { return (t & T_MY_BIT) == 0; }  // ufindex.h:82

// ---- constants, state1.h:12-19 ---------------------------------------------------------
const int SECONDARY_HIT_MAX_DELTA = 12;
const unsigned PRIME_STRIDE = 27;
const unsigned SCANK = 4;
const int MAX_TL = 1000;
const unsigned BRN = 2;  // alignhsp.cpp:11

// trace bits, tracebit.h:4-7
const byte TB_DM = 1, TB_IM = 2, TB_MD = 4, TB_MI = 8, TB_POISON = 0x10;

// ---- alphabet tables (semantics of alpha.cpp:1309, 3005, 3525) -------------------------
byte g_Letter[256], g_CompChar[256], g_CompLetter[256];
struct TableInit {
    TableInit() {
        memset(g_Letter, 0xFF, 256);
        memset(g_CompLetter, 0xFF, 256);
        memset(g_CompChar, '?', 256);
        const char *s = "ACGTU";
        const byte v[5] = {0, 1, 2, 3, 3};
        for (int i = 0; i < 5; ++i) {
            g_Letter[(byte)s[i]] = v[i];
            g_Letter[(byte)(s[i] | 0x20)] = v[i];
            g_CompLetter[(byte)s[i]] = 3 - v[i];
            if (s[i] != 'U') g_CompLetter[(byte)(s[i] | 0x20)] = 3 - v[i];  // 'u' is invalid there
        }
        const char *from = "ABCDGHKMNRSTUVWXY";
        const char *to = "TVGHCDMKNYSAABWXR";
        for (int i = 0; from[i]; ++i) {
            g_CompChar[(byte)from[i]] = (byte)to[i];
            if (from[i] != 'U') g_CompChar[(byte)(from[i] | 0x20)] = (byte)(to[i] | 0x20);
        }
    }
} g_TableInit;

inline uint64 murmur64(uint64 h) {  // ufindex.h:50
    h ^= (h >> 33);
    h *= 0xff51afd7ed558ccdULL;
    h ^= (h >> 33);
    h *= 0xc4ceb9fe1a85ec53ULL;
    h ^= (h >> 33);
    return h;
}

struct Params {  // State1::SetMethod, state1.cpp:147-183
    int MM, GO, GE, MIN_HSP_PCT, TERM3_PCT, XDROP, MAXPEN, XP1, XP3, XP4;
    unsigned R;
    int pe_method;
};

Params MakeParams(const uo_params *p) {
    Params P;
    if (p->method == 7) {
        P = Params{-4, -6, -2, 35, 35, 12, 75, 8, 6, 5, 8, 4};
    } else {
        P = Params{-3, -5, -1, 20, 60, 9, 100, 1, 1, 1, 12, 4};
    }
    if (p->band_radius >= 0) P.R = (unsigned)p->band_radius;
    P.pe_method = p->pe_method == 5 ? 5 : 4;
    return P;
}

}  // namespace

struct uo_index {
    int fd = -1;
    byte *map = nullptr;
    size_t map_len = 0;
    uint32 WordLength = 0, MaxIx = 0, SeqDataSize = 0;
    uint64 SlotCount = 0, ShiftMask = 0;
    std::vector<std::string> Labels;
    std::vector<uint32> SeqLengths, Offsets;
    const byte *Blob = nullptr;
    const byte *SeqData = nullptr;

    inline byte T(uint64 pos) const { return pos < SeqDataSize ? SeqData[pos] : 0; }
    inline uint64 WordToSlot(uint64 w) const { return murmur64(w) % SlotCount; }  // ufindex.h:60

    // UFIndex::PosToCoordL, ufindex.cpp:729-755. Returns UINT32_MAX in padding.
    uint32 PosToCoordL(uint32 Pos, int &SeqIndexOut, unsigned &L) const {
        const unsigned SeqCount = (unsigned)Labels.size();
        int64 Lo = 0, Hi = (int64)SeqCount - 1;
        while (Lo <= Hi) {
            unsigned SeqIndex = (unsigned)((Lo + Hi) / 2);
            uint32 Offset = Offsets[SeqIndex];
            uint32 SeqLength = SeqLengths[SeqIndex];
            if (Pos >= Offset && Pos < Offset + SeqLength) {
                SeqIndexOut = (int)SeqIndex;
                L = SeqLength;
                return Pos - Offset;
            } else if (Pos > Offset)
                Lo = (int64)SeqIndex + 1;
            else
                Hi = (int64)SeqIndex - 1;
        }
        SeqIndexOut = -1;
        return UINT32_MAX;
    }
};

namespace {

struct Hit {  // ufihit.h
    uint32 pos;
    bool plus;
    int score;
    std::string path;
};
struct HSP {  // ufihsp.h
    uint32 qstart, dbstart, len;
    int score;
    bool plus, aligned;
};

// DiagBox::GetRange_j, diagbox.h:150-170
inline void RangeJ(unsigned LA, unsigned LB, unsigned dlo, unsigned dhi, unsigned i, unsigned &Startj,
                   unsigned &Endj) {
    Startj = (dlo + i >= LA) ? dlo + i - LA : 0;
    if (Startj >= LB) Startj = LB - 1;
    Endj = (dhi + i + 1 >= LA) ? dhi + i + 1 - LA : 0;
    if (Endj > LB) Endj = LB;
}

// PathInfo::TrimLeftIs, pathinfo.cpp:168-185
unsigned TrimLeftIs(std::string &p) {
    unsigned n = 0;
    while (n < p.size() && p[n] == 'I') ++n;
    p.erase(0, n);
    return n;
}
// PathInfo::TrimRightIs, pathinfo.cpp:187-202 (never removes index 0)
void TrimRightIs(std::string &p) {
    if (p.empty()) return;
    for (size_t i = p.size() - 1; i > 0; --i) {
        if (p[i] == 'I')
            p.pop_back();
        else
            return;
    }
}

// State1::Viterbi, viterbi.cpp:11-261 + TraceBackBitMem, tracebackbitmem.cpp:8-75
float Viterbi(const Params &P, const byte *A, unsigned LA, const byte *B, unsigned LB, bool Left,
              bool Right, std::string &Path, uo_stats *st) {
    Path.clear();
    const int GAP_OPEN_SCORE = P.GO, GAP_EXT_SCORE = P.GE, MISMATCH_SCORE = P.MM;
    if (LA == 0 || LB == 0) {  // viterbi.cpp:14-36 (same integer-type arithmetic)
        if (LA == 0 && LB == 0) return 0.0f;
        if (LA == 0) {
            Path.assign(LB, 'I');
            return float(GAP_OPEN_SCORE + (LB - 1) * GAP_EXT_SCORE);
        }
        Path.assign(LA, 'D');
        return float(GAP_OPEN_SCORE + (LA - 1) * GAP_EXT_SCORE);
    }
    const float NEG = -9e9f;  // MINUS_INFINITY, mx.h:12
    unsigned DiagLo = std::min(LA, LB), DiagHi = std::max(LA, LB);  // viterbi.cpp:42-52
    if (DiagLo > P.R)
        DiagLo -= P.R;
    else
        DiagLo = 1;
    DiagHi += P.R;
    unsigned MaxDiag = LA + LB - 1;
    if (DiagHi > MaxDiag) DiagHi = MaxDiag;

    float OpenA = float(GAP_OPEN_SCORE), ExtA = float(GAP_EXT_SCORE);
    if (Left) OpenA = ExtA = 0;

    std::vector<float> Mb(LB + 3, NEG), Db(LB + 3, NEG);
    float *Mrow = Mb.data() + 1, *Drow = Db.data() + 1;  // Mrow[-1] usable
    const size_t W = (size_t)LB + 1;
    std::vector<byte> TB((size_t)(LA + 1) * W, TB_POISON);
    if (st) st->dp_calls++;

    for (unsigned i = 0; i < LA; ++i) {
        unsigned Startj, Endj;
        RangeJ(LA, LB, DiagLo, DiagHi, i, Startj, Endj);
        if (Endj == 0) continue;
        float OpenB = float((Startj == 0 && Left) ? 0 : GAP_OPEN_SCORE);
        float ExtB = float((Startj == 0 && Left) ? 0 : GAP_EXT_SCORE);
        byte a = A[i];
        float I0 = NEG;
        float M0;
        if (i == 0)
            M0 = 0;
        else
            M0 = (Startj == 0) ? NEG : Mrow[(int)Startj - 1];
        byte *TBrow = &TB[(size_t)i * W];
        if (Startj > 0) TBrow[Startj - 1] = TB_IM;
        if (st) st->dp_cells += Endj - Startj;
        for (unsigned j = Startj; j < Endj; ++j) {
            byte b = B[j];
            byte bits = 0;
            float Saved = M0;
            float xM = M0;
            if (Drow[j] > xM) { xM = Drow[j]; bits = TB_DM; }
            if (I0 > xM) { xM = I0; bits = TB_IM; }
            M0 = Mrow[j];
            Mrow[j] = xM + (a == b ? 1 : MISMATCH_SCORE);
            float md = Saved + OpenB;
            Drow[j] += ExtB;
            if (md >= Drow[j]) { Drow[j] = md; bits |= TB_MD; }
            float mi = Saved + OpenA;
            I0 += ExtA;
            if (mi >= I0) { I0 = mi; bits |= TB_MI; }
            OpenB = float(GAP_OPEN_SCORE);
            ExtB = float(GAP_EXT_SCORE);
            TBrow[j] = bits;
        }
        {  // viterbi.cpp:187-200
            TBrow[LB] = 0;
            float md = M0 + GAP_OPEN_SCORE;
            Drow[LB] += GAP_EXT_SCORE;
            if (md >= Drow[LB]) { Drow[LB] = md; TBrow[LB] = TB_MD; }
        }
        OpenA = float(GAP_OPEN_SCORE);
        ExtA = float(GAP_EXT_SCORE);
    }
    unsigned Startj, Endj;
    RangeJ(LA, LB, DiagLo, DiagHi, LA - 1, Startj, Endj);
    byte *TBrow = &TB[(size_t)LA * W];
    float I1 = NEG;
    Mrow[(int)Startj - 1] = NEG;
    float GapOp = float(GAP_OPEN_SCORE), GapEx = float(GAP_EXT_SCORE);
    if (Right) GapOp = GapEx = 0;
    for (unsigned j = Startj; j < Endj; ++j) {  // viterbi.cpp:222-236
        TBrow[j] = 0;
        float mi = Mrow[(int)j - 1] + GapOp;
        I1 += GapEx;
        if (mi > I1) { I1 = mi; TBrow[j] = TB_MI; }
    }
    float Score = Mrow[LB - 1];
    char State = 'M';
    if (Drow[LB] > Score) { Score = Drow[LB]; State = 'D'; }
    if (I1 > Score) { Score = I1; State = 'I'; }

    // TraceBackBitMem
    size_t i = LA, j = LB;
    std::string rev;
    auto tb = [&](size_t ii, size_t jj) -> byte {
        byte t = TB[ii * W + jj];
        if (t & TB_POISON) {
            if (st) st->tb_poison_reads++;
            t = 0;
        }
        return t;
    };
    for (;;) {
        if (i == 0 && j == 0) break;
        rev.push_back(State);
        byte t;
        if (State == 'M') {
            if (i == 0 || j == 0) break;  // reference asserts
            t = tb(i - 1, j - 1);
            State = (t & TB_DM) ? 'D' : (t & TB_IM) ? 'I' : 'M';
            --i; --j;
        } else if (State == 'D') {
            if (i == 0) break;
            t = tb(i - 1, j);
            State = (t & TB_MD) ? 'M' : 'D';
            --i;
        } else {
            if (j == 0) break;
            t = tb(i, j - 1);
            State = (t & TB_MI) ? 'M' : 'I';
            --j;
        }
    }
    Path.assign(rev.rbegin(), rev.rend());
    return Score;
}

// ---- per-read search state (State1, state1.h / state1.cpp) -----------------------------
struct S1 {
    const uo_index &ix;
    const Params &P;
    uo_stats *st;
    const byte *Q = nullptr;
    unsigned QL = 0;
    std::vector<byte> RC;
    std::vector<uint64> SlotsP, SlotsM;
    std::vector<byte> BlobP, BlobM;
    std::vector<byte> PendP, PendM;  // stored as bytes: state1.h:86-87
    unsigned nPendP = 0, nPendM = 0;
    std::vector<uint32> PosVec;
    std::vector<Hit> Hits;
    std::vector<HSP> HSPs;
    unsigned HitCount = 0, HSPCount = 0;
    int Top = -1;
    int MaxPenalty = -1, BestScore = 0, SecondBestScore = 0, BestHSPScore = 0;
    unsigned Mapq = (unsigned)-1;

    S1(const uo_index &ix_, const Params &P_, uo_stats *st_) : ix(ix_), P(P_), st(st_) {
        PosVec.resize(std::max<uint32>(ix.MaxIx, 1) + 1);
    }

    const byte *Seq(bool Plus) const { return Plus ? Q : RC.data(); }

    void GetBlob(uint64 Slot, byte *dst) {  // ufindex.h:184
        memcpy(dst, ix.Blob + 5 * Slot, 5);
        if (st) st->probes++;
    }
    static uint32 BlobPos(const byte *b) {
        uint32 v;
        memcpy(&v, b + 1, 4);
        return v;
    }
    byte GetTally(uint64 Slot) const { return ix.Blob[5 * Slot]; }
    uint32 GetPos(uint64 Slot) const { return BlobPos(ix.Blob + 5 * Slot); }

    // State1::SetSlotsVec, state1.cpp:396-438
    void SetSlotsVec(const byte *S, unsigned L, uint64 *Slots) const {
        const unsigned W = ix.WordLength;
        uint64 Word = 0;
        byte K = 0;
        for (uint32 p = 0; p < W - 1 && p < L; ++p) {
            byte Letter = g_Letter[S[p]];
            if (Letter == 0xFF) { K = 0; Word = 0; continue; }
            if (K < W) ++K;
            Word = (Word << 2) | Letter;
        }
        for (uint32 p = W - 1; p < L; ++p) {
            byte Letter = g_Letter[S[p]];
            if (Letter == 0xFF) { K = 0; Word = 0; Slots[p - W + 1] = UINT64_MAX; continue; }
            if (K < W) ++K;
            Word = (Word << 2) | Letter;
            Slots[p - W + 1] = (K == W) ? ix.WordToSlot(Word & ix.ShiftMask) : UINT64_MAX;
            if (st) st->slot_hashes++;
        }
    }

    void SetQuery(const byte *q, unsigned L) {
        Q = q;
        QL = L;
        RC.resize(L);
        for (unsigned i = 0; i < L; ++i) RC[L - 1 - i] = g_CompChar[q[i]];  // RevCompSeq, seqinfo.cpp:9
        SlotsP.assign(L, UINT64_MAX);
        SlotsM.assign(L, UINT64_MAX);
        BlobP.assign(5 * (size_t)L, 0);
        BlobM.assign(5 * (size_t)L, 0);
        SetSlotsVec(Q, L, SlotsP.data());
        SetSlotsVec(RC.data(), L, SlotsM.data());
    }

    bool LongPhase = false;   // statistics only: inside phase 5 / pending round 2 (second visit of rows longer than 2)
    // UFIndex::GetRow_Blob, ufindex.cpp:883-943
    unsigned GetRow_Blob(uint64 Slot, const byte *ptrBlob, uint32 *Pv) {
        if (st) st->row_calls++;
        byte T = *ptrBlob;
        if (TallyOther(T)) return 0;
        uint64 Slot2 = Slot;
        uint32 Pos = BlobPos(ptrBlob);
        unsigned K = 0;
        for (;;) {
            if (K > 0) {
                T = GetTally(Slot2);
                Pos = GetPos(Slot2);
                if (st) { st->row_hops++; if (LongPhase) st->row_hops_long++; }
            }
            Pv[K++] = Pos;
            if (K == ix.MaxIx) return K;
            if (T == T_PLUS1 || T == T_BOTH1) return 1;
            if (T == T_END) return K;
            if (T == T_LONG_MINE || T == T_LONG_OTHER) {
                uint32 StepA = Pos & 0xffff, StepB = Pos >> 16;
                uint64 SlotA = (Slot2 + StepA) % ix.SlotCount;
                Slot2 = (SlotA + StepB) % ix.SlotCount;
                Pv[K - 1] = GetPos(SlotA);
                if (st) { st->row_hops++; if (LongPhase) st->row_hops_long++; }
            } else {
                byte Next = T & T_NEXT_MASK;
                Slot2 = (Slot2 + Next) % ix.SlotCount;
            }
        }
    }

    bool OverlapsHit(uint32 DBStartPos) const {  // state1.cpp:230-239 (strand ignored)
        for (unsigned i = 0; i < HitCount; ++i)
            if (DBStartPos / 64 == Hits[i].pos / 64) return true;
        return false;
    }
    unsigned OverlapsHSP(uint32 StartPosQ, uint32 StartPosDB) const {  // state1.cpp:241-252
        int64 Diag = int64(StartPosDB) - int64(StartPosQ);
        for (unsigned i = 0; i < HSPCount; ++i)
            if (Diag == int64(HSPs[i].dbstart) - int64(HSPs[i].qstart)) return i;
        return UINT_MAX;
    }

    // State1::AddHitX, state1.cpp:508-551
    unsigned AddHitX(uint32 StartPosDB, bool Plus, int Score, const std::string &Path) {
        if (Score < 10) return UINT_MAX;
        if (OverlapsHit(StartPosDB)) return UINT_MAX;
        int Pen = int(QL) - Score;
        int MaxPen = Pen - 2 * P.MM;
        if (MaxPen < MaxPenalty) MaxPenalty = MaxPen;
        unsigned HitIndex = HitCount;
        if (Hits.size() < HitCount + 1) Hits.resize(HitCount + 1);
        Hit &H = Hits[HitIndex];
        H.score = Score;
        H.plus = Plus;
        H.pos = StartPosDB;
        H.path = Path;
        if (Score > BestScore) {
            SecondBestScore = BestScore;
            BestScore = Score;
            Top = (int)HitIndex;
        } else if (Score == BestScore)
            SecondBestScore = Score;
        else {
            if (Score < BestScore - SECONDARY_HIT_MAX_DELTA) return UINT_MAX;
            if (Score > SecondBestScore) SecondBestScore = Score;
        }
        ++HitCount;
        return HitIndex;
    }

    // State1::AddHSPX, state1.cpp:553-591
    void AddHSPX(unsigned StartPosQ, uint32 StartPosDB, bool Plus, unsigned Length, int Score) {
        if (Score < BestScore - 4) return;
        unsigned k = OverlapsHSP(StartPosQ, StartPosDB);
        if (k != UINT_MAX) {
            HSP &h = HSPs[k];
            if (Score > h.score) h = HSP{StartPosQ, StartPosDB, Length, Score, Plus, false};
            return;
        }
        if (HSPs.size() < HSPCount + 1) HSPs.resize(HSPCount + 1);
        HSPs[HSPCount++] = HSP{StartPosQ, StartPosDB, Length, Score, Plus, false};
        if (Score > BestHSPScore) BestHSPScore = Score;
    }

    // State1::AddHSPScan, extendscan.cpp:8-49
    unsigned AddHSPScan(unsigned StartPosQ, uint32 StartPosDB, bool Plus, unsigned Length, int Score) {
        unsigned k = OverlapsHSP(StartPosQ, StartPosDB);
        if (k != UINT_MAX) {
            HSP &h = HSPs[k];
            if (Score > h.score) h = HSP{StartPosQ, StartPosDB, Length, Score, Plus, false};
            return k;
        }
        k = HSPCount++;
        if (HSPs.size() < HSPCount) HSPs.resize(HSPCount);
        HSPs[k] = HSP{StartPosQ, StartPosDB, Length, Score, Plus, false};
        if (Score > BestHSPScore) BestHSPScore = Score;
        return k;
    }

    // ExtendPen of a position that came out of GetRow_Blob (statistics only: the compared bytes are also counted
    // separately so that bench.py can attribute algorithmic bytes to the probe and the row kernels).
    bool InRows = false;
    int ExtendPenRow(uint32 SeedPosQ, uint32 SeedPosDB, bool Plus) {
        InRows = true;
        const uint64 c0 = st ? st->compare_bytes : 0;
        int r = ExtendPen(SeedPosQ, SeedPosDB, Plus);
        if (st) st->compare_bytes_rows += st->compare_bytes - c0;
        if (st && LongPhase) st->compare_bytes_rows_long += st->compare_bytes - c0;
        InRows = false;
        return r;
    }

    // State1::ExtendPen, extendpen.cpp:9-95.  +score: new full-length hit; -2: HSP; -1 otherwise.
    int ExtendPen(uint32 SeedPosQ, uint32 SeedPosDB, bool Plus) {
        if (st) st->extend_calls++;
        if (SeedPosDB < SeedPosQ) return -1;
        uint32 DBLo = SeedPosDB - SeedPosQ;
        if (OverlapsHit(DBLo)) return -1;
        const byte *QSeq = Seq(Plus);
        const int W = (int)ix.WordLength;
        const int MinHSPScore = int(P.MIN_HSP_PCT * QL / 100.0);
        int Pen = 0, Score = W, Best = 0;
        int EndPos = int(SeedPosQ) + W - 1;
        for (int qp = EndPos + 1; qp < int(QL); ++qp) {
            if (st) st->compare_bytes++;
            if (QSeq[qp] == ix.T((uint64)DBLo + qp)) {
                ++Score;
                if (Score > Best) { Best = Score; EndPos = qp; }
            } else {
                Pen -= P.MM;
                if (Pen > MaxPenalty) return -1;
                Score += P.MM;
                if (Best - Score > P.XDROP) break;
            }
        }
        int StartPos = int(SeedPosQ);
        for (int qp = StartPos - 1; qp >= 0; --qp) {
            if (st) st->compare_bytes++;
            if (QSeq[qp] == ix.T((uint64)DBLo + qp)) {
                ++Score;
                if (Score > Best) { Best = Score; StartPos = qp; }
            } else {
                Pen -= P.MM;
                if (Pen > MaxPenalty) return -1;
                Score += P.MM;
                if (Best - Score > P.XDROP) break;
            }
        }
        if (StartPos == 0 && EndPos == int(QL) - 1) {
            AddHitX(DBLo, Plus, Best, "");
            return Best;
        }
        if (Best >= MinHSPScore) {
            AddHSPX(unsigned(StartPos), DBLo + unsigned(StartPos), Plus, unsigned(EndPos - StartPos + 1), Best);
            return -2;
        }
        return -1;
    }

    // State1::ExtendScan, extendscan.cpp:51-187
    unsigned ExtendScan(uint32 SeedPosQ, uint32 SeedPosDB, bool Plus) {
        if (st) st->extend_calls++;
        if (SeedPosDB < SeedPosQ) return UINT_MAX;
        uint32 DBLo = SeedPosDB - SeedPosQ;
        const byte *QSeq = Seq(Plus);
        const int W = (int)ix.WordLength;
        const int MinHSPScore = W * 2;
        int Pen = 0, Score = W, Best = 0;
        int EndPos = int(SeedPosQ) + W - 1;
        for (int qp = EndPos + 1; qp < int(QL); ++qp) {
            if (st) st->compare_bytes++;
            if (QSeq[qp] == ix.T((uint64)DBLo + qp)) {
                ++Score;
                if (Score > Best) { Best = Score; EndPos = qp; }
            } else {
                Pen -= P.MM;
                if (Pen > MaxPenalty) return UINT_MAX;
                Score += P.MM;
                if (Best - Score > P.XDROP) break;
            }
        }
        int StartPos = int(SeedPosQ);
        for (int qp = StartPos - 1; qp >= 0; --qp) {
            if (st) st->compare_bytes++;
            if (QSeq[qp] == ix.T((uint64)DBLo + qp)) {
                ++Score;
                if (Score > Best) { Best = Score; StartPos = qp; }
            } else {
                if (Pen > MaxPenalty) return UINT_MAX;  // Pen is NOT incremented here (quirk 5)
                Score += P.MM;
                if (Best - Score > P.XDROP) break;
            }
        }
        if (StartPos == 0 && EndPos == int(QL) - 1) return AddHitX(DBLo, Plus, Best, "");
        if (Best < MinHSPScore) return UINT_MAX;
        unsigned k = AddHSPScan(unsigned(StartPos), DBLo + unsigned(StartPos), Plus,
                                unsigned(EndPos - StartPos + 1), Best);
        if (k == UINT_MAX) return UINT_MAX;
        return AlignHSP(k);
    }

    // State1::AlignHSP, alignhsp.cpp:60-172
    unsigned AlignHSP(unsigned HSPIndex) {
        HSP &h = HSPs[HSPIndex];
        if (h.aligned) return UINT_MAX;
        h.aligned = true;
        int TotalPen = int(h.len) - h.score;
        int TotalScore = h.score;
        if (TotalPen > MaxPenalty) return UINT_MAX;
        const unsigned StartPosQ = h.qstart, StartPosDB = h.dbstart, HSPLength = h.len;
        const bool Plus = h.plus;
        const unsigned TL = ix.SeqDataSize;
        unsigned CombinedTLo = StartPosDB;
        const byte *Qs = Seq(Plus);
        std::string LeftPath, RightPath;
        std::vector<byte> Win;
        if (StartPosQ > 0) {
            if (StartPosDB < StartPosQ) return UINT_MAX;
            unsigned LeftQL = StartPosQ;
            unsigned LeftTHi = StartPosDB - 1;
            unsigned LeftTL = LeftQL + BRN * P.R;
            if (LeftTL >= LeftTHi) return UINT_MAX;
            unsigned LeftTLo = LeftTHi - LeftTL + 1;
            Win.resize(LeftTL);
            for (unsigned i = 0; i < LeftTL; ++i) {
                Win[i] = ix.T((uint64)LeftTLo + i);
                if (Win[i] == '-') return UINT_MAX;
            }
            int LeftScore = (int)Viterbi(P, Qs, LeftQL, Win.data(), LeftTL, true, false, LeftPath, st);
            unsigned LeftICount = TrimLeftIs(LeftPath);
            CombinedTLo = LeftTLo + LeftICount;
            int AllGapScore = P.GO + (LeftQL - 1) * P.GE;
            if (AllGapScore > LeftScore) LeftScore = AllGapScore;
            TotalScore += LeftScore;
            TotalPen += int(LeftQL) - LeftScore;
            if (TotalPen > MaxPenalty) return UINT_MAX;
        }
        const unsigned RightQLo = StartPosQ + HSPLength;
        if (RightQLo < QL) {
            unsigned RightQL = QL - RightQLo;
            unsigned RightTLo = StartPosDB + HSPLength;
            unsigned RightTHi = RightTLo + RightQL + BRN * P.R;
            if (RightTHi >= TL) RightTHi = TL - 1;
            if (RightTHi < RightTLo) return UINT_MAX;  // reference would wrap and crash
            unsigned RightTL = RightTHi - RightTLo + 1;
            Win.resize(RightTL);
            for (unsigned i = 0; i < RightTL; ++i) {
                Win[i] = ix.T((uint64)RightTLo + i);
                if (Win[i] == '-') return UINT_MAX;
            }
            int RightScore = (int)Viterbi(P, Qs + RightQLo, RightQL, Win.data(), RightTL, false, true, RightPath, st);
            TrimRightIs(RightPath);
            int AllGapScore = P.GO + (RightQL - 1) * P.GE;
            if (AllGapScore > RightScore) RightScore = AllGapScore;
            TotalScore += RightScore;
            TotalPen += int(RightQL) - RightScore;
            if (TotalPen > MaxPenalty) return UINT_MAX;
        }
        std::string Path = LeftPath + std::string(HSPLength, 'M') + RightPath;
        return AddHitX(CombinedTLo, Plus, TotalScore, Path);
    }

    // State1::CalcMAPQ6, search1m6.cpp:9-33
    unsigned CalcMAPQ6() const {
        if (HitCount == 0) return 0;
        if (BestScore <= 0) return 0;
        double BestPossible = double(QL);
        double Second = double(SecondBestScore);
        if (Second < BestPossible / 2.0) {
            Second = BestPossible / 2.0;
            if (BestScore <= Second) return 0;
        }
        double Fract = double(BestScore) / BestPossible;
        double Drop = BestScore - Second;
        if (Drop > 40) Drop = 40;
        unsigned mapq = (unsigned)(Drop * Fract * Fract);
        if (mapq > 40) mapq = 40;
        return mapq;
    }

    void ResetSearch() {
        HitCount = 0;
        HSPCount = 0;
        Top = -1;
        BestScore = 0;
        SecondBestScore = 0;
        BestHSPScore = 0;
        Mapq = (unsigned)-1;
        MaxPenalty = P.MAXPEN;
    }

    // State1::Search_Lo, search1m6.cpp:35-277
    void Search_Lo() {
        const unsigned W = ix.WordLength;
        if (QL < W) {  // reference underflows (quirk 9); we report "no hit"
            Mapq = 0;
            return;
        }
        const unsigned QWordCount = QL - (W - 1);
        MaxPenalty = P.MAXPEN;
        const int MinScorePhase1 = int(QL) + P.XP1 * P.MM;
        const int MinScorePhase3 = int(QL) + P.XP3 * P.MM;
        const int MinScorePhase4 = int(QL) + P.XP4 * P.MM;
        const int TermHSPScorePhase3 = (int(QL) * P.TERM3_PCT) / 100;
        BestHSPScore = 0;

        auto probe = [&](uint32 QPos, bool Plus, bool &Done) {
            const uint64 Slot = (Plus ? SlotsP : SlotsM)[QPos];
            byte *Bl = (Plus ? BlobP : BlobM).data() + 5 * QPos;
            if (Slot == UINT64_MAX) { Bl[0] = T_FREE; return; }
            GetBlob(Slot, Bl);
            if (Bl[0] != T_BOTH1) return;
            int Score = ExtendPen(QPos, BlobPos(Bl), Plus);
            if (Score >= MinScorePhase1) { Mapq = CalcMAPQ6(); Done = true; }
        };
        bool Done = false;
        for (uint32 QPos = 0; QPos < QWordCount; QPos += W) {  // phase 1
            probe(QPos, true, Done);
            if (Done) return;
            probe(QPos, false, Done);
            if (Done) return;
        }
        for (uint32 QPos = 0; QPos < QWordCount; ++QPos) {  // phase 2
            if (QPos % W == 0) continue;
            probe(QPos, true, Done);
            if (Done) return;
            probe(QPos, false, Done);
            if (Done) return;
        }
        if (BestHSPScore > TermHSPScorePhase3) {  // phase 3
            for (unsigned i = 0; i < HSPCount; ++i) AlignHSP(i);
            if (BestScore >= MinScorePhase1) { Mapq = CalcMAPQ6(); return; }
        }
        std::vector<uint32> TodoP, TodoM;  // phase 4
        for (int strand = 0; strand < 2; ++strand) {
            const bool Plus = (strand == 0);
            const byte *Bv = (Plus ? BlobP : BlobM).data();
            const uint64 *Sv = (Plus ? SlotsP : SlotsM).data();
            std::vector<uint32> &Todo = Plus ? TodoP : TodoM;
            for (uint32 QPos = 0; QPos < QWordCount; ++QPos) {
                byte T = Bv[5 * QPos];
                if (T == T_FREE || T == T_BOTH1 || TallyOther(T)) continue;
                unsigned RowLength = GetRow_Blob(Sv[QPos], Bv + 5 * QPos, PosVec.data());
                if (RowLength > 2) { Todo.push_back(QPos); continue; }
                for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], Plus);
            }
        }
        if (BestScore >= MinScorePhase3) { Mapq = CalcMAPQ6(); return; }
        LongPhase = true;
        for (int strand = 0; strand < 2; ++strand) {  // phase 5
            const bool Plus = (strand == 0);
            const byte *Bv = (Plus ? BlobP : BlobM).data();
            const uint64 *Sv = (Plus ? SlotsP : SlotsM).data();
            for (uint32 QPos : (Plus ? TodoP : TodoM)) {
                unsigned RowLength = GetRow_Blob(Sv[QPos], Bv + 5 * QPos, PosVec.data());
                for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], Plus);
            }
        }
        LongPhase = false;
        if (BestScore >= MinScorePhase4) { Mapq = CalcMAPQ6(); return; }
        for (unsigned i = 0; i < HSPCount; ++i) AlignHSP(i);  // phase 6
        Mapq = CalcMAPQ6();
    }

    // ---------------- paired-end helpers ----------------
    // State1::InitPE, state1.cpp:95-127
    void InitPE(const byte *q, unsigned L) {
        SetQuery(q, L);
        PendP.assign(L + 1, 0);
        PendM.assign(L + 1, 0);
        nPendP = nPendM = 0;
        ResetSearch();
    }

    // State1::GetFirstBoth1Seed, getseed.cpp:9-54
    unsigned GetFirstBoth1Seed(uint32 &QPos, bool &Plus, uint32 &DBPos) {
        const unsigned QWC = QL - (ix.WordLength - 1);
        for (unsigned k = 0; k < QWC; ++k) {
            QPos = (k * PRIME_STRIDE) % QWC;
            uint64 Slot = SlotsP[QPos];
            if (Slot != UINT64_MAX) {
                byte *Bl = BlobP.data() + 5 * QPos;
                GetBlob(Slot, Bl);
                byte T = Bl[0];
                if (!TallyOther(T)) {
                    if (T != T_BOTH1)
                        PendP[nPendP++] = (byte)QPos;
                    else {
                        DBPos = BlobPos(Bl);
                        Plus = true;
                        return k;
                    }
                }
            }
            Slot = SlotsM[QPos];
            if (Slot == UINT64_MAX) continue;
            byte *Bl = BlobM.data() + 5 * QPos;
            GetBlob(Slot, Bl);
            byte T = Bl[0];
            if (TallyOther(T)) continue;
            if (T != T_BOTH1) { PendM[nPendM++] = (byte)QPos; continue; }
            DBPos = BlobPos(Bl);
            Plus = false;
            return k;
        }
        return UINT_MAX;
    }

    // State1::GetNextBoth1Seed, getseed.cpp:56-138
    unsigned GetNextBoth1Seed(unsigned ak, uint32 &aQPos, bool &Plus, uint32 &DBPos) {
        const unsigned QWC = QL - (ix.WordLength - 1);
        if (Plus) {  // getseed.cpp:64-86: minus strand at the same k (no pending push for non-BOTH1)
            unsigned QPos = (ak * PRIME_STRIDE) % QWC;
            uint64 Slot = SlotsM[QPos];
            if (Slot != UINT64_MAX) {
                byte *Bl = BlobM.data() + 5 * QPos;
                GetBlob(Slot, Bl);
                byte T = Bl[0];
                if (TallyMine(T) && T == T_BOTH1) {
                    uint32 NewDBPos = BlobPos(Bl);
                    if (NewDBPos - QPos != DBPos - aQPos) {
                        DBPos = NewDBPos;
                        aQPos = QPos;
                        Plus = false;
                        return ak;
                    } else
                        PendM[nPendM++] = (byte)QPos;
                }
            }
        }
        for (unsigned k = ak + 1; k < QWC; ++k) {
            unsigned QPos = (k * PRIME_STRIDE) % QWC;
            uint64 Slot = SlotsP[QPos];
            if (Slot != UINT64_MAX) {
                byte *Bl = BlobP.data() + 5 * QPos;
                GetBlob(Slot, Bl);
                byte T = Bl[0];
                if (!TallyOther(T)) {
                    if (T != T_BOTH1)
                        PendP[nPendP++] = (byte)QPos;
                    else {
                        uint32 NewDBPos = BlobPos(Bl);
                        if (NewDBPos - QPos != DBPos - aQPos) {
                            DBPos = NewDBPos;
                            aQPos = QPos;
                            Plus = true;
                            return k;
                        }
                    }
                }
            }
            Slot = SlotsM[QPos];
            if (Slot == UINT64_MAX) continue;
            byte *Bl = BlobM.data() + 5 * QPos;
            GetBlob(Slot, Bl);
            byte T = Bl[0];
            if (TallyOther(T)) continue;
            if (T != T_BOTH1) { PendM[nPendM++] = (byte)QPos; continue; }
            uint32 NewDBPos = BlobPos(Bl);
            if (NewDBPos - QPos == DBPos - aQPos) continue;
            DBPos = NewDBPos;
            aQPos = QPos;
            Plus = false;
            return k;
        }
        return UINT_MAX;
    }

    // State1::SearchPE_Pending, search1pepend.cpp:9-130 (callers always pass k == UINT_MAX)
    void SearchPE_Pending() {
        MaxPenalty = P.MAXPEN;
        const int MinScorePhase1 = int(QL) + P.XP1 * P.MM;
        const int TermHSPScorePhase3 = (int(QL) * P.TERM3_PCT) / 100;
        if (BestScore >= MinScorePhase1) { Mapq = CalcMAPQ6(); return; }
        if (BestHSPScore >= TermHSPScorePhase3) {
            for (unsigned i = 0; i < HSPCount; ++i) AlignHSP(i);
            if (BestScore >= MinScorePhase1) { Mapq = CalcMAPQ6(); return; }
        }
        unsigned nP2 = 0, nM2 = 0;
        for (unsigned i = 0; i < nPendP; ++i) {
            unsigned QPos = PendP[i];
            unsigned RowLength = GetRow_Blob(SlotsP[QPos], BlobP.data() + 5 * QPos, PosVec.data());
            if (RowLength > 2) { PendP[nP2++] = (byte)QPos; continue; }
            for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], true);
        }
        for (unsigned i = 0; i < nPendM; ++i) {
            unsigned QPos = PendM[i];
            unsigned RowLength = GetRow_Blob(SlotsM[QPos], BlobM.data() + 5 * QPos, PosVec.data());
            if (RowLength > 2) { PendM[nM2++] = (byte)QPos; continue; }
            for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], false);
        }
        LongPhase = true;
        for (unsigned i = 0; i < nP2; ++i) {
            unsigned QPos = PendP[i];
            unsigned RowLength = GetRow_Blob(SlotsP[QPos], BlobP.data() + 5 * QPos, PosVec.data());
            for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], true);
        }
        for (unsigned i = 0; i < nM2; ++i) {
            unsigned QPos = PendM[i];
            unsigned RowLength = GetRow_Blob(SlotsM[QPos], BlobM.data() + 5 * QPos, PosVec.data());
            for (unsigned r = 0; r < RowLength; ++r) ExtendPenRow(QPos, PosVec[r], false);
        }
        LongPhase = false;
        int B = std::max(BestScore, BestHSPScore) - 8;
        for (unsigned i = 0; i < HSPCount; ++i) {
            if (HSPs[i].score < B) continue;
            AlignHSP(i);
        }
        Mapq = CalcMAPQ6();
    }

    // State1::ScanSlots, scanslots.cpp:7-62
    void ScanSlots(uint32 DBLo, unsigned DBSegLength, bool Plus) {
        const unsigned W = ix.WordLength;
        const unsigned QWC = QL - (W - 1);
        const uint64 *Sv = (Plus ? SlotsP : SlotsM).data();
        if (QL <= W * 4) return;
        uint64 Word = 0;
        byte K = 0;
        for (uint32 p = 0; p < DBSegLength; ++p) {
            if (st) st->compare_bytes++;
            byte Letter = g_Letter[ix.T((uint64)DBLo + p)];
            if (Letter == 0xFF) { K = 0; Word = 0; continue; }
            if (K < W) ++K;
            Word = (Word << 2) | Letter;
            if (p >= W - 1 && K == W) {
                uint64 Slot = ix.WordToSlot(Word & ix.ShiftMask);
                if (st) st->slot_hashes++;
                for (unsigned k = 0; k < SCANK; ++k) {
                    unsigned QPos = (k * PRIME_STRIDE) % QWC;
                    if (Slot == Sv[QPos]) ExtendScan(QPos, DBLo + p - W + 1, Plus);
                }
            }
        }
    }

    // State1::Scan, scan.cpp:14-39
    void Scan(uint32 DBPos, unsigned DBSegLength, bool Plus, bool DoVit) {
        if (st) st->scan_calls++;
        int SavedMaxPenalty = MaxPenalty;
        unsigned SavedHitCount = HitCount;
        MaxPenalty = 130;
        ScanSlots(DBPos, DBSegLength, Plus);
        MaxPenalty = SavedMaxPenalty;
        if (HitCount > SavedHitCount) return;
        if (!DoVit) return;
        std::vector<byte> Win(DBSegLength);
        for (unsigned i = 0; i < DBSegLength; ++i) Win[i] = ix.T((uint64)DBPos + i);
        std::string Path;
        const uint64 cells0 = st ? st->dp_cells : 0;
        float Score = Viterbi(P, Seq(Plus), QL, Win.data(), DBSegLength, true, true, Path, st);
        if (st) st->dp_cells_scan += st->dp_cells - cells0;
        if (Score >= QL / 3.0) {
            unsigned LeftICount = TrimLeftIs(Path);
            TrimRightIs(Path);
            AddHitX(DBPos + LeftICount, Plus, int(Score), Path);
        }
    }
};

// ---- pair state (State2, state2.h / state2.cpp / search2*.cpp) --------------------------
struct S2 {
    S1 F, R;
    const Params &P;
    std::vector<unsigned> PairF, PairR;
    std::vector<int> PairScore;
    int BestPairScore = 0, SecondBestPairScore = 0;
    unsigned BestPairIndex = 0, SecondPairIndex = UINT_MAX;
    int TermPairScorePhase1 = 0;

    S2(const uo_index &ix, const Params &P_, uo_stats *st) : F(ix, P_, st), R(ix, P_, st), P(P_) {}

    // State2::FindPairs, state2.cpp:20-85
    void FindPairs() {
        PairF.clear(); PairR.clear(); PairScore.clear();
        const unsigned QL2 = (F.QL + R.QL) / 2;
        BestPairIndex = SecondPairIndex = UINT_MAX;
        BestPairScore = SecondBestPairScore = -1;
        for (unsigned hf = 0; hf < F.HitCount; ++hf) {
            const Hit &Hf = F.Hits[hf];
            if (Hf.score < F.SecondBestScore - 12) continue;
            for (unsigned hr = 0; hr < R.HitCount; ++hr) {
                const Hit &Hr = R.Hits[hr];
                if (Hr.score < R.SecondBestScore - 12) continue;
                int64 TL = std::llabs(int64(Hf.pos) - int64(Hr.pos)) + int64(QL2);
                if (TL > 1000) continue;
                if (Hr.plus == Hf.plus) continue;
                int Total = Hf.score + Hr.score;
                if (Total > BestPairScore) {
                    SecondPairIndex = BestPairIndex;
                    SecondBestPairScore = BestPairScore;
                    BestPairScore = Total;
                    BestPairIndex = (unsigned)PairScore.size();
                } else if (Total == BestPairScore) {
                    SecondPairIndex = (unsigned)PairScore.size();
                    SecondBestPairScore = BestPairScore;
                } else if (Total > SecondBestPairScore) {
                    SecondPairIndex = BestPairIndex;
                    SecondBestPairScore = Total;
                }
                PairScore.push_back(Total);
                PairF.push_back(hf);
                PairR.push_back(hr);
            }
        }
    }

    // State2::ScanPair, state2.cpp:87-137 (quirk 6: both QL_* are the forward mate's length)
    void ScanPair() {
        const unsigned HitCountF = F.HitCount, HitCountR = R.HitCount;
        const unsigned SEG = 1024;
        bool DoVitF = (int(F.Mapq) >= 10), DoVitR = (int(R.Mapq) >= 10);
        for (unsigned h = 0; h < HitCountF; ++h) {
            unsigned QLx = F.QL;
            if (F.Hits[h].score < F.SecondBestScore) continue;
            uint32 DBPos = F.Hits[h].pos;
            if (F.Hits[h].plus)
                R.Scan(DBPos, SEG, false, DoVitF);
            else if (DBPos >= SEG)
                R.Scan(DBPos - SEG, SEG + 2 * QLx, true, DoVitF);
        }
        for (unsigned h = 0; h < HitCountR; ++h) {
            unsigned QLx = F.QL;
            if (R.Hits[h].score < R.SecondBestScore) continue;
            uint32 DBPos = R.Hits[h].pos;
            if (R.Hits[h].plus)
                F.Scan(DBPos, SEG, false, DoVitR);
            else if (DBPos >= SEG)
                F.Scan(DBPos - SEG, SEG + 2 * QLx, true, DoVitR);
        }
    }

    // State2::AdjustTopHitsAndMapqs, search2.cpp:8-57
    void AdjustTopHitsAndMapqs() {
        if (PairScore.empty()) {
            F.Mapq /= 2;
            R.Mapq /= 2;
            return;
        }
        unsigned QL = F.QL + R.QL;
        double Fract = double(BestPairScore) / double(QL);
        double Drop = BestPairScore - SecondBestPairScore;
        if (Drop > 30) Drop = 30;
        unsigned mapq = (unsigned)(Drop * Fract * Fract);
        if (mapq > 40) mapq = 40;
        if (mapq > F.Mapq) F.Mapq = mapq;
        if (mapq > R.Mapq) R.Mapq = mapq;
        if (BestPairIndex != UINT_MAX) {
            F.Top = (int)PairF[BestPairIndex];
            R.Top = (int)PairR[BestPairIndex];
        }
    }

    // State2::ExtendBoth1Pair4 / 5, search2m4.cpp:189-208, search2m5.cpp:134-156
    bool ExtendBoth1Pair(uint32 QPosf, uint32 DBPosf, bool Plusf, uint32 QPosr, uint32 DBPosr) {
        int FwdScore = F.ExtendPen(QPosf, DBPosf, Plusf);
        if (FwdScore <= 0) return false;
        int RevScore = R.ExtendPen(QPosr, DBPosr, !Plusf);
        if (RevScore <= 0) return false;
        if (FwdScore + RevScore < TermPairScorePhase1) return false;
        F.Mapq = 40;
        R.Mapq = 40;
        return true;
    }

    // State2::Search4 / Search5, search2m4.cpp:15-187, search2m5.cpp:9-132
    void Search(const byte *q1, unsigned L1, const byte *q2, unsigned L2) {
        F.InitPE(q1, L1);
        R.InitPE(q2, L2);
        const unsigned W = F.ix.WordLength;
        if (L1 < W || L2 < W) {  // reference underflows (quirk 9)
            F.Mapq = R.Mapq = 0;
            return;
        }
        BestPairScore = SecondBestPairScore = 0;
        BestPairIndex = 0;
        SecondPairIndex = UINT_MAX;
        PairF.clear(); PairR.clear(); PairScore.clear();
        const unsigned QLf = L1, QLr = L2, QL2 = (QLf + QLr) / 2;
        TermPairScorePhase1 = int(QLf) + int(QLr) + 5 * P.MM;
        std::vector<uint32> B1Qf, B1Qr, B1Df, B1Dr;
        std::vector<char> B1Pf, B1Pr;
        uint32 QPosf = 0, QPosr = 0, DBPosf = 0, DBPosr = 0;
        bool Plusf = false, Plusr = false;
        unsigned kf = F.GetFirstBoth1Seed(QPosf, Plusf, DBPosf);
        unsigned kr = R.GetFirstBoth1Seed(QPosr, Plusr, DBPosr);
        do {
            if (kf != UINT_MAX) {
                B1Qf.push_back(QPosf); B1Pf.push_back(Plusf); B1Df.push_back(DBPosf);
                for (size_t i = 0; i < B1Dr.size(); ++i) {
                    uint32 dbr = B1Dr[i];
                    int64 TL = std::llabs(int64(DBPosf) - int64(dbr)) + int64(QL2);
                    if (TL <= MAX_TL)
                        if (ExtendBoth1Pair(QPosf, DBPosf, Plusf, B1Qr[i], dbr)) return;
                }
            }
            if (kr != UINT_MAX) {
                B1Qr.push_back(QPosr); B1Pr.push_back(Plusr); B1Dr.push_back(DBPosr);
                for (size_t i = 0; i < B1Df.size(); ++i) {
                    uint32 dbf = B1Df[i];
                    int64 TL = std::llabs(int64(dbf) - int64(DBPosr)) + int64(QL2);
                    if (TL <= MAX_TL)
                        if (ExtendBoth1Pair(B1Qf[i], dbf, !Plusr, QPosr, DBPosr)) return;
                }
            }
            if (kf != UINT_MAX) kf = F.GetNextBoth1Seed(kf, QPosf, Plusf, DBPosf);
            if (kr != UINT_MAX) kr = R.GetNextBoth1Seed(kr, QPosr, Plusr, DBPosr);
        } while (kf != UINT_MAX || kr != UINT_MAX);

        for (size_t i = 0; i < B1Qf.size(); ++i) F.ExtendPen(B1Qf[i], B1Df[i], B1Pf[i] != 0);
        for (size_t i = 0; i < B1Qr.size(); ++i) R.ExtendPen(B1Qr[i], B1Dr[i], B1Pr[i] != 0);

        if (P.pe_method == 5) {  // search2m5.cpp:130-131
            F.SearchPE_Pending();
            R.SearchPE_Pending();
            return;
        }
        int TermF = (QLf * 9) / 10, TermR = (QLr * 9) / 10;  // search2m4.cpp:161-175
        if (F.BestScore >= TermF && R.BestScore >= TermR) {
            int64 TL = std::llabs(int64(F.Hits[F.Top].pos) - int64(R.Hits[R.Top].pos)) + int64(QL2);
            if (TL <= MAX_TL) {
                F.Mapq = 40;
                R.Mapq = 40;
                return;
            }
        }
        F.SearchPE_Pending();
        R.SearchPE_Pending();
        FindPairs();
        if (PairScore.empty()) {
            ScanPair();
            FindPairs();
        }
        AdjustTopHitsAndMapqs();
    }
};

// path string -> RLE runs
void PathToRuns(const std::string &path, std::vector<uint16_t> &runs) {
    size_t i = 0;
    while (i < path.size()) {
        char c = path[i];
        size_t j = i;
        while (j < path.size() && path[j] == c && j - i < 16383) ++j;
        unsigned op = (c == 'M') ? 0 : (c == 'D') ? 1 : 2;
        runs.push_back((uint16_t)(((j - i) << 2) | op));
        i = j;
    }
}

void FillResult(const S1 &s, uo_result &r, std::vector<uint16_t> &runs) {
    memset(&r, 0, sizeof(r));
    r.db_pos = 0xFFFFFFFFu;
    r.best = (int16_t)s.BestScore;
    r.second = (int16_t)s.SecondBestScore;
    r.mapq = (uint8_t)std::min(s.Mapq, 255u);
    r.hit_count = (uint8_t)std::min(s.HitCount, 255u);
    r.hsp_count = (uint8_t)std::min(s.HSPCount, 255u);
    if (s.Top >= 0) {
        const Hit &h = s.Hits[s.Top];
        r.db_pos = h.pos;
        r.score = (int16_t)h.score;
        r.flags = (h.plus ? 1 : 0) | 2;
        runs.clear();
        PathToRuns(h.path, runs);
        r.path_runs = (uint16_t)runs.size();
    } else
        runs.clear();
}

void AddStats(uo_stats *dst, const uo_stats &s) {
    if (!dst) return;
    dst->reads += s.reads; dst->probes += s.probes; dst->row_calls += s.row_calls;
    dst->row_hops += s.row_hops; dst->extend_calls += s.extend_calls;
    dst->compare_bytes += s.compare_bytes; dst->slot_hashes += s.slot_hashes;
    dst->dp_calls += s.dp_calls; dst->dp_cells += s.dp_cells; dst->scan_calls += s.scan_calls;
    dst->tb_poison_reads += s.tb_poison_reads;
    dst->compare_bytes_rows += s.compare_bytes_rows;
    dst->row_hops_long += s.row_hops_long; dst->compare_bytes_rows_long += s.compare_bytes_rows_long;
    dst->dp_cells_scan += s.dp_cells_scan;
}

// ---- CIGAR (cigar.cpp:4-41, 141-199; state1.cpp:717-734) --------------------------------
void RunsToCigar(const uint16_t *runs, unsigned nruns, unsigned QL, std::string &out) {
    out.clear();
    char tmp[32];
    if (nruns == 0) {
        snprintf(tmp, sizeof tmp, "%uM", QL);
        out = tmp;
        return;
    }
    std::vector<char> Ops;
    std::vector<unsigned> Lens;
    for (unsigned i = 0; i < nruns; ++i) {
        unsigned op = runs[i] & 3, len = runs[i] >> 2;
        char c = op == 0 ? 'M' : (op == 1 ? 'I' : 'D');  // D<->I swap, cigar.cpp:22-25
        if (!Ops.empty() && Ops.back() == c)
            Lens.back() += len;
        else {
            Ops.push_back(c);
            Lens.push_back(len);
        }
    }
    const size_t N = Ops.size();
    if (N >= 3) {  // CIGAROpsFixDanglingMs; the second block cannot fire after the first (see DESIGN.md)
        if (Ops[0] == 'M' && Lens[0] <= 2 && Lens[1] > 4 && Ops[2] == 'M') {
            Lens[2] += Lens[0];
            Ops.erase(Ops.begin());
            Lens.erase(Lens.begin());
        } else if (Ops[N - 1] == 'M' && Lens[N - 1] <= 2 && Lens[N - 2] > 4 && Ops[N - 3] == 'M') {
            Lens[N - 3] += Lens[N - 1];
            Ops.pop_back();
            Lens.pop_back();
        }
    }
    for (size_t i = 0; i < Ops.size(); ++i) {
        snprintf(tmp, sizeof tmp, "%u%c", Lens[i], Ops[i]);
        out += tmp;
    }
}

void AppendQName(std::string &o, const byte *Label, unsigned n) {  // setsam.cpp:32-44
    if (n > 2 && Label[n - 2] == '/' && (Label[n - 1] == '1' || Label[n - 1] == '2')) n -= 2;
    for (unsigned i = 0; i < n; ++i) {
        char c = (char)Label[i];
        if (c == ' ' || c == '\t') break;
        o.push_back(c);
    }
}

struct Mapped {
    int seq_index;   // -1 unmapped
    uint32 coord;    // m_MappedTargetPos
};

// State1::SetMappedPos, state1.cpp:129-145
Mapped SetMappedPos(const uo_index &ix, const uo_result &r, unsigned QL) {
    Mapped m{-1, UINT32_MAX};
    if (!(r.flags & 2)) return m;
    unsigned TargetL = 0;
    int si;
    uint32 c = ix.PosToCoordL(r.db_pos, si, TargetL);
    if (c + QL > TargetL) return m;  // uint32 arithmetic as in the reference
    m.seq_index = si;
    m.coord = c;
    return m;
}

void SamUnmapped(std::string &o, uint32 aFlags, const byte *Label, unsigned LabelLen, const byte *Seq,
                 const byte *Qual, unsigned QL) {  // SetSAM_Unmapped, setsam.cpp:12-73
    uint32 Flags = 0x04;
    if (aFlags & 0x01) Flags |= 0x01;
    if (aFlags & 0x40) Flags |= 0x40;
    else if (aFlags & 0x80) Flags |= 0x80;
    if (aFlags & 0x08) Flags |= 0x08;
    else if (aFlags & 0x20) Flags |= 0x20;
    AppendQName(o, Label, LabelLen);
    o.push_back('\t');
    o += std::to_string(Flags);
    o += "\t*\t0\t0\t*\t*\t0\t0\t";
    o.append((const char *)Seq, QL);
    o.push_back('\t');
    if (Qual == nullptr) o.push_back('*');
    else o.append((const char *)Qual, QL);
    o.push_back('\n');
}

// State1::SetSAM, setsam.cpp:75-207
void SamRecord(const uo_index &ix, std::string &o, uint32 Flags, const Mapped &self, const uo_result &r,
               const uint16_t *runs, int MateSeqIndex, uint32 MateTargetPos, int TLEN, const byte *Label,
               unsigned LabelLen, const byte *Seq, const byte *Qual, unsigned QL) {
    if (self.seq_index < 0) {
        SamUnmapped(o, Flags, Label, LabelLen, Seq, Qual, QL);
        return;
    }
    const bool Plus = (r.flags & 1) != 0;
    AppendQName(o, Label, LabelLen);
    o.push_back('\t');
    o += std::to_string(Flags);
    o.push_back('\t');
    o += ix.Labels[self.seq_index];
    o.push_back('\t');
    o += std::to_string(self.coord + 1);
    o.push_back('\t');
    o += std::to_string((unsigned)r.mapq);
    o.push_back('\t');
    std::string cig;
    RunsToCigar(runs + r.path_off, r.path_runs, QL, cig);
    o += cig;
    o.push_back('\t');
    if (MateSeqIndex < 0 || ix.Labels[MateSeqIndex] == "" || ix.Labels[MateSeqIndex] == "*") o.push_back('*');
    else if (MateSeqIndex == self.seq_index || ix.Labels[MateSeqIndex] == ix.Labels[self.seq_index]) o.push_back('=');
    else o += ix.Labels[MateSeqIndex];
    o.push_back('\t');
    if (MateTargetPos == 0 || MateTargetPos == UINT32_MAX) o.push_back('0');
    else o += std::to_string(MateTargetPos + 1);
    o.push_back('\t');
    o += std::to_string(TLEN);
    o.push_back('\t');
    if (Plus) o.append((const char *)Seq, QL);
    else for (unsigned i = 0; i < QL; ++i) o.push_back((char)g_CompChar[Seq[QL - 1 - i]]);
    o.push_back('\t');
    if (Qual == nullptr) o.push_back('*');
    else if (Plus) o.append((const char *)Qual, QL);
    else for (unsigned i = 1; i <= QL; ++i) o.push_back((char)Qual[QL - i]);
    o.push_back('\n');
}

uint32 GetPairedFlags(bool First, bool RevComp, bool MateRevComp, bool MateUnmapped) {  // output2.cpp:18-36
    uint32 Flags = First ? 0x41 : 0x81;
    if (RevComp) Flags |= 0x10;
    if (MateUnmapped) Flags |= 0x08;
    else if (MateRevComp) Flags |= 0x20;
    return Flags;
}

char *ToMalloc(const std::string &s, size_t *len) {
    char *p = (char *)malloc(s.size() + 1);
    memcpy(p, s.data(), s.size());
    p[s.size()] = 0;
    if (len) *len = s.size();
    return p;
}

bool IsPrime64(uint64 n) {
    if (n < 2) return false;
    if (n % 2 == 0) return n == 2;
    for (uint64 d = 3; d * d <= n; d += 2)
        if (n % d == 0) return false;
    return true;
}

}  // namespace

extern "C" {

uo_index *uo_index_open(const char *path) {  // UFIndex::FromFile, ufindexio.cpp:60-115
    int fd = open(path, O_RDONLY);
    if (fd < 0) return nullptr;
    struct stat sb;
    if (fstat(fd, &sb) != 0) { close(fd); return nullptr; }
    byte *m = (byte *)mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) { close(fd); return nullptr; }
    uo_index *ix = new uo_index;
    ix->fd = fd;
    ix->map = m;
    ix->map_len = (size_t)sb.st_size;
    size_t o = 0;
    auto u32 = [&]() { uint32 v; memcpy(&v, m + o, 4); o += 4; return v; };
    auto u64 = [&]() { uint64 v; memcpy(&v, m + o, 8); o += 8; return v; };
    bool ok = (u32() == 0x55464931u);
    ix->WordLength = u32();
    ix->MaxIx = u32();
    ix->SeqDataSize = u32();
    ix->SlotCount = u64();
    uint32 SeqCount = u32();
    for (uint32 i = 0; ok && i < SeqCount; ++i) {
        ix->SeqLengths.push_back(u32());
        ix->Offsets.push_back(u32());
        uint32 n = u32();
        ix->Labels.emplace_back((const char *)m + o, n);
        ix->Labels.back() = std::string(ix->Labels.back().c_str());  // reference builds from a C string
        o += n;
    }
    ok = ok && (u32() == 0x55464932u);
    ix->Blob = m + o;
    o += 5 * (size_t)ix->SlotCount;
    ok = ok && o + 4 <= ix->map_len && (u32() == 0x55464933u);
    ix->SeqData = m + o;
    o += ix->SeqDataSize;
    ok = ok && o + 4 <= ix->map_len && (u32() == 0x55464935u);
    ix->ShiftMask = (ix->WordLength >= 32) ? ~0ULL : ((1ULL << (2 * ix->WordLength)) - 1);
    if (!ok) { uo_index_close(ix); return nullptr; }
    return ix;
}

void uo_index_close(uo_index *ix) {
    if (!ix) return;
    if (ix->map) munmap(ix->map, ix->map_len);
    if (ix->fd >= 0) close(ix->fd);
    delete ix;
}
uint64_t uo_index_slot_count(const uo_index *ix) { return ix->SlotCount; }
uint32_t uo_index_seq_size(const uo_index *ix) { return ix->SeqDataSize; }
uint32_t uo_index_word_length(const uo_index *ix) { return ix->WordLength; }
uint32_t uo_index_max_ix(const uo_index *ix) { return ix->MaxIx; }
uint32_t uo_index_contig_count(const uo_index *ix) { return (uint32_t)ix->Labels.size(); }
const uint8_t *uo_index_blob(const uo_index *ix) { return ix->Blob; }
const uint8_t *uo_index_seq(const uo_index *ix) { return ix->SeqData; }

int uo_map_se(const uo_index *ix, const uo_params *p, const uint8_t *seqs, const uint32_t *offs, uint32_t n,
              uo_result *res, uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used, uo_stats *stats,
              int threads) {
    const Params P = MakeParams(p);
    if (threads < 1) threads = 1;
    std::vector<std::vector<uint16_t>> allruns(n);
    int rc = 0;
#pragma omp parallel num_threads(threads)
    {
        uo_stats lst;
        memset(&lst, 0, sizeof lst);
        S1 s(*ix, P, stats ? &lst : nullptr);
#pragma omp for schedule(dynamic, 256)
        for (int64_t i = 0; i < (int64_t)n; ++i) {
            const unsigned L = offs[i + 1] - offs[i];
            s.SetQuery(seqs + offs[i], L);   // State1::Search, search1.cpp:7-24
            s.ResetSearch();
            s.Search_Lo();
            lst.reads++;
            FillResult(s, res[i], allruns[i]);
        }
#pragma omp critical
        AddStats(stats, lst);
    }
    uint32_t used = 0;
    for (uint32_t i = 0; i < n; ++i) {
        res[i].path_off = used;
        if (used + allruns[i].size() > runs_cap) { rc = -2; res[i].path_runs = 0; continue; }
        if (!allruns[i].empty()) memcpy(runs + used, allruns[i].data(), allruns[i].size() * 2);
        used += (uint32_t)allruns[i].size();
    }
    if (runs_used) *runs_used = used;
    return rc;
}

int uo_map_pe(const uo_index *ix, const uo_params *p, const uint8_t *seqs1, const uint32_t *offs1,
              const uint8_t *seqs2, const uint32_t *offs2, uint32_t n, uo_result *res1, uo_result *res2,
              uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used, uo_stats *stats, int threads) {
    const Params P = MakeParams(p);
    if (threads < 1) threads = 1;
    std::vector<std::vector<uint16_t>> ar1(n), ar2(n);
    int rc = 0;
#pragma omp parallel num_threads(threads)
    {
        uo_stats lst;
        memset(&lst, 0, sizeof lst);
        S2 s(*ix, P, stats ? &lst : nullptr);
#pragma omp for schedule(dynamic, 256)
        for (int64_t i = 0; i < (int64_t)n; ++i) {
            s.Search(seqs1 + offs1[i], offs1[i + 1] - offs1[i], seqs2 + offs2[i], offs2[i + 1] - offs2[i]);
            lst.reads += 2;
            FillResult(s.F, res1[i], ar1[i]);
            FillResult(s.R, res2[i], ar2[i]);
        }
#pragma omp critical
        AddStats(stats, lst);
    }
    uint32_t used = 0;
    for (uint32_t i = 0; i < n; ++i) {
        for (int m = 0; m < 2; ++m) {
            uo_result &r = m ? res2[i] : res1[i];
            std::vector<uint16_t> &a = m ? ar2[i] : ar1[i];
            r.path_off = used;
            if (used + a.size() > runs_cap) { rc = -2; r.path_runs = 0; continue; }
            if (!a.empty()) memcpy(runs + used, a.data(), a.size() * 2);
            used += (uint32_t)a.size();
        }
    }
    if (runs_used) *runs_used = used;
    return rc;
}

char *uo_sam_header(const uo_index *ix, const char *version, const char *cmdline, size_t *len) {
    std::string o;  // State1::WriteSAMHeader, state1.cpp:736-752
    for (size_t i = 0; i < ix->Labels.size(); ++i)
        o += "@SQ\tSN:" + ix->Labels[i] + "\tLN:" + std::to_string(ix->SeqLengths[i]) + "\n";
    o += std::string("@PG\tID:urmap\tPN:urmap\tVN:") + version + "\tCL:" + cmdline + "\n";
    return ToMalloc(o, len);
}

char *uo_sam_se(const uo_index *ix, uint32_t n, const uint8_t *seqs, const uint32_t *offs, const uint8_t *quals,
                const uint8_t *labels, const uint32_t *label_offs, const uo_result *res, const uint16_t *runs,
                size_t *len) {
    std::string o;
    for (uint32_t i = 0; i < n; ++i) {  // State1::Output1, output1.cpp:8-17: SetSAM(0, "*", UINT32_MAX, 0)
        const unsigned QL = offs[i + 1] - offs[i];
        Mapped m = SetMappedPos(*ix, res[i], QL);
        SamRecord(*ix, o, 0, m, res[i], runs, -1, UINT32_MAX, 0, labels + label_offs[i],
                  label_offs[i + 1] - label_offs[i], seqs + offs[i], quals ? quals + offs[i] : nullptr, QL);
    }
    return ToMalloc(o, len);
}

char *uo_sam_pe(const uo_index *ix, uint32_t n, const uint8_t *seqs1, const uint32_t *offs1, const uint8_t *quals1,
                const uint8_t *labels1, const uint32_t *label_offs1, const uint8_t *seqs2, const uint32_t *offs2,
                const uint8_t *quals2, const uint8_t *labels2, const uint32_t *label_offs2, const uo_result *res1,
                const uo_result *res2, const uint16_t *runs, size_t *len) {
    std::string o;
    for (uint32_t i = 0; i < n; ++i) {  // State2::SetSAM2, output2.cpp:71-132
        const unsigned L1 = offs1[i + 1] - offs1[i], L2 = offs2[i + 1] - offs2[i];
        Mapped m1 = SetMappedPos(*ix, res1[i], L1), m2 = SetMappedPos(*ix, res2[i], L2);
        const bool Mapped1 = m1.seq_index >= 0, Mapped2 = m2.seq_index >= 0;
        const bool Has1 = Mapped1, Has2 = Mapped2;  // SetMappedPos clears m_TopHit when unmapped
        const bool Plus1 = Has1 && (res1[i].flags & 1), Plus2 = Has2 && (res2[i].flags & 1);
        const bool StrandsConsistent = Has1 && Has2 && (Plus1 != Plus2);
        int TLEN1 = 0, TLEN2 = 0;
        bool CorrectlyPaired = false;
        if (Mapped1 && Mapped2) {
            if (m1.coord <= m2.coord) {
                TLEN1 = int(m2.coord + L2) - int(m1.coord);
                if (TLEN1 > 0 && TLEN1 < 1000 && StrandsConsistent) CorrectlyPaired = true;
                if (TLEN1 > 1000) TLEN1 = 0;
                TLEN2 = -TLEN1;
            } else {
                TLEN2 = int(m1.coord + L1) - int(m2.coord);
                if (TLEN2 > 0 && TLEN2 < 1000 && StrandsConsistent) CorrectlyPaired = true;
                if (TLEN2 > 1000) TLEN2 = 0;
                TLEN1 = -TLEN2;
            }
        }
        const bool RevComp1 = Mapped1 && !(res1[i].flags & 1), RevComp2 = Mapped2 && !(res2[i].flags & 1);
        uint32 Flags1 = GetPairedFlags(true, RevComp1, RevComp2, !Mapped2);
        uint32 Flags2 = GetPairedFlags(false, RevComp2, RevComp1, !Mapped1);
        if (CorrectlyPaired) { Flags1 |= 0x02; Flags2 |= 0x02; }
        SamRecord(*ix, o, Flags1, m1, res1[i], runs, m2.seq_index, m2.coord, TLEN1, labels1 + label_offs1[i],
                  label_offs1[i + 1] - label_offs1[i], seqs1 + offs1[i], quals1 ? quals1 + offs1[i] : nullptr, L1);
        SamRecord(*ix, o, Flags2, m2, res2[i], runs, m1.seq_index, m1.coord, TLEN2, labels2 + label_offs2[i],
                  label_offs2[i + 1] - label_offs2[i], seqs2 + offs2[i], quals2 ? quals2 + offs2[i] : nullptr, L2);
    }
    return ToMalloc(o, len);
}

void uo_free(void *p) { free(p); }

void uo_slots(const uo_index *ix, const uint8_t *seq, uint32_t L, uint64_t *plus, uint64_t *minus) {
    const uo_params up{6, 4, -1, 10};
    Params P = MakeParams(&up);
    S1 s(*ix, P, nullptr);
    s.SetQuery(seq, L);
    const uint32_t n = L >= ix->WordLength ? L - ix->WordLength + 1 : 0;
    for (uint32_t i = 0; i < n; ++i) { plus[i] = s.SlotsP[i]; minus[i] = s.SlotsM[i]; }
}

void uo_revcomp(const uint8_t *seq, uint32_t L, uint8_t *out) {
    for (uint32_t i = 0; i < L; ++i) out[L - 1 - i] = g_CompChar[seq[i]];
}

float uo_viterbi(const uo_params *p, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB, int left,
                 int right, char *path) {
    Params P = MakeParams(p);
    std::string s;
    float sc = Viterbi(P, A, LA, B, LB, left != 0, right != 0, s, nullptr);
    memcpy(path, s.c_str(), s.size() + 1);
    return sc;
}

float uo_viterbi_ex(const uo_params *p, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB, int left,
                    int right, char *path, uint64_t *tb_poison_reads) {
    Params P = MakeParams(p);
    std::string s;
    uo_stats st{};
    float sc = Viterbi(P, A, LA, B, LB, left != 0, right != 0, s, &st);
    memcpy(path, s.c_str(), s.size() + 1);
    *tb_poison_reads = st.tb_poison_reads;
    return sc;
}

void uo_path_to_cigar(const char *path, uint32_t QL, char *out) {
    std::vector<uint16_t> runs;
    PathToRuns(path, runs);
    std::string c;
    RunsToCigar(runs.data(), (unsigned)runs.size(), QL, c);
    memcpy(out, c.c_str(), c.size() + 1);
}

// Functional comparison of two indexes over the same genome: for every slot the head class
// (none / BOTH1 / PLUS1 / list) and the list of positions GetRow_Blob returns must agree; where overflow
// elements are parked may differ.  Returns the number of differing slots.
uint64_t uo_index_functional_diff(const uo_index *a, const uo_index *b, uint64_t *first_bad) {
    if (a->SlotCount != b->SlotCount || a->SeqDataSize != b->SeqDataSize || a->MaxIx != b->MaxIx) return ~0ull;
    if (memcmp(a->SeqData, b->SeqData, a->SeqDataSize) != 0) return ~0ull;
    Params P = Params{-3, -5, -1, 20, 60, 9, 100, 1, 1, 1, 12, 4};
    S1 sa(*a, P, nullptr), sb(*b, P, nullptr);
    std::vector<uint32> pa(a->MaxIx + 2), pb(b->MaxIx + 2);
    uint64_t bad = 0;
    for (uint64 s = 0; s < a->SlotCount; ++s) {
        const byte *ra = a->Blob + 5 * s, *rb = b->Blob + 5 * s;
        const bool ma = TallyMine(ra[0]), mb = TallyMine(rb[0]);
        bool same = (ma == mb);
        if (same && ma) {
            const int ca = ra[0] == T_BOTH1 ? 2 : (ra[0] == T_PLUS1 ? 1 : 0);
            const int cb = rb[0] == T_BOTH1 ? 2 : (rb[0] == T_PLUS1 ? 1 : 0);
            same = (ca == cb);
            if (same) {
                unsigned na = sa.GetRow_Blob(s, ra, pa.data()), nb = sb.GetRow_Blob(s, rb, pb.data());
                same = (na == nb) && std::equal(pa.begin(), pa.begin() + na, pb.begin());
            }
        }
        if (!same) {
            if (bad == 0 && first_bad) *first_bad = s;
            ++bad;
        }
    }
    return bad;
}

uint64_t uo_get_prime(uint64_t n) {
    // prime.cpp:11 scans primes.h, whose entries are "first prime >= x" for x = 100, then
    // x <- x*100/95 (integer); regenerated here instead of copying the table.
    uint64_t x = 100;
    for (int i = 0; i < 410; ++i) {
        uint64_t pr = x;
        while (!IsPrime64(pr)) ++pr;
        if (pr >= n) return pr;
        x = x * 100 / 95;
    }
    return 0;
}

}  // extern "C"
