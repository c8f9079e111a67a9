// urmb_internal.h -- structures shared by the CUDA kernels and the C-ABI layer.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/urmb.h"

// The kernels are compiled twice: namespace urmb with the capacities every read normally fits into, and namespace urmb_big
// (urmb_big.cu, -DURMB_BIG) with capacities no read of up to URMB_MAX_READ_LEN bases can exceed (2 strands x 233 k-mers x
// MaxIx 32 positions = 14 912 candidates, each at most one hit or one HSP): the reads that overflow the first are mapped
// again by the second (urmb_wait), so that results do not depend on a capacity (the reference's lists grow, state1.cpp:190).
#ifndef URMB_NS
#define URMB_NS urmb
#endif
namespace URMB_NS {

#ifdef URMB_BIG
constexpr int kHitCap = 16384;
constexpr int kHspCap = 16384;
constexpr int kRunCap = 192;
constexpr int kRunPool = 32768;
#else
constexpr int kHitCap = 256;    // hits kept per mate (reference grows without bound, state1.cpp:190)
constexpr int kHspCap = 256;    // HSPs kept per mate
constexpr int kRunCap = 64;     // RLE runs per stored path
constexpr int kRunPool = 2048;  // path runs of all hits of one mate
#endif
constexpr int kMaxLen = URMB_MAX_READ_LEN;
constexpr int kScanSeg = 1024;  // SCAN_DB_SEG_LENGTH, state2.cpp:91
constexpr int kBigCols = kScanSeg + 2 * kMaxLen + 8;   // widest mate-rescue window (+1 column)
constexpr int kBigRows = kMaxLen + 1;

struct DevIndex {
    const uint8_t *blob;   // 5 B/slot AoS exactly as in the UFI file (+URMB_BLOB_PAD)
    const uint8_t *seq;    // upper-case genome, 1 B/base (+URMB_SEQ_PAD zero bytes)
    const uint64_t *seq2;  // derived: genome packed 2 bit/base, base g in word g>>5 at bits 63-2(g&31),62-2(g&31)
    const uint32_t *seqx;  // derived: bit (g&31) of word g>>5 set when byte g is not one of "ACGT" (exact byte path)
    const uint32_t *seqc;  // derived: bit b set when any byte of [1024 b, 1024 (b+1)) is not one of "ACGT" (tiny, cache
                           // resident: windows whose coarse bits are clear never load seqx)
    uint64_t slot_count;
    uint64_t magic;        // floor(2^64 / slot_count) for the Barrett reduction
    uint64_t shift_mask;   // 2^(2W)-1
    uint32_t seq_size;
    uint32_t word_len;
    uint32_t max_ix;
};

// floor(2^64 / p), the multiplier of the Barrett reduction h % p (mod_slots; DevIndex::magic)
inline uint64_t barrett_magic(uint64_t p) { return (uint64_t)((((unsigned __int128)1) << 64) / p); }

struct DevParams {  // State1::SetMethod constants, state1.cpp:147-183
    int MM, GO, GE, MIN_HSP_PCT, TERM3_PCT, XDROP, MAXPEN, XP1, XP3, XP4;
    uint32_t R;
    int pe_method;
    uint32_t flags;   // tuning switches (URMB_FLAGS): bit 5 = do not consult the coarse exception bitmap (seqc); bit 8 = test hook:
                      // every fifth read is treated as over a capacity (exercises the in-stream big-capacity rerun);
                      // bit 9 = no first look in the probe kernel (paired input)
    int rescue_rounds; // mate rescue: rounds of (window scans, batched full-window DPs) before the last round that runs the DPs in
                       // place.  0 by default (URMB_RESCUE_ROUNDS): every kernel of the chain has to wait for room on SMs the
                       // main kernels of the following batches fill, so a short chain finishes a batch sooner (profiles/r06g)
};

struct DevBatch {
    const uint8_t *seqs;   // mate-1 reads then mate-2 reads, concatenated
    const uint32_t *offs;  // n_reads+1 offsets into seqs
    uint32_t n_reads;      // SE: n ; PE: 2n (read n+i is the mate of read i)
    uint32_t n_units;      // reads (SE) or pairs (PE)
    uint32_t qcap;         // padded max word count per read (multiple of 32)
    uint32_t seqcap;       // padded max read length (multiple of 32)
    int paired;
};

struct DevProbe {   // output of the probe+extend kernel, [n_reads][2 strands][qcap]
    uint8_t *tally;
    uint32_t *pos;
    uint32_t *ext;     // BOTH1 slots: packed state-independent result of the gapless extension (EXT_NONE otherwise)
    uint8_t *view;     // [n_reads][view_stride] staged read: packed strands, invalid-letter bits, flags, reverse complement
    uint32_t view_stride;
    uint8_t *done;     // [n_units] or null.  Paired input: 1 = the pair left State2::Search4/5 inside the seed loop on the probe
                       // kernel's first look (result records written there; no probe rows, no staged read exist for it)
};
constexpr uint32_t kViewHdr = 224;   // packed strands (144) + bad bits (72) + flags (4) + pad; then seqcap bytes of rc
inline uint32_t view_stride_for(uint32_t seqcap) { return kViewHdr + seqcap; }

// Device counters of one batch slot (u32 each).  CT_RUNS / CT_OVERFLOW / CT_*_TOTAL live for the whole batch; the
// others are per chunk and are zeroed by the launcher between chunks.
constexpr int kRescueRounds = 6;   // most suspend-at-DP rounds of the mate rescue (DevParams::rescue_rounds of them run; a last round
                                   // finishes what is left in place)
enum {
    CT_RUNS = 0,        // path runs used in DevOut::runs
    CT_OVERFLOW = 1,    // reads that exceeded a per-read capacity
    CT_RESCUE = 2,      // pairs that need mate rescue (whole batch): the first rescue_cap of them own an entry of the rescue pool
    CT_RESCUE_HEAD = 3, // work-queue head of the legacy (search from scratch) mate-rescue kernel
    CT_TODO_TOTAL = 4,  // pairs that went through the staged second pass (whole batch, statistics)
    CT_RESCUE_LEGACY = 5, // pairs queued for the legacy mate-rescue kernel (rescue pool full)
    CT_RESCUE_DPS = 6,  // full-window DPs run by the rescue rounds (statistics)
    CT_OVF_LIST = 7,    // entries of DevOut::ovf_list (reads over a capacity, appended by the fast kernels)
    CT_CHUNK0 = 8,      // first per-chunk counter
    CT_HEAD = 8,        // work-queue head of the first-pass kernel
    CT_TODO = 9,        // pairs of this chunk saved for the staged second pass
    CT_STAGE_A = 10, CT_STAGE_B = 11, CT_STAGE_C = 12, CT_FINISH = 13, CT_STAGE_B2 = 14,   // work-queue heads of the stage kernels
    CT_CHUNK_END = 16,  // [CT_CHUNK0, CT_CHUNK_END) are zeroed by the launcher between chunks
    // mate-rescue rounds (whole batch): round r scans the pairs of list r (round 0: every pool entry) and appends the
    // ones that stop at a full-window DP to list r + 1; the DP kernel of round r works through list r + 1
    CT_RQ_COUNT = 16,                           // [kRescueRounds + 2] entries of list r
    CT_RQ_SCAN = CT_RQ_COUNT + kRescueRounds + 2,   // [kRescueRounds + 2] work-queue heads of the scan kernels
    CT_RQ_DP = CT_RQ_SCAN + kRescueRounds + 2,      // [kRescueRounds + 2] work-queue heads of the DP kernels
    // statistics of the mate rescue (URMB_DEBUG): pairs by number of scan windows at entry (<= 4, <= 16, <= 64, <= 256, more),
    // longest time one pair spent in a scan kernel (clock64 ticks >> 10) and its number of windows
    CT_DBG_WIN = CT_RQ_DP + kRescueRounds + 2,      // [5]
    CT_DBG_MAXT = CT_DBG_WIN + 5,
    CT_DBG_MAXW = CT_DBG_MAXT + 1,
    CT_DBG_OVF = CT_DBG_MAXW + 1,                   // [5] reads over a capacity, by capacity (hits, path runs, run pool, HSPs, path assembly)
    // big-capacity rerun (urmb_big.cu): ovf_list entries already turned into units, units listed so far, first unit and
    // work-queue head of the current pass
    CT_OVF_DONE = CT_DBG_OVF + 5,
    CT_OVF_UNITS = CT_OVF_DONE + 1,
    CT_OVF_BASE = CT_OVF_UNITS + 1,
    CT_OVF_HEAD = CT_OVF_BASE + 1,
    CT_DBG_HSPS = CT_OVF_HEAD + 1,                   // [4] reads by final HSP count: <= 256, <= 512, <= 1024, more (statistics of the big-capacity rerun)
    CT_DBG_MAXHSP = CT_DBG_HSPS + 4,
    CT_FIRST_LOOK = CT_DBG_MAXHSP + 1,               // pairs finished by the probe kernel's first look (statistics)
    CT_COUNT = CT_FIRST_LOOK + 1
};

struct RescueSave;
struct DevOut {
    urmb_result *res;      // [n_reads]
    uint16_t *runs;        // pool
    uint32_t runs_cap;
    uint32_t *counters;    // [CT_COUNT]
    uint32_t *todo;        // [chunk pairs] pairs of the current chunk saved for the staged second pass
    uint32_t *rescue;      // [n_units] pairs for the legacy mate-rescue kernel (State2::ScanPair from scratch)
    urmb_second *second;   // [n_reads] or null: State2's second pair (m_SecondHit, search2.cpp:49-56), zero-filled per launch
    RescueSave *rpool;     // [rescue_cap] saved states of the pairs that need mate rescue (null: legacy kernel only)
    uint32_t rescue_cap;
    uint32_t *rq[2];       // [rescue_cap] each: work lists of the rescue rounds (pool entry indexes), ping-pong
    uint32_t *ovf_list;    // [ovf_cap] reads whose search went over a per-mate capacity (null: not recorded); the big-capacity
    uint32_t ovf_cap;      //           build searches them again (urmb_big.cu)
    uint32_t *ovf_units;   // [ovf_cap] the units (reads / pairs) of ovf_list without duplicates: work list of the rerun kernels
};

struct MateScratch {
    uint32_t hit_pos[kHitCap];
    int16_t hit_score[kHitCap];
    uint8_t hit_plus[kHitCap];
    uint8_t hit_nruns[kHitCap];
    uint16_t hit_roff[kHitCap];     // first run of the hit's path in runs_pool
    uint16_t runs_pool[kRunPool];
    uint32_t hsp_dbstart[kHspCap];
    uint16_t hsp_qstart[kHspCap];
    uint16_t hsp_len[kHspCap];
    int16_t hsp_score[kHspCap];
    uint8_t hsp_flags[kHspCap];   // bit0 plus, bit1 aligned
    uint8_t pend[2][kMaxLen];     // m_QPosPendingVec_{Plus,Minus} (bytes, state1.h:86)
    uint8_t todo[2][kMaxLen];     // phase-5 todo lists (search1m6.cpp:170,205)
};

// Per-mate search state that survives between the stage kernels of the paired-end second pass.
struct MateHdr {
    int32_t HitCount, HSPCount, Top, MaxPenalty, Best, Second, BestHSP, nRuns;
    uint32_t Mapq;
    int32_t nPend[2];
    int32_t overflow;
    int32_t done;      // SearchPE_Pending has finished for this mate (Mapq is final)
    int32_t pad[3];
};
struct MateSave {
    MateHdr h;
    MateScratch s;
};

// Mate rescue (State2::ScanPair, state2.cpp:87-137) continues from the saved states of the pair.  A pair whose next step
// is a full-window Viterbi (State1::Scan, scan.cpp:27) stops there: the DP is a pure function of (read strand, window), so
// it is queued for a kernel that runs all pending DPs of the batch side by side, and the pair resumes in the next round.
struct RescuePos {
    int32_t state;            // 0 fresh, 1 stopped at a DP (request below; the result is filled in by the DP kernel)
    int32_t loop, h;          // position in ScanPair's two loops (h = next hit index)
    int32_t hcF, hcR;         // hit counts at entry
    int32_t dovF, dovR;       // DoVit of the two loops (Mapq >= 10 at entry)
    uint32_t dp_pos, dp_len;  // window of the requested DP
    int32_t dp_plus, dp_mate; // strand of the scanned mate; which mate is scanned (0 = forward read, 1 = reverse read)
};
struct RescueHdr {
    uint32_t unit;            // pair index in the batch
    RescuePos p;
    float dp_score;
    int32_t dp_nrev, dp_ovf;
    uint16_t dp_runs[kRunCap + 8];   // reversed RLE path of the DP
};
struct RescueSave {
    MateSave m[2];
    RescueHdr h;
};

struct WarpScratch {
    MateScratch m[2];
    uint16_t runs_a[kRunCap + 8];   // reversed runs of the current DP
    uint16_t runs_l[kRunCap + 8];   // left-flank path
    uint16_t runs_p[3 * kRunCap + 8]; // assembled path
    float rowM[kBigCols + 8];
    float rowD[kBigCols + 8];
    uint8_t tb[(size_t)kBigRows * kBigCols];   // mate-rescue traceback, 1 B / cell
};

struct LaunchCfg {
    int blocks;
    int warps_per_block;
    size_t smem_bytes;
};

// implemented in urmb_kernels.cu
// o: result records and counters for the first look of paired input (null, or pr.done null: every read is probed in full)
int launch_probe(const DevIndex &ix, const DevParams &P, const DevBatch &b, const DevProbe &pr, void *stream, int sm_count,
                 const struct DevOut *o = nullptr);
// Per-context resources of the search kernels: per-warp scratch and the pool of saved mate states (2 per pair of a chunk).
struct SearchRes {
    WarpScratch *scratch;
    int n_scratch_warps;
    MateSave *pool;
    uint32_t pool_pairs;   // chunk size of the paired-end second pass
};
// Optional hook called before (phase 0) and after (phase 1) every kernel launch of launch_search / launch_rescue with
// the kernel class (URMB_KCLASSES numbering): the API layer records CUDA events there.
struct LaunchTrace {
    void (*mark)(void *user, int klass, int phase);
    void *user;
};
int launch_search(const DevIndex &ix, const DevParams &P, const DevBatch &b, const DevProbe &pr, const DevOut &o,
                  const SearchRes &R, void *stream, int sm_count, int *warps_used, const LaunchTrace *tr);
// Paired-end mate rescue (State2::ScanPair) of the pairs queued by launch_search; may run on another stream (it only
// touches the batch's own buffers and R.scratch).  Returns the number of kernels launched or a negative cudaError.
int launch_rescue(const DevIndex &ix, const DevParams &P, const DevBatch &b, const DevProbe &pr, const DevOut &o,
                  const SearchRes &R, void *stream, int sm_count, const LaunchTrace *tr);
int launch_search_monolithic(const DevIndex &ix, const DevParams &P, const DevBatch &b, const DevProbe &pr, const DevOut &o,
                             const SearchRes &R, void *stream, int sm_count);
int launch_overflow_rerun(const DevIndex &ix, const DevParams &P, const DevBatch &b, const DevProbe &pr, const DevOut &o,
                          const SearchRes &R, void *stream, int sm_count);
int max_search_warps(int sm_count);
// n_bytes = seq_data_size + URMB_SEQ_PAD; seq2 holds n_bytes/32+2 words, seqx n_bytes/32+2 words
size_t packed_words(size_t n_bytes);
// seqc holds coarse_words(n_bytes) words and must be zero-filled before the launch
size_t coarse_words(size_t n_bytes);
int launch_pack_genome(const uint8_t *seq, size_t n_bytes, uint64_t *seq2, uint32_t *seqx, uint32_t *seqc, void *stream);

// implemented in urmb_fasta.cu: FASTA bytes -> SeqData (UfiBuilder::ReadFasta of urmb_host.cpp)
struct FastaTable {
    std::vector<std::string> labels, dropped;   // labels as the file has them (NUL bytes included): kept / dropped records
    std::vector<uint32_t> lengths, offsets;     // kept records: length and offset in SeqData
    std::vector<uint64_t> nstart;               // kept records: kept-byte index of the first byte
    uint64_t seq_size = 0;                      // SeqData bytes
};
// The parse reads whole tiles: the device buffer holds the len raw bytes, then zero bytes up to fasta_padded_len(len).
uint64_t fasta_padded_len(uint64_t len);
// Lines before the first header (at position first) must be empty after '\r' removal: "" or "expected '>' in line N".
std::string fasta_check_head(const uint8_t *fa, uint64_t first);
// Header starts h[0..R] (h[R] = len), their line ends e[0..R) and K[0..R], the kept bytes before each header (K[R]: all of
// them) -> record table; "" or an error message.
std::string fasta_table(const uint8_t *fa, const uint64_t *h, const uint64_t *e, const uint64_t *K, uint64_t R, FastaTable &t);
// Parses d_fa (len raw bytes, padded) on the current device, on stream st.  On success *d_seq is a new buffer with SeqData and
// URMB_SEQ_PAD zero bytes and *kernel_ms the device time of the parse; h_fa: the same bytes on the host (labels, lines before
// the first header).  Errors: URMB_E_IO (bad FASTA, no sequence), URMB_E_UNSUPPORTED (too big), URMB_E_CUDA / URMB_E_NOMEM.
int fasta_parse_device(const uint8_t *d_fa, const uint8_t *h_fa, uint64_t len, void *st, void **d_seq, FastaTable &tab,
                       float *kernel_ms, std::string &err);

}  // namespace URMB_NS
