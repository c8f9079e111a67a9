// tests/kunit/kunit_cases.cuh -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// Runs the kernels' device functions one case at a time: the flank and rescue DPs, the gapless extension, read staging
// and k-mer hashing, the Barrett reduction, the complement table, genome packing and CalcMAPQ6.  The code under test is
// the product source itself (included below), compiled two ways:
//   * by nvcc for sm_100a into tests/kunit/libkunit.so (kunit.cu), and once more with -DURMB_BIG (libkunit_big.so);
//   * by g++ on top of the lock-step warp emulator into tests/emu/libemu.so (emu.cpp).
// The __global__ wrappers run one warp per case (lanes cooperate where the product function is warp-cooperative) and
// walk the cases in a warp-strided loop; the extern "C" entry points below are the same for both builds, only the memory
// calls differ (device memory and copies on the GPU, host memory under the emulator).  tests/kunit/kunit_py.py is the
// Python side; tests/test_kernel_units.py holds the cases and the references.
#ifndef URMB_EMU
#include <cuda_runtime.h>
#endif
#include <stdlib.h>
#include <string.h>

#include "../../urmap_b200/csrc/urmb_kernels.cu"

namespace URMB_NS {
namespace kunit {

// State1::SetMethod constants as urmb_api.cu make_params sets them (method 6 / 7, -map2 -veryfast forces R = 4)
inline DevParams params(int method, int pe_method, int band_radius, uint32_t flags) {
    DevParams P;
    if (method == 7) P = DevParams{-4, -6, -2, 35, 35, 12, 75, 8, 6, 5, 8u, 4, 3u};
    else P = DevParams{-3, -5, -1, 20, 60, 9, 100, 1, 1, 1, 12u, 4, 3u};
    P.pe_method = (pe_method == 5) ? 5 : 4;
    if (band_radius >= 0) P.R = (uint32_t)band_radius;
    else if (pe_method == 5) P.R = 4;
    P.flags = flags;
    P.rescue_rounds = 0;
    return P;
}

// ---- memory of the two builds -------------------------------------------------------------------------------------
#ifdef URMB_EMU
inline void *mem_alloc(size_t n) { return calloc(n ? n : 1, 1); }
inline void mem_free(void *p) { free(p); }
inline void mem_put(void *d, const void *s, size_t n) { if (n) memcpy(d, s, n); }
inline void mem_get(void *d, const void *s, size_t n) { if (n) memcpy(d, s, n); }
inline void mem_zero(void *d, size_t n) { memset(d, 0, n); }
inline int mem_sync() { return 0; }
constexpr int kWarpsPerBlock = 1;
inline int blocks_for(uint32_t) { return 1; }   // the emulator runs one warp after the other: one warp walks every case
#else
inline void *mem_alloc(size_t n) {
    void *p = nullptr;
    return cudaMalloc(&p, n ? n : 1) == cudaSuccess ? p : nullptr;
}
inline void mem_free(void *p) { if (p) cudaFree(p); }
inline void mem_put(void *d, const void *s, size_t n) { if (n) cudaMemcpy(d, s, n, cudaMemcpyHostToDevice); }
inline void mem_get(void *d, const void *s, size_t n) { if (n) cudaMemcpy(d, s, n, cudaMemcpyDeviceToHost); }
inline void mem_zero(void *d, size_t n) { cudaMemset(d, 0, n); }
inline int mem_sync() {
    const cudaError_t e = cudaDeviceSynchronize();
    return e == cudaSuccess ? (int)cudaGetLastError() : (int)e;
}
constexpr int kWarpsPerBlock = 4;
inline int blocks_for(uint32_t n) {   // at most 8 warps per SM of a B200
    const uint32_t b = (n + kWarpsPerBlock - 1) / kWarpsPerBlock;
    return (int)(b < 1 ? 1 : (b > 296 ? 296 : b));
}
#endif

// Device buffers of one call, freed together.
struct Bufs {
    void *p[24];
    int n = 0;
    bool ok = true;
    template <class T> T *alloc(size_t count) {
        void *q = mem_alloc(count * sizeof(T));
        if (!q) ok = false;
        p[n++] = q;
        return (T *)q;
    }
    template <class T> T *put(const T *src, size_t count) {
        T *d = alloc<T>(count);
        if (d) mem_put(d, src, count * sizeof(T));
        return d;
    }
    ~Bufs() {
        for (int i = 0; i < n; ++i) mem_free(p[i]);
    }
};

__device__ __forceinline__ int ku_lane() { return (int)(threadIdx.x & 31u); }
__device__ __forceinline__ uint32_t ku_warp() { return blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); }
__device__ __forceinline__ uint32_t ku_nwarps() { return gridDim.x * (blockDim.x >> 5); }

// ---- flank and rescue DP ------------------------------------------------------------------------------------------
// Shared memory of one warp, laid out as make_env / smem_per_warp lay out the DP area of the search kernels (window of
// seqcap + 64 bytes, trace bits of tb_rows = seqcap + 2 rows of 32 bytes + column LB + row LA), with a guard of kGuard
// canary bytes after each area.  A DP that writes past its area changes a canary and the case reports it.
constexpr uint32_t kGuard = 64;
constexpr uint8_t kCanary = 0xA5;
constexpr uint16_t kRunCanary = 0xBEEF;
__host__ __device__ inline uint32_t dp_win_bytes(uint32_t seqcap) { return seqcap + 64; }
__host__ __device__ inline uint32_t dp_tb_bytes(uint32_t seqcap) { return (seqcap + 2) * 32 + (seqcap + 2) + 66; }
__host__ __device__ inline uint32_t dp_smem_per_warp(uint32_t seqcap) {
    return (dp_win_bytes(seqcap) + kGuard + dp_tb_bytes(seqcap) + kGuard + 15) & ~15u;
}
constexpr int kRunsOut = kRunCap + 8;   // u16 per case in the runs output (WarpScratch::runs_a)

struct DpArgs {
    DevParams P;
    uint32_t seqcap, n;
    int kind;                       // 0: flank_viterbi (band or row-block fallback), 1: viterbi_full (mate rescue)
    const uint8_t *A, *B;           // concatenated; B is readable 64 bytes past each window
    const uint32_t *aoff, *boff;    // n + 1 offsets
    const uint8_t *lr;              // bit 0 Left, bit 1 Right
    WarpScratch *ws;                // one per warp
    float *score;
    int32_t *nrev, *ovf;
    uint16_t *runs;                 // [n][kRunsOut] reversed runs as the DP leaves them in runs_a
    uint32_t *guard;                // bit 0 window guard, bit 1 trace guard, bit 2 runs_a guard changed
};

// One case: the DP as align_hsp (kind 0: window staged in s_win, the fallback reads it from ix.seq + TLo) or scan_mate
// (kind 1: window in global memory) calls it.
__device__ void dp_case(const DpArgs &a, uint32_t c, uint8_t *sw) {
    const int lane = ku_lane();
    const uint32_t wb = dp_win_bytes(a.seqcap), tbb = dp_tb_bytes(a.seqcap);
    uint8_t *win = sw, *g0 = sw + wb, *tb = g0 + kGuard, *g1 = tb + tbb;
    WarpScratch *ws = a.ws + ku_warp();
    // stale contents differ from case to case: a DP that reads what it did not write gives varying answers
    for (uint32_t k = lane; k < wb; k += 32) win[k] = (uint8_t)((k + c) * 0x9Du);
    for (uint32_t k = lane; k < tbb; k += 32) tb[k] = (uint8_t)((k * 0x3Bu + c * 0x71u) >> 1);
    for (uint32_t k = lane; k < kGuard; k += 32) g0[k] = g1[k] = kCanary;
    if (lane < 8) ws->runs_a[kRunCap + lane] = kRunCanary;
    const uint8_t *A = a.A + a.aoff[c], *B = a.B + a.boff[c];
    const uint32_t LA = a.aoff[c + 1] - a.aoff[c], LB = a.boff[c + 1] - a.boff[c];
    const bool Left = a.lr[c] & 1, Right = (a.lr[c] >> 1) & 1;
    Env E;
    E.ix = DevIndex{};
    E.ix.seq = B;   // TLo = 0
    E.P = a.P;
    E.ws = ws;
    E.s_win = win;
    E.s_tb = tb;
    E.tb_stride = 4 * a.P.R + 6;
    E.tb_rows = a.seqcap + 2;
    E.lane_ = lane;
    __syncwarp();
    int nrev = 0, ovf = 0;
    float sc;
    if (a.kind == 0) {
        for (uint32_t k = lane; k < LB && k < wb; k += 32) win[k] = B[k];
        __syncwarp();
        sc = flank_viterbi(E, A, LA, 0, LB, Left, Right, nrev, ovf);
    } else {
        sc = viterbi_full(E, A, LA, B, LB, Left, Right, nrev, ovf);
    }
    __syncwarp();
    bool bad0 = false, bad1 = false;
    for (uint32_t k = lane; k < kGuard; k += 32) { bad0 |= g0[k] != kCanary; bad1 |= g1[k] != kCanary; }
    const bool bad2 = lane < 8 && ws->runs_a[kRunCap + lane] != kRunCanary;
    const uint32_t g = (__any_sync(FULL, bad0) ? 1u : 0u) | (__any_sync(FULL, bad1) ? 2u : 0u) | (__any_sync(FULL, bad2) ? 4u : 0u);
    for (int k = lane; k < kRunsOut; k += 32) a.runs[(size_t)c * kRunsOut + k] = k < nrev ? ws->runs_a[k] : 0;
    if (lane == 0) {
        a.score[c] = sc;
        a.nrev[c] = nrev;
        a.ovf[c] = ovf;
        a.guard[c] = g;
    }
    __syncwarp();
}

__global__ void dp_kernel(const DpArgs a) {
    URMB_DYN_SMEM(smem);
    uint8_t *sw = smem + (size_t)(threadIdx.x >> 5) * dp_smem_per_warp(a.seqcap);
    for (uint32_t c = ku_warp(); c < a.n; c += ku_nwarps()) dp_case(a, c, sw);
}

// ---- read staging, hashing -----------------------------------------------------------------------------------------
__host__ __device__ inline uint32_t read_smem_per_warp(uint32_t seqcap) {
    return ((uint32_t)kReadViewBytes + 2 * seqcap + 15) & ~15u;
}
__device__ ReadView stage(const uint8_t *src, uint32_t L, uint32_t seqcap, uint8_t *sw) {
    uint64_t *s_pk = reinterpret_cast<uint64_t *>(sw);
    uint32_t *s_bad = reinterpret_cast<uint32_t *>(sw + 2 * kPkWords * 8);
    uint8_t *s_q = sw + kReadViewBytes, *s_rc = s_q + seqcap;
    ReadView rv;
    stage_read(ku_lane(), src, L, seqcap, s_q, s_rc, s_pk, s_bad, rv);
    return rv;
}

struct SlotArgs {
    DevIndex ix;
    uint32_t seqcap, n;
    const uint8_t *seqs;
    const uint32_t *offs;       // n + 1
    const uint32_t *outoff;     // n: first output of read r; read r writes 2 (L - W + 1) slots, plus strand first
    uint64_t *slots;
    uint8_t *flags;             // n: bit 0 hasbad, bit 1 slow
};
__global__ void slot_kernel(const SlotArgs a) {
    URMB_DYN_SMEM(smem);
    uint8_t *sw = smem + (size_t)(threadIdx.x >> 5) * read_smem_per_warp(a.seqcap);
    for (uint32_t r = ku_warp(); r < a.n; r += ku_nwarps()) {
        const uint32_t L = a.offs[r + 1] - a.offs[r];
        const ReadView rv = stage(a.seqs + a.offs[r], L, a.seqcap, sw);
        const uint32_t nq = L >= a.ix.word_len ? L - a.ix.word_len + 1 : 0;
        for (uint32_t k = ku_lane(); k < 2 * nq; k += 32)
            a.slots[a.outoff[r] + k] = slot_of(a.ix, rv, k >= nq ? 1 : 0, k >= nq ? k - nq : k);
        if (ku_lane() == 0) a.flags[r] = (rv.hasbad ? 1 : 0) | (rv.slow ? 2 : 0);
        __syncwarp();
    }
}

__global__ void mod_kernel(const uint64_t *h, const uint64_t *p, const uint64_t *magic, uint64_t *r, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        r[i] = mod_slots(h[i], p[i], magic[i]);
}

__global__ void compchar_kernel(uint8_t *out) {
    for (uint32_t c = threadIdx.x; c < 256; c += blockDim.x) out[c] = (uint8_t)compchar_of(c);
}

// ---- gapless extension ---------------------------------------------------------------------------------------------
struct ExtArgs {
    DevIndex ix;
    DevParams P;
    uint32_t seqcap, n;
    const uint8_t *seqs;
    const uint32_t *offs;
    const uint32_t *cs;        // [n][5]: read, plus, SeedPosQ, SeedPosDB, LeftCountsPen
    const int32_t *pen;        // [n] PenBound
    uint32_t *out;             // [n][3]: pure_ext_t<false>, pure_ext_t<true>, pure_ext_bytes
};
__global__ void ext_kernel(const ExtArgs a) {
    URMB_DYN_SMEM(smem);
    uint8_t *sw = smem + (size_t)(threadIdx.x >> 5) * read_smem_per_warp(a.seqcap);
    for (uint32_t c = ku_warp(); c < a.n; c += ku_nwarps()) {
        const uint32_t *cs = a.cs + 5 * (size_t)c;
        const uint32_t r = cs[0], L = a.offs[r + 1] - a.offs[r];
        const ReadView rv = stage(a.seqs + a.offs[r], L, a.seqcap, sw);
        if (ku_lane() == 0) {   // lane-local in the product: one candidate per lane
            const bool Plus = cs[1] != 0, lcp = cs[4] != 0;
            const uint32_t sq = cs[2], sdb = cs[3];
            a.out[3 * (size_t)c + 0] = pure_ext_t<false>(a.ix, a.P, rv, Plus, sq, sdb, lcp, a.pen[c]);
            a.out[3 * (size_t)c + 1] = pure_ext_t<true>(a.ix, a.P, rv, Plus, sq, sdb, lcp, a.pen[c]);
            a.out[3 * (size_t)c + 2] = sdb < sq ? EXT_NONE
                                                : pure_ext_bytes(Plus ? rv.q : rv.rc, a.ix.seq + (sdb - sq), (int)L, (int)a.ix.word_len,
                                                                 a.P.MM, a.P.XDROP, sq, lcp);
        }
        __syncwarp();
    }
}

// ---- CalcMAPQ6 -----------------------------------------------------------------------------------------------------
__global__ void mapq_kernel(const int32_t *in /* [n][4]: QL, Best, Second, HitCount */, uint32_t *out, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Mate m;
        m.QL = (uint32_t)in[4 * (size_t)i];
        m.Best = in[4 * (size_t)i + 1];
        m.Second = in[4 * (size_t)i + 2];
        m.HitCount = in[4 * (size_t)i + 3];
        out[i] = calc_mapq6(m);
    }
}

}  // namespace kunit
}  // namespace URMB_NS

// ---- entry points (tests/kunit/kunit_py.py) ------------------------------------------------------------------------
// Every entry point returns 0 or a CUDA error / -1 for a failed allocation, and frees what it allocated.
namespace ku = URMB_NS::kunit;

extern "C" int ku_run_cap() { return URMB_NS::kRunCap; }

extern "C" int ku_dp(int method, int pe_method, int band_radius, uint32_t seqcap, int kind, uint32_t n, const uint8_t *A,
                     const uint32_t *aoff, const uint8_t *B /* boff[n] + 64 bytes */, const uint32_t *boff, const uint8_t *lr,
                     float *score, int32_t *nrev, int32_t *ovf, uint16_t *runs, uint32_t *guard) {
    using namespace URMB_NS;
    if (n == 0) return 0;
    ku::Bufs m;
    ku::DpArgs a;
    a.P = ku::params(method, pe_method, band_radius, 0);
    a.seqcap = seqcap;
    a.n = n;
    a.kind = kind;
    a.A = m.put(A, aoff[n] + 1);
    a.B = m.put(B, boff[n] + 64);
    a.aoff = m.put(aoff, n + 1);
    a.boff = m.put(boff, n + 1);
    a.lr = m.put(lr, n);
    // one WarpScratch per warp (0.4 MB, 1.2 MB in the big-capacity build): at most 256 MB of them on the device
    int blocks = ku::blocks_for(n);
    const size_t max_blocks = ((size_t)256 << 20) / (sizeof(WarpScratch) * ku::kWarpsPerBlock);
    if ((size_t)blocks > max_blocks) blocks = max_blocks > 0 ? (int)max_blocks : 1;
    const size_t nw = (size_t)blocks * ku::kWarpsPerBlock;
    a.ws = m.alloc<WarpScratch>(nw);
    a.score = m.alloc<float>(n);
    a.nrev = m.alloc<int32_t>(n);
    a.ovf = m.alloc<int32_t>(n);
    a.runs = m.alloc<uint16_t>((size_t)n * ku::kRunsOut);
    a.guard = m.alloc<uint32_t>(n);
    if (!m.ok) return -1;
    const size_t smem = (size_t)ku::kWarpsPerBlock * ku::dp_smem_per_warp(seqcap);
    URMB_LAUNCH(ku::dp_kernel, blocks, 32 * ku::kWarpsPerBlock, smem, nullptr, a);
    int rc = ku::mem_sync();
    if (rc) return rc;
    ku::mem_get(score, a.score, n * sizeof(float));
    ku::mem_get(nrev, a.nrev, n * sizeof(int32_t));
    ku::mem_get(ovf, a.ovf, n * sizeof(int32_t));
    ku::mem_get(runs, a.runs, (size_t)n * ku::kRunsOut * sizeof(uint16_t));
    ku::mem_get(guard, a.guard, n * sizeof(uint32_t));
    return ku::mem_sync();
}

static URMB_NS::DevIndex ku_index(uint64_t slot_count, uint32_t word_len) {
    URMB_NS::DevIndex ix{};
    ix.slot_count = slot_count;
    ix.magic = URMB_NS::barrett_magic(slot_count);
    ix.shift_mask = (word_len >= 32) ? ~0ull : ((1ull << (2 * word_len)) - 1);
    ix.word_len = word_len;
    return ix;
}

// Slots of every k-mer of both strands of n reads: slots[outoff[r] ...] = plus strand then minus strand.
extern "C" int ku_slots(uint64_t slot_count, uint32_t word_len, uint32_t seqcap, uint32_t n, const uint8_t *seqs,
                        const uint32_t *offs, const uint32_t *outoff, uint32_t nout, uint64_t *slots, uint8_t *flags) {
    if (n == 0) return 0;
    ku::Bufs m;
    ku::SlotArgs a;
    a.ix = ku_index(slot_count, word_len);
    a.seqcap = seqcap;
    a.n = n;
    a.seqs = m.put(seqs, offs[n] + 64);
    a.offs = m.put(offs, n + 1);
    a.outoff = m.put(outoff, n);
    a.slots = m.alloc<uint64_t>(nout);
    a.flags = m.alloc<uint8_t>(n);
    if (!m.ok) return -1;
    const int blocks = ku::blocks_for(n);
    URMB_LAUNCH(ku::slot_kernel, blocks, 32 * ku::kWarpsPerBlock, ku::kWarpsPerBlock * ku::read_smem_per_warp(seqcap), nullptr, a);
    int rc = ku::mem_sync();
    if (rc) return rc;
    ku::mem_get(slots, a.slots, nout * sizeof(uint64_t));
    ku::mem_get(flags, a.flags, n);
    return ku::mem_sync();
}

// r[i] = mod_slots(h[i], p[i], barrett_magic(p[i]))
extern "C" int ku_mod(uint32_t n, const uint64_t *h, const uint64_t *p, uint64_t *r) {
    if (n == 0) return 0;
    ku::Bufs m;
    uint64_t *magic = (uint64_t *)malloc(n * sizeof(uint64_t));
    for (uint32_t i = 0; i < n; ++i) magic[i] = URMB_NS::barrett_magic(p[i]);
    const uint64_t *dh = m.put(h, n), *dp = m.put(p, n), *dm = m.put(magic, n);
    free(magic);
    uint64_t *dr = m.alloc<uint64_t>(n);
    if (!m.ok) return -1;
    URMB_LAUNCH(ku::mod_kernel, ku::blocks_for(n / 32 + 1), 32 * ku::kWarpsPerBlock, 0, nullptr, dh, dp, dm, dr, n);
    int rc = ku::mem_sync();
    if (rc) return rc;
    ku::mem_get(r, dr, n * sizeof(uint64_t));
    return ku::mem_sync();
}

extern "C" int ku_compchar(uint8_t *out /* 256 */) {
    ku::Bufs m;
    uint8_t *d = m.alloc<uint8_t>(256);
    if (!m.ok) return -1;
    URMB_LAUNCH(ku::compchar_kernel, 1, 32, 0, nullptr, d);
    int rc = ku::mem_sync();
    if (rc) return rc;
    ku::mem_get(out, d, 256);
    return ku::mem_sync();
}

// pack_genome_kernel (through launch_pack_genome) of n_bytes bytes: seq2 / seqx hold packed_words(n_bytes) words, seqc
// coarse_words(n_bytes) words.
extern "C" size_t ku_packed_words(size_t n_bytes) { return URMB_NS::packed_words(n_bytes); }
extern "C" size_t ku_coarse_words(size_t n_bytes) { return URMB_NS::coarse_words(n_bytes); }
extern "C" int ku_pack(const uint8_t *seq, size_t n_bytes, uint64_t *seq2, uint32_t *seqx, uint32_t *seqc) {
    using namespace URMB_NS;
    ku::Bufs m;
    const size_t nw = packed_words(n_bytes), nc = coarse_words(n_bytes);
    const uint8_t *ds = m.put(seq, n_bytes);
    uint64_t *d2 = m.alloc<uint64_t>(nw);
    uint32_t *dx = m.alloc<uint32_t>(nw), *dc = m.alloc<uint32_t>(nc);
    if (!m.ok) return -1;
    ku::mem_zero(dc, nc * 4);
    int rc = launch_pack_genome(ds, n_bytes, d2, dx, dc, nullptr);
    if (rc) return rc;
    if ((rc = ku::mem_sync())) return rc;
    ku::mem_get(seq2, d2, nw * 8);
    ku::mem_get(seqx, dx, nw * 4);
    ku::mem_get(seqc, dc, nc * 4);
    return ku::mem_sync();
}

// The three gapless extensions of every candidate: genome of seq_size bytes (padded here with URMB_SEQ_PAD zero bytes
// and packed by launch_pack_genome), reads staged by stage_read.
extern "C" int ku_ext(int method, uint32_t flags, uint32_t word_len, const uint8_t *genome, uint32_t seq_size, uint32_t seqcap,
                      uint32_t nreads, const uint8_t *seqs, const uint32_t *offs, uint32_t n, const uint32_t *cs,
                      const int32_t *pen, uint32_t *out) {
    using namespace URMB_NS;
    if (n == 0) return 0;
    ku::Bufs m;
    const size_t nbytes = (size_t)seq_size + URMB_SEQ_PAD, nw = packed_words(nbytes), nc = coarse_words(nbytes);
    uint8_t *dg = m.alloc<uint8_t>(nbytes);
    uint64_t *d2 = m.alloc<uint64_t>(nw);
    uint32_t *dx = m.alloc<uint32_t>(nw), *dc = m.alloc<uint32_t>(nc);
    if (!m.ok) return -1;
    ku::mem_zero(dg, nbytes);
    ku::mem_put(dg, genome, seq_size);
    ku::mem_zero(dc, nc * 4);
    int rc = launch_pack_genome(dg, nbytes, d2, dx, dc, nullptr);
    if (rc) return rc;
    ku::ExtArgs a;
    a.ix = ku_index(2, word_len);
    a.ix.seq = dg;
    a.ix.seq2 = d2;
    a.ix.seqx = dx;
    a.ix.seqc = dc;
    a.ix.seq_size = seq_size;
    a.P = ku::params(method, 4, -1, flags);
    a.seqcap = seqcap;
    a.n = n;
    a.seqs = m.put(seqs, offs[nreads] + 64);
    a.offs = m.put(offs, nreads + 1);
    a.cs = m.put(cs, 5 * (size_t)n);
    a.pen = m.put(pen, n);
    a.out = m.alloc<uint32_t>(3 * (size_t)n);
    if (!m.ok) return -1;
    URMB_LAUNCH(ku::ext_kernel, ku::blocks_for(n), 32 * ku::kWarpsPerBlock, ku::kWarpsPerBlock * ku::read_smem_per_warp(seqcap),
                nullptr, a);
    if ((rc = ku::mem_sync())) return rc;
    ku::mem_get(out, a.out, 3 * (size_t)n * 4);
    return ku::mem_sync();
}

extern "C" int ku_mapq(uint32_t n, const int32_t *in, uint32_t *out) {
    if (n == 0) return 0;
    ku::Bufs m;
    const int32_t *di = m.put(in, 4 * (size_t)n);
    uint32_t *dout = m.alloc<uint32_t>(n);
    if (!m.ok) return -1;
#ifdef URMB_EMU
    const int blocks = 1;
#else
    const int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
#endif
    URMB_LAUNCH(ku::mapq_kernel, blocks, 256, 0, nullptr, di, dout, n);
    int rc = ku::mem_sync();
    if (rc) return rc;
    ku::mem_get(out, dout, n * 4);
    return ku::mem_sync();
}
