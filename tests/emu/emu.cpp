// tests/emu/emu.cpp -- DEBUGGING HARNESS, NOT PRODUCT CODE (see tests/emu/cuda_runtime.h).
// Compiles urmap_b200/csrc/urmb_kernels.cu as C++ on top of a lock-step fiber emulation of one warp.
#include "cuda_runtime.h"

#include "../kunit/kunit_cases.cuh"   // urmb_kernels.cu and the single-case runners of tests/kunit
#include "../../urmap_b200/csrc/urmb_build.cu"

emu_dim3 threadIdx, blockIdx, blockDim, gridDim;

namespace emu {

struct Lane {
    ucontext_t ctx;
    char *stack = nullptr;
    bool done = false, waiting = false;
    Kind kind = K_NONE;
    uint64_t value = 0, result = 0;
    int arg = 0, site = 0;
};
static Lane g_lanes[32];
static ucontext_t g_sched;
static int g_cur = 0;
static const std::function<void()> *g_body = nullptr;
static uint8_t *g_smem = nullptr;
static const size_t kStack = 1 << 20;

uint8_t *smem_base() { return g_smem; }

static void lane_entry() {
    (*g_body)();
    g_lanes[g_cur].done = true;
    swapcontext(&g_lanes[g_cur].ctx, &g_sched);
}

uint64_t collective(Kind kind, uint64_t value, int arg, int site) {
    Lane &L = g_lanes[g_cur];
    L.kind = kind;
    L.value = value;
    L.arg = arg;
    L.site = site;
    L.waiting = true;
    swapcontext(&L.ctx, &g_sched);
    return L.result;
}

static void run_warp(int warp) {
    for (int l = 0; l < 32; ++l) {
        Lane &L = g_lanes[l];
        if (!L.stack) L.stack = (char *)malloc(kStack);
        getcontext(&L.ctx);
        L.ctx.uc_stack.ss_sp = L.stack;
        L.ctx.uc_stack.ss_size = kStack;
        L.ctx.uc_link = &g_sched;
        makecontext(&L.ctx, lane_entry, 0);
        L.done = L.waiting = false;
    }
    for (;;) {
        for (int l = 0; l < 32; ++l) {
            Lane &L = g_lanes[l];
            if (L.done || L.waiting) continue;
            g_cur = l;
            threadIdx.x = (unsigned)(warp * 32 + l);
            swapcontext(&g_sched, &L.ctx);
        }
        int ndone = 0;
        for (int l = 0; l < 32; ++l) ndone += g_lanes[l].done;
        if (ndone == 32) return;
        if (ndone != 0) {
            fprintf(stderr, "EMU: %d lanes exited while others wait at a collective (site %d)\n", ndone,
                    g_lanes[0].done ? -1 : g_lanes[0].site);
            abort();
        }
        const Kind k = g_lanes[0].kind;
        const int site = g_lanes[0].site;
        for (int l = 1; l < 32; ++l)
            if (g_lanes[l].kind != k || g_lanes[l].site != site) {
                fprintf(stderr, "EMU: warp divergence at a collective: lane0 kind %d line %d, lane%d kind %d line %d\n", k,
                        site, l, g_lanes[l].kind, g_lanes[l].site);
                abort();
            }
        unsigned bal = 0;
        for (int l = 0; l < 32; ++l)
            if (g_lanes[l].value & 1) bal |= 1u << l;
        for (int l = 0; l < 32; ++l) {
            Lane &L = g_lanes[l];
            switch (k) {
                case K_SHFL: L.result = g_lanes[L.arg & 31].value; break;
                case K_SHFL_UP: L.result = (l - L.arg >= 0) ? g_lanes[l - L.arg].value : L.value; break;
                case K_SHFL_DOWN: L.result = (l + L.arg < 32) ? g_lanes[l + L.arg].value : L.value; break;
                case K_SHFL_XOR: L.result = g_lanes[(l ^ L.arg) & 31].value; break;
                case K_BALLOT: L.result = bal; break;
                case K_ANY: L.result = bal != 0; break;
                default: L.result = 0; break;
            }
            L.waiting = false;
        }
    }
}

void launch(const std::function<void()> &body, int grid, int block, size_t smem) {
    g_body = &body;
    gridDim.x = (unsigned)grid;
    blockDim.x = (unsigned)block;
    std::vector<uint8_t> sm(smem + 64, 0xCD);
    g_smem = sm.data();
    for (int b = 0; b < grid; ++b) {
        blockIdx.x = (unsigned)b;
        for (int w = 0; w < block / 32; ++w) run_warp(w);
    }
    g_smem = nullptr;
}

}  // namespace emu

using namespace urmb;

static DevParams emu_make_params(const urmb_params &p) {  // same table as urmb_api.cu make_params
    uint32_t flags = 0;
    if (const char *f = getenv("URMB_FLAGS")) flags = (uint32_t)strtoul(f, nullptr, 0);
    DevParams P = kunit::params(p.method, p.pe_method, p.band_radius, flags);
    if (const char *f = getenv("URMB_RESCUE_ROUNDS")) P.rescue_rounds = std::min(std::max(atoi(f), 0), (int)kRescueRounds);
    return P;
}

// Optional output of State2's second pair (-tabbedout): set before emu_map, n_reads entries, zero-filled here.
static urmb_second *g_emu_second = nullptr;
static uint32_t g_emu_first_look = 0;   // pairs the probe kernel's first look finished in the last emu_map call
extern "C" uint32_t emu_first_look() { return g_emu_first_look; }
extern "C" void emu_set_second(urmb_second *p) { g_emu_second = p; }

// seqs/offs: n_reads+1 offsets; for paired input read n_units+i is the mate of read i.
extern "C" int emu_map(const uint8_t *blob, const uint8_t *seq_padded, uint32_t seq_size, uint64_t slot_count,
                       uint32_t word_len, uint32_t max_ix, const urmb_params *p, const uint8_t *seqs,
                       const uint32_t *offs, uint32_t n_units, int paired, urmb_result *res, uint16_t *runs,
                       uint32_t runs_cap, uint32_t *counters /*[8]*/) {
    DevIndex ix;
    ix.blob = blob;
    ix.seq = seq_padded;
    ix.slot_count = slot_count;
    ix.magic = barrett_magic(slot_count);
    ix.shift_mask = (word_len >= 32) ? ~0ull : ((1ull << (2 * word_len)) - 1);
    ix.seq_size = seq_size;
    ix.word_len = word_len;
    ix.max_ix = max_ix;
    const size_t nbytes = (size_t)seq_size + 4096, nwords = packed_words(nbytes);
    std::vector<uint64_t> seq2(nwords);
    std::vector<uint32_t> seqx(nwords), seqc(coarse_words(nbytes), 0);
    launch_pack_genome(seq_padded, nbytes, seq2.data(), seqx.data(), seqc.data(), nullptr);
    ix.seq2 = seq2.data();
    ix.seqx = seqx.data();
    ix.seqc = seqc.data();
    DevParams P = emu_make_params(*p);
    const uint32_t nreads = paired ? 2 * n_units : n_units;
    uint32_t maxlen = 0;
    for (uint32_t i = 0; i < nreads; ++i) maxlen = std::max(maxlen, offs[i + 1] - offs[i]);
    if (maxlen > (uint32_t)kMaxLen) return URMB_E_UNSUPPORTED;
    const uint32_t qwc = maxlen >= word_len ? maxlen - word_len + 1 : 1;
    DevBatch b;
    b.seqs = seqs;
    b.offs = offs;
    b.n_reads = nreads;
    b.n_units = n_units;
    b.qcap = (qwc + 31) & ~31u;
    b.seqcap = (std::max(maxlen, 32u) + 31) & ~31u;
    b.paired = paired;
    std::vector<uint8_t> tally((size_t)nreads * 2 * b.qcap);
    std::vector<uint32_t> pos((size_t)nreads * 2 * b.qcap);
    std::vector<uint32_t> ext((size_t)nreads * 2 * b.qcap);
    std::vector<uint8_t> view((size_t)nreads * view_stride_for(b.seqcap) + 64, 0xCD);
    std::vector<uint8_t> done(n_units + 1, 0xCD);
    DevProbe pr{tally.data(), pos.data(), ext.data(), view.data(), view_stride_for(b.seqcap), paired ? done.data() : nullptr};
    uint32_t ct[CT_COUNT];
    memset(ct, 0, sizeof ct);
    std::vector<uint32_t> todo(n_units + 1), rescue(n_units + 1);
    if (g_emu_second) memset(g_emu_second, 0, sizeof(urmb_second) * nreads);
    // a tiny rescue pool: the first pairs that need mate rescue continue from their saved states (rescue rounds), the
    // others take the legacy kernel -- both paths are exercised
    uint32_t rcap = 6;
    if (const char *f = getenv("URMB_EMU_RESCUE_CAP")) rcap = (uint32_t)strtoul(f, nullptr, 0);
    RescueSave *rpool = rcap ? (RescueSave *)malloc(sizeof(RescueSave) * rcap) : nullptr;
    if (rpool) memset(rpool, 0xEE, sizeof(RescueSave) * rcap);
    std::vector<uint32_t> rq0(rcap + 1), rq1(rcap + 1);
    DevOut o{res, runs, runs_cap, ct, todo.data(), rescue.data(), paired ? g_emu_second : nullptr, rpool, rcap, {rq0.data(), rq1.data()}, nullptr, 0u, nullptr};
    const int nw = 4;
    WarpScratch *ws = (WarpScratch *)malloc(sizeof(WarpScratch) * nw);
    memset(ws, 0xEE, sizeof(WarpScratch) * nw);
    // a small odd chunk so that several chunks and a ragged last one are exercised
    uint32_t chunk = 37;
    if (const char *f = getenv("URMB_CHUNK_PAIRS")) chunk = (uint32_t)strtoul(f, nullptr, 0);
    MateSave *pool = (MateSave *)malloc(sizeof(MateSave) * 2 * chunk);
    memset(pool, 0xEE, sizeof(MateSave) * 2 * chunk);
    SearchRes R{ws, nw, pool, chunk};
    launch_probe(ix, P, b, pr, nullptr, 1, &o);
    int nk = launch_search(ix, P, b, pr, o, R, nullptr, 1, nullptr, nullptr);
    if (nk >= 0) nk = launch_rescue(ix, P, b, pr, o, R, nullptr, 1, nullptr);
    free(ws);
    free(pool);
    free(rpool);
    memcpy(counters, ct, 32);
    g_emu_first_look = ct[CT_FIRST_LOOK];
    return nk < 0 ? nk : 0;
}

// One flank DP (State1::Viterbi through flank_viterbi: band across the lanes when it fits) under emulation: score and the
// forward path string ("M", "D", "I" as in the reference).  B must stay readable for 64 bytes past LB.
static void emu_dp_kernel(Env E, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB, bool Left, bool Right, float *score,
                          int *nrev, int *ovf) {
    URMB_DYN_SMEM(smem);
    E.lane_ = (int)(threadIdx.x & 31);
    E.s_win = smem;
    E.s_tb = smem + kMaxLen + 64;
    for (uint32_t k = E.lane_; k < LB && k < (uint32_t)kMaxLen + 64; k += 32) E.s_win[k] = B[k];
    __syncwarp();
    int n = 0, o = 0;
    const float sc = (LB > 512) ? (getenv("EMU_OLD_FULL") ? viterbi_warp<true>(E, A, LA, B, LB, Left, Right, n, o) : viterbi_full(E, A, LA, B, LB, Left, Right, n, o))
                                : flank_viterbi(E, A, LA, 0, LB, Left, Right, n, o);
    if (E.lane_ == 0) { *score = sc; *nrev = n; *ovf = o; }
}
extern "C" float emu_flank_dp(const urmb_params *p, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB, int left, int right,
                              char *path /* LA + LB + 1 */, int *ovf) {
    static WarpScratch *ws = (WarpScratch *)malloc(sizeof(WarpScratch));
    Env E;
    E.P = emu_make_params(*p);
    E.ix = DevIndex{};
    E.ix.seq = B;   // viterbi_warp<true> reads the window from ix.seq + TLo (TLo = 0)
    E.ws = ws;
    E.tb_rows = kMaxLen + 2;
    E.tb_stride = 4 * E.P.R + 6;
    float sc = 0;
    int nrev = 0, o = 0;
    const size_t smem = (size_t)kMaxLen + 64 + (size_t)E.tb_rows * 32 + E.tb_rows + 66 + 64;
    emu::launch([&]() { emu_dp_kernel(E, A, LA, B, LB, left != 0, right != 0, &sc, &nrev, &o); }, 1, 32, smem);
    size_t k = 0;
    for (int r = nrev - 1; r >= 0; --r)
        for (uint32_t t = 0; t < (uint32_t)(ws->runs_a[r] >> 2); ++t) path[k++] = "MDI"[ws->runs_a[r] & 3];
    path[k] = 0;
    if (ovf) *ovf = o;
    return sc;
}

// Device index builder under emulation (scan passes done on the host: they use __syncthreads).
extern "C" int emu_build_index(const uint8_t *seq, uint64_t seq_size, uint64_t slot_count, uint32_t word_len,
                               uint32_t max_ix, uint8_t *blob /* 5*slot_count+16 */, uint64_t *stats) {
    BuildArgs a{};
    a.seq = seq;
    a.seq_size = seq_size;
    a.slot_count = slot_count;
    a.magic = barrett_magic(slot_count);
    a.shift_mask = (word_len >= 32) ? ~0ull : ((1ull << (2 * word_len)) - 1);
    a.word_len = word_len;
    a.max_ix = max_ix;
    a.blob = blob;
    const uint64_t cwords = (slot_count + 3) / 4 + 1;
    std::vector<uint32_t> cntP(cwords, 0), cntM(cwords, 0), fill(cwords, 0), base(slot_count, 0),
        errors(4, 0);
    std::vector<uint64_t> flagged(1u << 16, 0);
    std::vector<uint8_t> qzero(slot_count / 8 + 16, 0);
    a.cntP = cntP.data(); a.cntM = cntM.data(); a.fill = fill.data(); a.base = base.data();
    a.qzero = qzero.data(); a.errors = errors.data();
    a.flagged = flagged.data(); a.flagged_cap = (uint32_t)flagged.size();
    const int T = 256;
    const uint64_t gpos = (seq_size + T - 1) / T, gslot = (slot_count + T - 1) / T;
    emu::launch([&]() { build_init_kernel(a); }, (int)(((slot_count + 3) / 4 + T - 1) / T), T, 0);
    emu::launch([&]() { build_count_kernel(a); }, (int)gpos, T, 0);
    uint64_t run = 0;
    for (uint64_t s = 0; s < slot_count; ++s) {
        base[s] = (uint32_t)run;
        uint32_t n = (cntP[s >> 2] >> ((s & 3) * 8)) & 255u, m = (cntM[s >> 2] >> ((s & 3) * 8)) & 255u;
        run += (n >= 1 && n <= max_ix && m <= max_ix) ? n : 0;
    }
    std::vector<uint32_t> pool(run + 1, 0);
    a.pool = pool.data();
    emu::launch([&]() { build_scatter_kernel(a); }, (int)gpos, T, 0);
    emu::launch([&]() { build_heads_kernel(a); }, (int)gslot, T, 0);
    {   // the carry scan (build_carry_*_kernel use __syncthreads) restated sequentially: two rounds over the ring
        int64_t q = 0;
        for (int round = 0; round < 2; ++round)
            for (uint64_t s = 0; s < slot_count; ++s) {
                const MaxPlus m = mp_slot(a, s);
                const int64_t t = q + m.B;
                q = m.A > t ? m.A : t;
                if (round == 1 && q == 0) qzero[s >> 3] |= (uint8_t)(1u << (s & 7));
            }
    }
    emu::launch([&]() { build_segment_kernel(a); }, (int)gslot, T, 0);
    emu::launch([&]() { build_repair_kernel(a); }, 1, 32, 0);
    if (stats) { stats[0] = run; stats[1] = errors[2]; stats[2] = errors[1]; }
    if (getenv("URMB_BUILD_DEBUG")) fprintf(stderr, "[emu build] %u segment(s) repaired\n", errors[0]);
    return 0;
}
