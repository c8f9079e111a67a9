// urmb_api.cu -- C-ABI layer (include/urmb.h): UFI loader, per-GPU context, batch slots, streams.
//
// There is deliberately no CPU mapping path here: every urmb_map_* / urmb_submit call runs the CUDA
// kernels or fails with URMB_E_NODEVICE / URMB_E_CUDA.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <mutex>
#include <vector>
#include <string>
#include <thread>
#include <vector>

#include "urmb_internal.h"

using namespace urmb;

// urmb_big.cu: the same kernels with per-mate capacities no read can exceed (reads that overflowed the fast build)
extern "C" size_t urmb_big_scratch_bytes();
extern "C" size_t urmb_big_save_bytes();
extern "C" int urmb_big_rerun_listed(const void *ix, const void *P, const void *batch, const void *probe, const void *out, void *scratch,
                                     int n_scratch_warps, void *stream, int sm_count);
extern "C" int urmb_big_map(const void *ix, const void *P, const void *batch, const void *probe, const void *out, void *scratch,
                            int n_scratch_warps, void *pool, uint32_t pool_pairs, void *stream, int sm_count);

static constexpr uint32_t kOvfCap = 4096;    // reads per batch the in-stream big-capacity rerun takes (more: host path in urmb_wait)
static constexpr int kBigWarps = 256;        // per-warp scratch entries of the big-capacity kernels, per side stream

static std::string g_last_error;
static std::mutex g_err_mu;

static void set_global_error(const std::string &s) {
    std::lock_guard<std::mutex> l(g_err_mu);
    g_last_error = s;
}

// ---------------------------------------------------------------------------------------
// UFI file (ufindexio.cpp:15-49 writer / 60-115 reader). All integers little-endian, no padding.
// ---------------------------------------------------------------------------------------
struct urmb_index_host {
    int fd = -1;
    uint8_t *map = nullptr;
    size_t map_len = 0;
    uint32_t word_length = 0, max_ix = 0, seq_data_size = 0;
    uint64_t slot_count = 0;
    std::vector<std::string> labels;
    std::vector<uint32_t> lengths, offsets;
    const uint8_t *blob = nullptr;
    const uint8_t *seq = nullptr;
    // urmb_index_from_fasta: header only (blob / seq null), the labels of the dropped records and the times of the steps
    std::vector<std::string> dropped;
    double fasta_times[5] = {0, 0, 0, 0, 0};
};

extern "C" int urmb_index_load_host(const char *path, urmb_index_host **out) {
    if (!path || !out) return URMB_E_ARG;
    *out = nullptr;
    int fd = open(path, O_RDONLY);
    if (fd < 0) { set_global_error(std::string("cannot open ") + path); return URMB_E_IO; }
    struct stat sb;
    if (fstat(fd, &sb) != 0 || sb.st_size < 40) { close(fd); set_global_error("UFI file too small"); return URMB_E_IO; }
    uint8_t *m = (uint8_t *)mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) { close(fd); set_global_error("mmap failed"); return URMB_E_IO; }
    urmb_index_host *h = new urmb_index_host;
    h->fd = fd;
    h->map = m;
    h->map_len = (size_t)sb.st_size;
    size_t o = 0;
    bool ok = true;
    auto need = [&](size_t n) { if (o + n > h->map_len) ok = false; return ok; };
    auto u32 = [&]() -> uint32_t { uint32_t v = 0; if (need(4)) { memcpy(&v, m + o, 4); o += 4; } return v; };
    auto u64 = [&]() -> uint64_t { uint64_t v = 0; if (need(8)) { memcpy(&v, m + o, 8); o += 8; } return v; };
    ok = (u32() == 0x55464931u) && ok;  // 'UFI1'
    h->word_length = u32();
    h->max_ix = u32();
    h->seq_data_size = u32();
    h->slot_count = u64();
    uint32_t nseq = u32();
    for (uint32_t i = 0; ok && i < nseq; ++i) {
        h->lengths.push_back(u32());
        h->offsets.push_back(u32());
        uint32_t n = u32();
        if (!need(n)) break;
        std::string lab((const char *)m + o, n);
        h->labels.push_back(std::string(lab.c_str()));  // the reference builds the label from a C string
        o += n;
    }
    ok = ok && (u32() == 0x55464932u);  // 'UFI2'
    h->blob = m + o;
    // header sanity before any size arithmetic (a corrupt slot count must not wrap 5 * slot_count)
    ok = ok && h->word_length >= 1 && h->word_length <= 32 && h->max_ix >= 1 && h->slot_count >= 2 &&
         o <= h->map_len && h->slot_count <= (h->map_len - o) / 5;
    if (ok && need(5 * (size_t)h->slot_count)) o += 5 * (size_t)h->slot_count;
    ok = ok && (u32() == 0x55464933u);  // 'UFI3'
    h->seq = m + o;
    if (ok && need(h->seq_data_size)) o += h->seq_data_size;
    ok = ok && (u32() == 0x55464935u);  // 'UFI5'
    if (!ok) {
        set_global_error(std::string("not a UFI file (bad magic or truncated): ") + path);
        urmb_index_free_host(h);
        return URMB_E_IO;
    }
    *out = h;
    return URMB_OK;
}

extern "C" void urmb_index_free_host(urmb_index_host *h) {
    if (!h) return;
    if (h->map) munmap(h->map, h->map_len);
    if (h->fd >= 0) close(h->fd);
    delete h;
}

extern "C" int urmb_index_info(const urmb_index_host *h, urmb_index_desc *d, uint32_t *n_contigs) {
    if (!h) return URMB_E_ARG;
    if (d) {
        d->word_length = h->word_length;
        d->max_ix = h->max_ix;
        d->seq_data_size = h->seq_data_size;
        d->reserved = 0;
        d->slot_count = h->slot_count;
        d->d_blob = h->blob;
        d->d_seq = h->seq;
    }
    if (n_contigs) *n_contigs = (uint32_t)h->labels.size();
    return URMB_OK;
}

extern "C" int urmb_index_contig(const urmb_index_host *h, uint32_t i, urmb_contig *out) {
    if (!h || !out || i >= h->labels.size()) return URMB_E_ARG;
    out->length = h->lengths[i];
    out->offset = h->offsets[i];
    out->label = h->labels[i].c_str();
    return URMB_OK;
}

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
struct Slot {
    cudaStream_t copy = nullptr;
    cudaEvent_t ev_h2d0 = nullptr, ev_h2d = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_k2 = nullptr, ev_d2h = nullptr;
    cudaEvent_t ev_rescue = nullptr;          // end of the mate-rescue kernel (rescue stream)
    std::vector<cudaEvent_t> kev;             // begin/end events of every kernel of the last launch
    std::vector<int> kclass;                  // kernel class of kev[2i], kev[2i+1]
    size_t nkev = 0;
    // pinned host staging
    uint8_t *h_seqs = nullptr; size_t h_seqs_cap = 0;
    uint32_t *h_offs = nullptr; size_t h_offs_cap = 0;
    urmb_result *h_res = nullptr; size_t h_res_cap = 0;
    urmb_second *d_second = nullptr; size_t d_second_cap = 0;   // only with params.want_second
    urmb_second *h_second = nullptr; size_t h_second_cap = 0;
    uint16_t *h_runs = nullptr; size_t h_runs_cap = 0;
    uint32_t *h_counters = nullptr;
    // device
    uint8_t *d_seqs = nullptr; size_t d_seqs_cap = 0;
    uint32_t *d_offs = nullptr; size_t d_offs_cap = 0;
    uint8_t *d_tally = nullptr; uint32_t *d_pos = nullptr; uint32_t *d_ext = nullptr; size_t d_probe_cap = 0;
    uint8_t *d_view = nullptr; size_t d_view_cap = 0;
    urmb_result *d_res = nullptr; size_t d_res_cap = 0;
    uint16_t *d_runs = nullptr; size_t d_runs_cap = 0;
    uint32_t *d_counters = nullptr;
    uint32_t *d_todo = nullptr; size_t d_todo_cap = 0;
    uint32_t *d_rescue = nullptr; size_t d_rescue_cap = 0;
    uint32_t *d_ovf = nullptr;                // reads over a per-mate capacity (kOvfCap entries), see DevOut::ovf_list
    uint32_t *d_ovf_units = nullptr;          // their units, work list of the rerun (DevOut::ovf_units)
    cudaStream_t big = nullptr;               // high-priority stream of the big-capacity rerun (a handful of blocks that
                                              // must get onto an SM while the persistent main kernels keep them all busy)
    cudaEvent_t ev_big = nullptr, ev_side = nullptr;
    // Mate rescue and big-capacity rerun of this slot's batch run on the slot's own low-priority side stream with their own
    // pool and scratch: the (occasionally long) tail of one batch then delays nothing but that batch's results.
    cudaStream_t side = nullptr;
    RescueSave *rpool = nullptr;              // saved states of the pairs that need mate rescue
    uint32_t *rq[2] = {nullptr, nullptr};     // work lists of the rescue rounds
    size_t rescue_cap = 0;
    WarpScratch *rescue_scratch = nullptr;    // n_rescue_warps entries
    void *big_scratch = nullptr;              // kBigWarps x urmb_big_scratch_bytes()
    DevBatch batch{};
    size_t seq_bytes = 0;
    bool staged = false, launched = false, downloaded = false;
    bool counted = false;             // the batch's overflow / too-long reads went into the context totals
    std::vector<uint32_t> too_long;   // reads of the staged batch that were not searched (longer than URMB_MAX_READ_LEN, or their mate is)
};

struct urmb_ctx {
    int device = 0;
    int sm_count = 0;
    urmb_params params{};
    DevParams P{};
    DevIndex ix{};
    bool have_index = false;
    void *own_blob = nullptr, *own_seq = nullptr;
    uint64_t *seq2 = nullptr;   // derived 2-bit packing of the genome + exception bits (built on the device)
    uint32_t *seqx = nullptr;
    uint32_t *seqc = nullptr;
    cudaStream_t compute = nullptr;
    // Second compute lane (URMB_LANES=2; off by default): consecutive launches alternate between two streams, each with its
    // own per-warp scratch and pool of saved mate states, so that the kernels of two batches can interleave.  Measured:
    // the persistent grids leave no room for each other, 26.6 M against 29.1 M reads/s on the paired-end workload
    // (profiles/r03p), so one lane stays the default.
    cudaStream_t compute2 = nullptr;
    WarpScratch *scratch2 = nullptr;
    MateSave *pool2 = nullptr;
    cudaEvent_t ev_lane = nullptr;
    int lanes = 1, lane_next = 0;
    cudaStream_t rescue = nullptr;            // low-priority side stream of the mate-rescue kernel
    cudaEvent_t ev_mark[2] = {nullptr, nullptr};
    bool rescue_inline = false;               // URMB_RESCUE_INLINE: run the rescue kernel on the compute stream
    WarpScratch *scratch = nullptr;
    int n_scratch_warps = 0;
    int n_rescue_warps = 0;
    MateSave *pool = nullptr;      // saved mate states of one chunk of the paired-end second pass (2 per pair)
    size_t pool_pairs = 0;
    // Resources of the big-capacity rerun (urmb_big.cu), allocated when a batch first needs them
    struct Big {
        static constexpr uint32_t kUnits = 1024;   // units per rerun piece
        static constexpr int kWarps = 256;         // per-warp scratch entries (bounds the grids)
        cudaStream_t stream = nullptr;
        uint8_t *d_seqs = nullptr, *d_tally = nullptr, *d_view = nullptr;
        uint32_t *d_offs = nullptr, *d_pos = nullptr, *d_ext = nullptr, *d_counters = nullptr, *d_todo = nullptr, *d_rescue = nullptr;
        urmb_result *d_res = nullptr, *h_res = nullptr;
        urmb_second *d_second = nullptr, *h_second = nullptr;
        uint16_t *d_runs = nullptr, *h_runs = nullptr;
        uint32_t *h_counters = nullptr, *h_offs = nullptr;
        void *scratch = nullptr, *pool = nullptr;
        size_t seq_cap = 0, probe_cap = 0, view_cap = 0, runs_cap = 0;
        bool ready = false;
    } big;
    int prio_lo = 0;
    bool no_rerun = false;         // URMB_NO_RERUN
    uint64_t rerun_total = 0;      // reads mapped again by the big-capacity build
    uint32_t force_rerun = 0;      // URMB_FORCE_RERUN=N (tests): every N-th unit is mapped again by the big-capacity build
    bool rescue_legacy = false;    // URMB_RESCUE_LEGACY: no rescue pool, every rescued pair is searched again from scratch
    uint32_t chunk_pairs = 1048576; // URMB_CHUNK_PAIRS (step time at 1 M pairs: 65.5 / 61.0 / 60.3 ms for 256k / 512k / 1M, profiles/r03s)
    Slot slots[URMB_SLOTS];
    uint64_t launches = 0;
    uint64_t overflow_total = 0;   // reads that exceeded a per-read capacity, over all finished batches
    uint64_t first_look_total = 0;   // pairs finished by the probe kernel's first look
    uint64_t unsupported_total = 0; // reads not searched because they (or their mates) are longer than URMB_MAX_READ_LEN
    std::string err;
};

static int fail(urmb_ctx *c, int code, const std::string &msg) {
    if (c) c->err = msg;
    set_global_error(msg);
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(c, URMB_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));       \
    } while (0)

static DevParams make_params(const urmb_params &p) {  // State1::SetMethod, state1.cpp:147-183
    DevParams P;
    if (p.method == 7) P = DevParams{-4, -6, -2, 35, 35, 12, 75, 8, 6, 5, 8u, 4, 3u};
    else P = DevParams{-3, -5, -1, 20, 60, 9, 100, 1, 1, 1, 12u, 4, 3u};
    P.pe_method = (p.pe_method == 5) ? 5 : 4;
    if (p.band_radius >= 0) P.R = (uint32_t)p.band_radius;
    else if (p.pe_method == 5) P.R = 4;   // map2.cpp:17-21
    P.flags = 0;       // URMB_FLAGS: see DevParams::flags
    if (const char *f = getenv("URMB_FLAGS")) P.flags = (uint32_t)strtoul(f, nullptr, 0);
    P.rescue_rounds = 0;
    if (const char *f = getenv("URMB_RESCUE_ROUNDS")) P.rescue_rounds = std::min(std::max(atoi(f), 0), (int)kRescueRounds);
    return P;
}

extern "C" const char *urmb_last_error(const urmb_ctx *c) {
    if (c) return c->err.c_str();
    return g_last_error.c_str();
}

static int ctx_init(urmb_ctx *c, int device);
extern "C" int urmb_ctx_create(int device, const urmb_params *p, urmb_ctx **out) {
    if (!out) return URMB_E_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_global_error("no CUDA device available (the mapping engine has no CPU fallback)");
        return URMB_E_NODEVICE;
    }
    if (device < 0 || device >= ndev) { set_global_error("bad device ordinal"); return URMB_E_ARG; }
    urmb_ctx *c = new urmb_ctx;
    c->device = device;
    urmb_params dflt{6, 4, -1, 10, 0};
    c->params = p ? *p : dflt;
    if (c->params.method != 7) c->params.method = 6;
    c->P = make_params(c->params);
    if (c->P.R > 12) { delete c; set_global_error("band radius > 12 unsupported"); return URMB_E_UNSUPPORTED; }
    const int rc = ctx_init(c, device);
    if (rc != URMB_OK) {   // the message is in the global error; streams, events and buffers created so far are released
        urmb_ctx_destroy(c);
        return rc;
    }
    *out = c;
    return URMB_OK;
}

static int ctx_init(urmb_ctx *c, int device) {
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    int prio_lo = 0, prio_hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CK(cudaStreamCreateWithPriority(&c->compute, cudaStreamNonBlocking, prio_hi));
    CK(cudaStreamCreateWithPriority(&c->compute2, cudaStreamNonBlocking, prio_hi));
    CK(cudaEventCreateWithFlags(&c->ev_lane, cudaEventDisableTiming));
    if (const char *f = getenv("URMB_LANES")) c->lanes = atoi(f) == 2 ? 2 : 1;
    CK(cudaStreamCreateWithPriority(&c->rescue, cudaStreamNonBlocking, prio_lo));
    c->prio_lo = prio_lo;
    for (auto &ev : c->ev_mark) CK(cudaEventCreate(&ev));
    if (const char *f = getenv("URMB_RESCUE_LEGACY")) c->rescue_legacy = atoi(f) != 0;
    if (const char *f = getenv("URMB_FORCE_RERUN")) c->force_rerun = (uint32_t)std::max(0, atoi(f));
    c->n_scratch_warps = max_search_warps(c->sm_count);
    // The rescue kernel is a queue of few, long work items that runs beside the next batch: a small persistent grid
    // (one block per SM) takes few registers away from the main kernels and still drains the queue in time.
    c->n_rescue_warps = c->sm_count * 16;   // four resident blocks of the last-round kernel per SM (profiles/r06h)
    if (const char *f = getenv("URMB_RESCUE_WARPS")) c->n_rescue_warps = std::max(4, atoi(f) & ~3);
    if (const char *f = getenv("URMB_RESCUE_INLINE")) c->rescue_inline = atoi(f) != 0;
    if (const char *f = getenv("URMB_CHUNK_PAIRS")) c->chunk_pairs = (uint32_t)std::max(1ul, strtoul(f, nullptr, 0));
    CK(cudaMalloc(&c->scratch, sizeof(WarpScratch) * (size_t)c->n_scratch_warps));
    if (c->lanes == 2) CK(cudaMalloc(&c->scratch2, sizeof(WarpScratch) * (size_t)c->n_scratch_warps));
    c->no_rerun = getenv("URMB_NO_RERUN") != nullptr;
    for (auto &s : c->slots) {
        CK(cudaStreamCreateWithFlags(&s.copy, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithPriority(&s.side, cudaStreamNonBlocking, getenv("URMB_RESCUE_PRIO_HI") ? prio_hi : prio_lo));
        for (cudaEvent_t *ev : {&s.ev_h2d0, &s.ev_h2d, &s.ev_k0, &s.ev_k1, &s.ev_k2, &s.ev_d2h, &s.ev_rescue}) CK(cudaEventCreate(ev));
        CK(cudaMalloc(&s.d_counters, CT_COUNT * sizeof(uint32_t)));
        CK(cudaMalloc(&s.d_ovf, kOvfCap * sizeof(uint32_t)));
        CK(cudaMalloc(&s.d_ovf_units, kOvfCap * sizeof(uint32_t)));
        CK(cudaStreamCreateWithPriority(&s.big, cudaStreamNonBlocking, prio_hi));
        CK(cudaEventCreateWithFlags(&s.ev_big, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&s.ev_side, cudaEventDisableTiming));
        CK(cudaHostAlloc(&s.h_counters, CT_COUNT * sizeof(uint32_t), cudaHostAllocDefault));
    }
    return URMB_OK;
}

static void free_slot(Slot &s) {
    if (s.copy) cudaStreamDestroy(s.copy);
    if (s.side) cudaStreamDestroy(s.side);
    if (s.big) cudaStreamDestroy(s.big);
    if (s.ev_big) cudaEventDestroy(s.ev_big);
    if (s.ev_side) cudaEventDestroy(s.ev_side);
    cudaFree(s.d_ovf_units);
    cudaFree(s.rpool); cudaFree(s.rq[0]); cudaFree(s.rq[1]); cudaFree(s.rescue_scratch); cudaFree(s.big_scratch);
    for (cudaEvent_t ev : {s.ev_h2d0, s.ev_h2d, s.ev_k0, s.ev_k1, s.ev_k2, s.ev_d2h, s.ev_rescue}) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : s.kev) cudaEventDestroy(ev);
    cudaFreeHost(s.h_seqs); cudaFreeHost(s.h_offs); cudaFreeHost(s.h_res); cudaFreeHost(s.h_runs); cudaFreeHost(s.h_counters);
    cudaFree(s.d_seqs); cudaFree(s.d_offs); cudaFree(s.d_tally); cudaFree(s.d_pos); cudaFree(s.d_ext); cudaFree(s.d_view);
    cudaFree(s.d_second); cudaFreeHost(s.h_second);
    cudaFree(s.d_res); cudaFree(s.d_runs); cudaFree(s.d_counters); cudaFree(s.d_todo); cudaFree(s.d_rescue); cudaFree(s.d_ovf);
}

extern "C" void urmb_ctx_destroy(urmb_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto &s : c->slots) free_slot(s);
    if (c->compute) cudaStreamDestroy(c->compute);
    if (c->compute2) cudaStreamDestroy(c->compute2);
    if (c->ev_lane) cudaEventDestroy(c->ev_lane);
    cudaFree(c->scratch2);
    cudaFree(c->pool2);
    if (c->rescue) cudaStreamDestroy(c->rescue);
    for (auto ev : c->ev_mark) if (ev) cudaEventDestroy(ev);
    cudaFree(c->scratch);
    cudaFree(c->pool);
    {
        urmb_ctx::Big &g = c->big;
        if (g.stream) cudaStreamDestroy(g.stream);
        cudaFree(g.d_seqs); cudaFree(g.d_tally); cudaFree(g.d_view); cudaFree(g.d_offs); cudaFree(g.d_pos); cudaFree(g.d_ext);
        cudaFree(g.d_counters); cudaFree(g.d_todo); cudaFree(g.d_rescue); cudaFree(g.d_res); cudaFree(g.d_second); cudaFree(g.d_runs);
        cudaFree(g.scratch); cudaFree(g.pool);
        cudaFreeHost(g.h_res); cudaFreeHost(g.h_second); cudaFreeHost(g.h_runs); cudaFreeHost(g.h_counters); cudaFreeHost(g.h_offs);
    }
    cudaFree(c->own_blob);
    cudaFree(c->own_seq);
    cudaFree(c->seq2);
    cudaFree(c->seqx);
    cudaFree(c->seqc);
    delete c;
}

static int set_index(urmb_ctx *c, const urmb_index_desc *d) {
    if (d->word_length < 8 || d->word_length > 32) return fail(c, URMB_E_UNSUPPORTED, "word length must be in [8,32]");
    if (d->max_ix < 1 || d->max_ix > URMB_MAX_IX) return fail(c, URMB_E_UNSUPPORTED, "max_ix must be in [1,1024]");
    if (d->slot_count < 2 || d->slot_count >= (1ull << 62)) return fail(c, URMB_E_ARG, "bad slot count");
    c->ix.blob = (const uint8_t *)d->d_blob;
    c->ix.seq = (const uint8_t *)d->d_seq;
    c->ix.slot_count = d->slot_count;
    c->ix.magic = barrett_magic(d->slot_count);
    c->ix.shift_mask = (d->word_length >= 32) ? ~0ull : ((1ull << (2 * d->word_length)) - 1);
    c->ix.seq_size = d->seq_data_size;
    c->ix.word_len = d->word_length;
    c->ix.max_ix = d->max_ix;
    // derived data: 2-bit packed genome + exception bits for the lane-local extension (not part of the UFI format)
    CK(cudaSetDevice(c->device));
    cudaFree(c->seq2);
    cudaFree(c->seqx);
    cudaFree(c->seqc);
    c->seq2 = nullptr;
    c->seqx = nullptr;
    c->seqc = nullptr;
    const size_t nbytes = (size_t)d->seq_data_size + URMB_SEQ_PAD, nwords = packed_words(nbytes);
    CK(cudaMalloc(&c->seq2, nwords * 8));
    CK(cudaMalloc(&c->seqx, nwords * 4));
    CK(cudaMalloc(&c->seqc, coarse_words(nbytes) * 4));
    CK(cudaMemsetAsync(c->seqc, 0, coarse_words(nbytes) * 4, c->compute));
    int e = launch_pack_genome(c->ix.seq, nbytes, c->seq2, c->seqx, c->seqc, c->compute);
    if (e) return fail(c, URMB_E_CUDA, std::string("pack launch: ") + cudaGetErrorString((cudaError_t)e));
    CK(cudaStreamSynchronize(c->compute));
    c->ix.seq2 = c->seq2;
    c->ix.seqx = c->seqx;
    c->ix.seqc = c->seqc;
    c->launches += 1;
    c->have_index = true;
    return URMB_OK;
}

extern "C" int urmb_index_attach(urmb_ctx *c, const urmb_index_desc *d) {
    if (!c || !d || !d->d_blob || !d->d_seq) return URMB_E_ARG;
    return set_index(c, d);
}

extern "C" int urmb_index_device_desc(const urmb_ctx *c, urmb_index_desc *out) {
    if (!c || !out || !c->have_index) return URMB_E_ARG;
    out->word_length = c->ix.word_len;
    out->max_ix = c->ix.max_ix;
    out->seq_data_size = c->ix.seq_size;
    out->reserved = 0;
    out->slot_count = c->ix.slot_count;
    out->d_blob = c->ix.blob;
    out->d_seq = c->ix.seq;
    return URMB_OK;
}

// Host (mapped file) -> device(s) through two page-locked staging buffers; the staging copy, which also takes the page
// faults of the mapping, is what bounds the load, so several threads share each chunk.  With more than one destination
// the chunk goes to the first GPU over PCIe and from there to every other GPU over NVLink (peer copies on the other GPUs'
// streams, all in flight together: through NVSwitch each runs at full link rate), pipelined chunk by chunk behind the
// upload -- the index reaches all GPUs in the time one GPU needs.
struct Fanout {
    int n = 0;
    urmb_ctx **ctxs = nullptr;
    std::vector<void *> dst;            // destination base per GPU
    std::vector<cudaStream_t> streams;  // [1..n): copy streams of the peers
};
static int upload_region(urmb_ctx *c, void *dst, const uint8_t *src, size_t n, const Fanout *fan = nullptr) {
    const size_t CH = 128u << 20;
    unsigned nt = std::thread::hardware_concurrency();
    nt = nt < 2 ? 1 : (nt > 8 ? 8 : nt);
    if (getenv("URMB_LOAD_THREADS")) nt = (unsigned)std::max(1, atoi(getenv("URMB_LOAD_THREADS")));
    uint8_t *stage[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr}, evc = nullptr;
    struct Release {   // every early return below releases the staging buffers and events
        uint8_t **stage; cudaEvent_t *ev, *evc;
        ~Release() {
            cudaFreeHost(stage[0]); cudaFreeHost(stage[1]);
            if (ev[0]) cudaEventDestroy(ev[0]);
            if (ev[1]) cudaEventDestroy(ev[1]);
            if (*evc) cudaEventDestroy(*evc);
        }
    } release{stage, ev, &evc};
    CK(cudaSetDevice(c->device));
    CK(cudaHostAlloc(&stage[0], CH, cudaHostAllocPortable));
    CK(cudaHostAlloc(&stage[1], CH, cudaHostAllocPortable));
    CK(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&evc, cudaEventDisableTiming));
    int k = 0;
    std::vector<std::thread> th;
    for (size_t o = 0; o < n; o += CH, k ^= 1) {
        const size_t m = std::min(CH, n - o);
        CK(cudaEventSynchronize(ev[k]));
        const size_t piece = ((m + nt - 1) / nt + 4095) & ~(size_t)4095;
        th.clear();
        for (unsigned t = 1; t < nt; ++t) {
            const size_t lo = std::min(m, t * piece), hi = std::min(m, (t + 1) * piece);
            if (hi > lo) th.emplace_back([=]() { memcpy(stage[k] + lo, src + o + lo, hi - lo); });
        }
        memcpy(stage[k], src + o, std::min(m, piece));
        for (auto &x : th) x.join();
        CK(cudaMemcpyAsync((uint8_t *)dst + o, stage[k], m, cudaMemcpyHostToDevice, c->compute));
        CK(cudaEventRecord(ev[k], c->compute));
        if (fan && fan->n > 1) {   // the chunk that just landed on GPU 0 goes on to the peers
            CK(cudaEventRecord(evc, c->compute));
            for (int g = 1; g < fan->n; ++g) {
                CK(cudaStreamWaitEvent(fan->streams[g], evc, 0));
                CK(cudaMemcpyPeerAsync((uint8_t *)fan->dst[g] + o, fan->ctxs[g]->device, (uint8_t *)dst + o, c->device, m, fan->streams[g]));
            }
        }
    }
    CK(cudaStreamSynchronize(c->compute));
    if (fan) for (int g = 1; g < fan->n; ++g) CK(cudaStreamSynchronize(fan->streams[g]));
    return URMB_OK;
}

extern "C" int urmb_index_upload(urmb_ctx *c, const urmb_index_host *h) {
    urmb_ctx *one[1] = {c};
    return urmb_index_broadcast(one, 1, h);
}

// UFIndex::FromFile for n GPUs of one process (state1.cpp:185 SetUFI on every worker): buffers on every GPU, one pass
// over the file (upload_region with the NVLink fan-out), derived data built on each GPU.  The one-process-per-GPU path
// (bench.py) instead broadcasts with NCCL and calls urmb_index_attach.
extern "C" int urmb_index_broadcast(urmb_ctx **ctxs, int n, const urmb_index_host *h) {
    if (!ctxs || n < 1 || !h) return URMB_E_ARG;
    for (int i = 0; i < n; ++i) if (!ctxs[i]) return URMB_E_ARG;
    urmb_ctx *c = ctxs[0];
    const size_t nb = 5 * (size_t)h->slot_count, ns = h->seq_data_size;
    Fanout fb, fs;
    fb.n = fs.n = n;
    fb.ctxs = fs.ctxs = ctxs;
    fb.dst.assign(n, nullptr); fs.dst.assign(n, nullptr);
    fb.streams.assign(n, nullptr); fs.streams.assign(n, nullptr);
    for (int i = 0; i < n; ++i) {
        urmb_ctx *d = ctxs[i];
        {   // errors below are reported against the context they belong to
            urmb_ctx *c = d;
            CK(cudaSetDevice(d->device));
            cudaFree(d->own_blob);
            cudaFree(d->own_seq);
            d->own_blob = d->own_seq = nullptr;
            CK(cudaMalloc(&d->own_blob, nb + URMB_BLOB_PAD));
            CK(cudaMalloc(&d->own_seq, ns + URMB_SEQ_PAD));
            CK(cudaMemset((uint8_t *)d->own_blob + nb, 0, URMB_BLOB_PAD));
            CK(cudaMemset((uint8_t *)d->own_seq + ns, 0, URMB_SEQ_PAD));
            if (i > 0) {
                int can = 0;
                cudaDeviceCanAccessPeer(&can, d->device, ctxs[0]->device);
                if (can) cudaDeviceEnablePeerAccess(ctxs[0]->device, 0);   // peer copies then go GPU to GPU over NVLink
                cudaGetLastError();
            }
        }
        fb.dst[i] = d->own_blob;
        fs.dst[i] = d->own_seq;
        fb.streams[i] = fs.streams[i] = d->slots[0].copy;
    }
    int rc = upload_region(c, c->own_blob, h->blob, nb, &fb);
    if (rc) return rc;
    rc = upload_region(c, c->own_seq, h->seq, ns, &fs);
    if (rc) return rc;
    std::vector<int> rcs(n, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i)   // derived data (2-bit genome, exception bits) on every GPU at once
        th.emplace_back([&, i]() {
            urmb_index_desc d;
            urmb_index_info(h, &d, nullptr);
            d.d_blob = ctxs[i]->own_blob;
            d.d_seq = ctxs[i]->own_seq;
            rcs[i] = set_index(ctxs[i], &d);
        });
    for (auto &t : th) t.join();
    for (int i = 0; i < n; ++i) if (rcs[i]) return rcs[i];
    return URMB_OK;
}

// Index of a FASTA file built on the devices of n contexts (no UFI file): the raw bytes go to every GPU through the
// fan-out of upload_region (3.1 GB for a human genome instead of the 30 GB table), then each GPU parses them
// (urmb_fasta.cu), frees them, builds the table (urmb_build_index_device) and derives its packed genome on its own host
// thread, all at the same time.
extern "C" int urmb_index_from_fasta(urmb_ctx **ctxs, int n, const uint8_t *fa, uint64_t fa_len, uint32_t word_length,
                                     uint32_t max_ix, uint64_t slot_count, urmb_index_host **header) {
    if (!ctxs || n < 1 || !header || (!fa && fa_len)) return URMB_E_ARG;
    *header = nullptr;
    for (int i = 0; i < n; ++i) if (!ctxs[i]) return URMB_E_ARG;
    urmb_ctx *c = ctxs[0];
    if (slot_count < 2) return fail(c, URMB_E_ARG, "bad slot count");
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    const uint64_t padded = fasta_padded_len(fa_len);
    std::vector<void *> d_fa(n, nullptr);
    struct Release {   // the raw bytes, on every return
        std::vector<urmb_ctx *> ctxs; std::vector<void *> *d_fa;
        ~Release() { for (size_t i = 0; i < ctxs.size(); ++i) if ((*d_fa)[i]) { cudaSetDevice(ctxs[i]->device); cudaFree((*d_fa)[i]); } }
    } release{std::vector<urmb_ctx *>(ctxs, ctxs + n), &d_fa};
    Fanout fan;
    fan.n = n;
    fan.ctxs = ctxs;
    fan.dst.assign(n, nullptr);
    fan.streams.assign(n, nullptr);
    for (int i = 0; i < n; ++i) {
        urmb_ctx *c = ctxs[i];   // errors below are reported against the context they belong to
        CK(cudaSetDevice(c->device));
        c->have_index = false;
        cudaFree(c->own_blob);
        cudaFree(c->own_seq);
        c->own_blob = c->own_seq = nullptr;
        CK(cudaMalloc(&d_fa[i], padded));
        CK(cudaMemset((uint8_t *)d_fa[i] + fa_len, 0, padded - fa_len));
        if (i > 0) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, c->device, ctxs[0]->device);
            if (can) cudaDeviceEnablePeerAccess(ctxs[0]->device, 0);
            cudaGetLastError();
        }
        fan.dst[i] = d_fa[i];
        fan.streams[i] = c->slots[0].copy;
    }
    int rc = upload_region(c, d_fa[0], fa, fa_len, &fan);
    if (rc) return rc;
    const double t1 = now();
    std::vector<int> rcs(n, 0);
    std::vector<FastaTable> tabs(n);
    std::vector<double> t_parse(n, 0), t_build(n, 0), t_pack(n, 0);
    std::vector<float> k_ms(n, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i)
        th.emplace_back([&, i]() {
            urmb_ctx *c = ctxs[i];
            rcs[i] = [&]() -> int {
                CK(cudaSetDevice(c->device));
                const double a = now();
                void *d_seq = nullptr;
                std::string err;
                int r = fasta_parse_device((const uint8_t *)d_fa[i], fa, fa_len, c->compute, &d_seq, tabs[i], &k_ms[i], err);
                cudaFree(d_fa[i]);   // before the build: the raw bytes are not needed any more
                d_fa[i] = nullptr;
                if (r) return fail(c, r, err);
                c->own_seq = d_seq;
                const double b = now();
                t_parse[i] = b - a;
                const uint64_t nb = 5 * slot_count;
                CK(cudaMalloc(&c->own_blob, nb + URMB_BLOB_PAD));
                uint64_t stats[3] = {0, 0, 0};
                r = urmb_build_index_device(c->own_seq, tabs[i].seq_size, slot_count, word_length, max_ix, c->own_blob, stats);
                if (r) return fail(c, r, urmb_build_last_error());
                if (stats[1])
                    return fail(c, URMB_E_OVERFLOW, std::to_string(stats[1]) + " list(s) would have to be truncated (TruncateSlot)");
                const double d = now();
                t_build[i] = d - b;
                urmb_index_desc desc{word_length, max_ix, (uint32_t)tabs[i].seq_size, 0, slot_count, c->own_blob, c->own_seq};
                r = set_index(c, &desc);
                t_pack[i] = now() - d;
                return r;
            }();
        });
    for (auto &t : th) t.join();
    for (int i = 0; i < n; ++i)
        if (rcs[i]) return fail(c, rcs[i], ctxs[i]->err);
    urmb_index_host *h = new urmb_index_host;
    const FastaTable &t = tabs[0];
    h->word_length = word_length;
    h->max_ix = max_ix;
    h->seq_data_size = (uint32_t)t.seq_size;
    h->slot_count = slot_count;
    for (const std::string &l : t.labels) h->labels.push_back(std::string(l.c_str()));   // as urmb_index_load_host reads them
    h->lengths = t.lengths;
    h->offsets = t.offsets;
    h->dropped = t.dropped;
    h->fasta_times[0] = t1 - t0;
    for (int i = 0; i < n; ++i) {
        h->fasta_times[1] = std::max(h->fasta_times[1], t_parse[i]);
        h->fasta_times[2] = std::max(h->fasta_times[2], t_build[i]);
        h->fasta_times[3] = std::max(h->fasta_times[3], t_pack[i]);
        h->fasta_times[4] = std::max(h->fasta_times[4], (double)k_ms[i] / 1e3);
    }
    *header = h;
    return URMB_OK;
}

extern "C" int urmb_index_dropped(const urmb_index_host *h, uint32_t i, const char **label) {
    if (!h || !label || i >= h->dropped.size()) return URMB_E_ARG;
    *label = h->dropped[i].c_str();
    return URMB_OK;
}

extern "C" int urmb_index_fasta_times(const urmb_index_host *h, double *t) {
    if (!h || !t) return URMB_E_ARG;
    memcpy(t, h->fasta_times, sizeof h->fasta_times);
    return URMB_OK;
}

// ---------------------------------------------------------------------------------------
// batches
// ---------------------------------------------------------------------------------------
template <class T>
static int grow_host(urmb_ctx *c, T *&p, size_t &cap, size_t need) {
    if (need <= cap) return URMB_OK;
    size_t ncap = std::max(need, cap * 2);
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    CK(cudaHostAlloc(&p, ncap * sizeof(T), cudaHostAllocDefault));
    cap = ncap;
    return URMB_OK;
}
template <class T>
static int grow_dev(urmb_ctx *c, T *&p, size_t &cap, size_t need) {
    if (need <= cap) return URMB_OK;
    size_t ncap = std::max(need, cap * 2);
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    CK(cudaMalloc(&p, ncap * sizeof(T)));
    cap = ncap;
    return URMB_OK;
}

// Page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. urmb_host_alloc or a pinned torch tensor) can be read
// by the copy engine directly; anything else goes through the slot's pinned staging buffer.
static bool is_pinned_host(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

static int check_batch(urmb_ctx *c, const urmb_batch *b) {
    if (!b || (b->n && (!b->seqs || !b->offs))) return fail(c, URMB_E_ARG, "null batch");
    return URMB_OK;
}

// Sizes every slot (and the pool of saved mate states) for batches of n_units reads / pairs of up to max_read_len bases,
// so that the first batches do not pay for the allocations.  Touches only the slots and the pool: the CLI calls it from
// a helper thread while urmb_index_broadcast is still copying the index.
// Side-stream resources of a slot for batches of n units: scratch of the rescue / rerun kernels, and for paired-end
// batches the rescue pool: one pair in eight (at least 4096, at most 131072 entries of 21.6 kB); pairs beyond that take
// the legacy kernel.
static int size_side_resources(urmb_ctx *c, Slot &s, size_t n, bool paired) {
    if (!s.big_scratch && !c->no_rerun) CK(cudaMalloc(&s.big_scratch, urmb_big_scratch_bytes() * (size_t)kBigWarps));
    if (!paired || c->P.pe_method == 5) return URMB_OK;
    if (!s.rescue_scratch) CK(cudaMalloc(&s.rescue_scratch, sizeof(WarpScratch) * (size_t)c->n_rescue_warps));
    if (c->rescue_legacy) return URMB_OK;
    const size_t want = std::min<size_t>(std::max<size_t>(n / 8, 4096), 131072);
    if (want <= s.rescue_cap) return URMB_OK;
    CK(cudaStreamSynchronize(s.side));
    cudaFree(s.rpool); cudaFree(s.rq[0]); cudaFree(s.rq[1]);
    s.rpool = nullptr; s.rq[0] = s.rq[1] = nullptr;
    s.rescue_cap = 0;
    CK(cudaMalloc(&s.rpool, sizeof(RescueSave) * want));
    CK(cudaMalloc(&s.rq[0], sizeof(uint32_t) * (want + 1)));
    CK(cudaMalloc(&s.rq[1], sizeof(uint32_t) * (want + 1)));
    s.rescue_cap = want;
    return URMB_OK;
}

extern "C" int urmb_reserve(urmb_ctx *c, uint32_t n_units, uint32_t max_read_len, int paired, uint32_t word_length) {
    if (!c || n_units == 0 || max_read_len == 0 || max_read_len > (uint32_t)kMaxLen || word_length < 8 || word_length > 32)
        return URMB_E_ARG;
    CK(cudaSetDevice(c->device));
    const size_t n = n_units, nreads = paired ? 2 * n : n;
    const size_t nbytes = nreads * max_read_len;
    if (nbytes >= 0xFFFFFFF0ull) return fail(c, URMB_E_UNSUPPORTED, "batch larger than 4 GB of bases");
    const uint32_t qwc = max_read_len >= word_length ? max_read_len - word_length + 1 : 1;
    const uint32_t qcap = (qwc + 31) & ~31u, seqcap = (std::max(max_read_len, 32u) + 31) & ~31u;
    int rc;
    for (auto &s : c->slots) {
        if ((rc = grow_host(c, s.h_offs, s.h_offs_cap, nreads + 1))) return rc;
        if ((rc = grow_dev(c, s.d_seqs, s.d_seqs_cap, nbytes + 64))) return rc;
        if ((rc = grow_dev(c, s.d_offs, s.d_offs_cap, nreads + 1))) return rc;
        const size_t probe_need = nreads * 2 * qcap;
        if (probe_need > s.d_probe_cap) {
            cudaFree(s.d_tally); cudaFree(s.d_pos); cudaFree(s.d_ext);
            s.d_tally = nullptr; s.d_pos = nullptr; s.d_ext = nullptr;
            s.d_probe_cap = 0;
            CK(cudaMalloc(&s.d_tally, probe_need));
            CK(cudaMalloc(&s.d_pos, probe_need * 4));
            CK(cudaMalloc(&s.d_ext, probe_need * 4));
            s.d_probe_cap = probe_need;
        }
        if ((rc = grow_dev(c, s.d_view, s.d_view_cap, nreads * view_stride_for(seqcap) + 64 + n))) return rc;   // + the pairs' first-look flags
        if ((rc = grow_dev(c, s.d_res, s.d_res_cap, nreads + 1))) return rc;
        if ((rc = grow_dev(c, s.d_todo, s.d_todo_cap, n + 1))) return rc;
        if ((rc = grow_dev(c, s.d_rescue, s.d_rescue_cap, n + 1))) return rc;
        if ((rc = grow_host(c, s.h_res, s.h_res_cap, nreads + 1))) return rc;
        if ((rc = grow_dev(c, s.d_runs, s.d_runs_cap, nreads * 8 + 4096))) return rc;
        if ((rc = grow_host(c, s.h_runs, s.h_runs_cap, s.d_runs_cap))) return rc;
    }
    const size_t units = paired ? n : (n + 1) / 2;
    const size_t want = std::min<size_t>(std::max<size_t>(units, 1), c->chunk_pairs);
    if (want > c->pool_pairs) {
        CK(cudaStreamSynchronize(c->compute));
        CK(cudaStreamSynchronize(c->compute2));
        cudaFree(c->pool);
        cudaFree(c->pool2);
        c->pool = c->pool2 = nullptr;
        c->pool_pairs = 0;
        CK(cudaMalloc(&c->pool, sizeof(MateSave) * 2 * want));
        if (c->lanes == 2) CK(cudaMalloc(&c->pool2, sizeof(MateSave) * 2 * want));
        c->pool_pairs = want;
    }
    for (auto &s : c->slots)
        if ((rc = size_side_resources(c, s, n, paired != 0))) return rc;
    return URMB_OK;
}

extern "C" int urmb_upload(urmb_ctx *c, int si, const urmb_batch *r1, const urmb_batch *r2) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    if (!c->have_index) return fail(c, URMB_E_ARG, "no index attached");
    int rc = check_batch(c, r1);
    if (rc) return rc;
    if (r2) {
        rc = check_batch(c, r2);
        if (rc) return rc;
        if (r2->n != r1->n) return fail(c, URMB_E_ARG, "mate batches differ in size (map2.cpp:31 dies here)");
    }
    CK(cudaSetDevice(c->device));
    Slot &s = c->slots[si];
    const uint32_t n = r1->n, nreads = r2 ? 2 * n : n;
    const size_t b1 = n ? r1->offs[n] - r1->offs[0] : 0, b2 = (r2 && n) ? r2->offs[n] - r2->offs[0] : 0;
    size_t nbytes = b1 + b2;
    if (nbytes >= 0xFFFFFFF0ull) return fail(c, URMB_E_UNSUPPORTED, "batch larger than 4 GB of bases");
    // previous use of this slot must have drained
    CK(cudaStreamSynchronize(s.copy));
    bool direct = n > 0 && !getenv("URMB_NO_DIRECT_H2D") && is_pinned_host(r1->seqs) && (!r2 || is_pinned_host(r2->seqs));
    if (!direct && (rc = grow_host(c, s.h_seqs, s.h_seqs_cap, nbytes + 64))) return rc;
    if ((rc = grow_host(c, s.h_offs, s.h_offs_cap, (size_t)nreads + 1))) return rc;
    if ((rc = grow_dev(c, s.d_seqs, s.d_seqs_cap, nbytes + 64))) return rc;
    if ((rc = grow_dev(c, s.d_offs, s.d_offs_cap, (size_t)nreads + 1))) return rc;
    uint32_t maxlen = 0;
    s.too_long.clear();
    if (n) {
        for (uint32_t i = 0; i < n; ++i) maxlen = std::max(maxlen, r1->offs[i + 1] - r1->offs[i]);
        if (r2) for (uint32_t i = 0; i < n; ++i) maxlen = std::max(maxlen, r2->offs[i + 1] - r2->offs[i]);
    }
    if (maxlen > (uint32_t)kMaxLen) {
        // Reads longer than URMB_MAX_READ_LEN are handled per read, not per batch: they (and their mates) go to the
        // device as empty reads, come back unmapped with bit 6 of urmb_result.flags set, and are counted
        // (urmb_unsupported_count).  The rest of the batch is mapped as usual.  The bases are staged read by read.
        direct = false;
        if ((rc = grow_host(c, s.h_seqs, s.h_seqs_cap, nbytes + 64))) return rc;
        size_t o = 0;
        maxlen = 0;
        for (int mate = 0; mate < (r2 ? 2 : 1); ++mate) {
            const urmb_batch *rb = mate ? r2 : r1;
            const urmb_batch *ob = mate ? r1 : r2;   // the other mate (null for single-end)
            for (uint32_t i = 0; i < n; ++i) {
                const uint32_t L = rb->offs[i + 1] - rb->offs[i];
                const bool skip = L > (uint32_t)kMaxLen || (ob && ob->offs[i + 1] - ob->offs[i] > (uint32_t)kMaxLen);
                s.h_offs[(size_t)mate * n + i] = (uint32_t)o;
                if (skip) { s.too_long.push_back(mate * n + i); continue; }
                memcpy(s.h_seqs + o, rb->seqs + rb->offs[i], L);
                o += L;
                maxlen = std::max(maxlen, L);
            }
        }
        s.h_offs[nreads] = (uint32_t)o;
        nbytes = o;
    } else if (n) {
        if (!direct) memcpy(s.h_seqs, r1->seqs + r1->offs[0], b1);
        const uint32_t o0 = r1->offs[0];
        for (uint32_t i = 0; i <= n; ++i) s.h_offs[i] = r1->offs[i] - o0;
        if (r2) {
            if (!direct) memcpy(s.h_seqs + b1, r2->seqs + r2->offs[0], b2);
            const uint32_t p0 = r2->offs[0];
            for (uint32_t i = 0; i <= n; ++i) s.h_offs[n + i] = (uint32_t)b1 + (r2->offs[i] - p0);
        }
    } else {
        s.h_offs[0] = 0;
    }
    const uint32_t W = c->ix.word_len;
    const uint32_t qwc = maxlen >= W ? maxlen - W + 1 : 1;
    DevBatch &b = s.batch;
    b.seqs = s.d_seqs;
    b.offs = s.d_offs;
    b.n_reads = nreads;
    b.n_units = n;
    b.qcap = (qwc + 31) & ~31u;
    b.seqcap = (std::max(maxlen, 32u) + 31) & ~31u;
    b.paired = r2 ? 1 : 0;
    s.seq_bytes = nbytes;
    const size_t probe_need = (size_t)nreads * 2 * b.qcap;
    if (probe_need > s.d_probe_cap) {
        cudaFree(s.d_tally); cudaFree(s.d_pos); cudaFree(s.d_ext);
        s.d_tally = nullptr; s.d_pos = nullptr; s.d_ext = nullptr;
        s.d_probe_cap = 0;
        size_t ncap = std::max(probe_need, (size_t)1024);
        CK(cudaMalloc(&s.d_tally, ncap));
        CK(cudaMalloc(&s.d_pos, ncap * 4));
        CK(cudaMalloc(&s.d_ext, ncap * 4));
        s.d_probe_cap = ncap;
    }
    if ((rc = grow_dev(c, s.d_view, s.d_view_cap, (size_t)nreads * view_stride_for(b.seqcap) + 64 + n))) return rc;   // + the pairs' first-look flags
    if ((rc = grow_dev(c, s.d_res, s.d_res_cap, (size_t)nreads + 1))) return rc;
    if ((rc = grow_dev(c, s.d_todo, s.d_todo_cap, (size_t)n + 1))) return rc;
    if ((rc = grow_dev(c, s.d_rescue, s.d_rescue_cap, (size_t)n + 1))) return rc;
    {   // pool of saved mate states (2 per pair, 1 per single-end read), shared by the slots: their kernels are
        // serialised on the compute stream
        const size_t units = r2 ? n : ((size_t)n + 1) / 2;
        const size_t want = std::min<size_t>(std::max<size_t>(units, 1), c->chunk_pairs);
        if (want > c->pool_pairs) {
            CK(cudaStreamSynchronize(c->compute));
            CK(cudaStreamSynchronize(c->compute2));
            cudaFree(c->pool);
            cudaFree(c->pool2);
            c->pool = c->pool2 = nullptr;
            c->pool_pairs = 0;
            CK(cudaMalloc(&c->pool, sizeof(MateSave) * 2 * want));
            if (c->lanes == 2) CK(cudaMalloc(&c->pool2, sizeof(MateSave) * 2 * want));
            c->pool_pairs = want;
        }
    }
    if ((rc = size_side_resources(c, s, n, r2 != nullptr))) return rc;
    if ((rc = grow_host(c, s.h_res, s.h_res_cap, (size_t)nreads + 1))) return rc;
    if (c->params.want_second && r2) {
        if ((rc = grow_dev(c, s.d_second, s.d_second_cap, (size_t)nreads + 1))) return rc;
        if ((rc = grow_host(c, s.h_second, s.h_second_cap, (size_t)nreads + 1))) return rc;
    }
    const size_t runs_need = (size_t)nreads * 8 + 4096;
    if ((rc = grow_dev(c, s.d_runs, s.d_runs_cap, runs_need))) return rc;
    if ((rc = grow_host(c, s.h_runs, s.h_runs_cap, s.d_runs_cap))) return rc;
    CK(cudaEventRecord(s.ev_h2d0, s.copy));
    if (direct) {   // the caller's pinned bases go to the device as they are; they must stay valid until urmb_wait
        CK(cudaMemcpyAsync(s.d_seqs, r1->seqs + r1->offs[0], b1, cudaMemcpyHostToDevice, s.copy));
        if (r2) CK(cudaMemcpyAsync(s.d_seqs + b1, r2->seqs + r2->offs[0], b2, cudaMemcpyHostToDevice, s.copy));
    } else {
        CK(cudaMemcpyAsync(s.d_seqs, s.h_seqs, nbytes, cudaMemcpyHostToDevice, s.copy));
    }
    CK(cudaMemcpyAsync(s.d_offs, s.h_offs, ((size_t)nreads + 1) * 4, cudaMemcpyHostToDevice, s.copy));
    CK(cudaEventRecord(s.ev_h2d, s.copy));
    s.staged = true;
    s.launched = false;
    s.downloaded = false;
    s.counted = false;
    return URMB_OK;
}

struct TraceCtx {
    Slot *s;
    cudaStream_t stream;
    cudaError_t err;
};
static void trace_mark(void *user, int klass, int phase) {
    TraceCtx *t = (TraceCtx *)user;
    Slot &s = *t->s;
    const size_t i = 2 * s.nkev + (size_t)phase;
    while (s.kev.size() <= i) {
        cudaEvent_t ev;
        cudaError_t e = cudaEventCreate(&ev);
        if (e != cudaSuccess) { t->err = e; return; }
        s.kev.push_back(ev);
    }
    cudaError_t e = cudaEventRecord(s.kev[i], t->stream);
    if (e != cudaSuccess) t->err = e;
    if (phase == 0) {
        if (s.kclass.size() <= s.nkev) s.kclass.resize(s.nkev + 1);
        s.kclass[s.nkev] = klass;
    } else {
        ++s.nkev;
    }
}

extern "C" int urmb_launch(urmb_ctx *c, int si) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    Slot &s = c->slots[si];
    if (!s.staged) return fail(c, URMB_E_ARG, "slot not staged");
    CK(cudaSetDevice(c->device));
    cudaStream_t side = s.side;
    const int lane = (c->lanes == 2 && !c->rescue_inline) ? c->lane_next : 0;   // compute lane of this launch
    if (c->lanes == 2) c->lane_next ^= 1;
    cudaStream_t cs = lane ? c->compute2 : c->compute;
    CK(cudaStreamWaitEvent(cs, s.ev_h2d, 0));
    if (s.launched) CK(cudaStreamWaitEvent(cs, s.ev_rescue, 0));   // an earlier launch of this very slot
    CK(cudaMemsetAsync(s.d_counters, 0, CT_COUNT * sizeof(uint32_t), cs));
    CK(cudaEventRecord(s.ev_k0, cs));
    s.nkev = 0;
    bool rescued = false;
    if (s.batch.n_reads) {
        DevProbe pr{s.d_tally, s.d_pos, s.d_ext, s.d_view, view_stride_for(s.batch.seqcap),
                    s.batch.paired ? s.d_view + (size_t)s.batch.n_reads * view_stride_for(s.batch.seqcap) + 64 : nullptr};
        urmb_second *second = (c->params.want_second && s.batch.paired) ? s.d_second : nullptr;
        if (second) CK(cudaMemsetAsync(second, 0, (size_t)s.batch.n_reads * sizeof(urmb_second), cs));
        const bool use_pool = s.batch.paired && s.rescue_cap && s.rpool;
        DevOut o{s.d_res, s.d_runs, (uint32_t)std::min<size_t>(s.d_runs_cap, 0xFFFFFFFFu), s.d_counters, s.d_todo, s.d_rescue, second,
                 use_pool ? s.rpool : nullptr, use_pool ? (uint32_t)s.rescue_cap : 0u,
                 {use_pool ? s.rq[0] : nullptr, use_pool ? s.rq[1] : nullptr},
                 s.big_scratch ? s.d_ovf : nullptr, s.big_scratch ? kOvfCap : 0u, s.big_scratch ? s.d_ovf_units : nullptr};
        SearchRes R{lane ? c->scratch2 : c->scratch, c->n_scratch_warps, lane ? c->pool2 : c->pool, (uint32_t)c->pool_pairs};
        DevParams P = c->P;
        TraceCtx tc{&s, cs, cudaSuccess};
        LaunchTrace tr{trace_mark, &tc};
        trace_mark(&tc, 0, 0);
        int e = launch_probe(c->ix, P, s.batch, pr, cs, c->sm_count, &o);
        trace_mark(&tc, 0, 1);
        if (e) return fail(c, URMB_E_CUDA, std::string("probe launch: ") + cudaGetErrorString((cudaError_t)e));
        CK(cudaEventRecord(s.ev_k1, cs));
        e = launch_search(c->ix, P, s.batch, pr, o, R, cs, c->sm_count, nullptr, &tr);
        if (e < 0) return fail(c, URMB_E_CUDA, std::string("search launch: ") + cudaGetErrorString((cudaError_t)-e));
        c->launches += 1 + (uint64_t)e;
        CK(cudaEventRecord(s.ev_k2, cs));
        // Mate rescue: few, long work items.  It runs on the low-priority side stream so that its tail overlaps the
        // kernels of the next batch instead of idling the GPU.
        SearchRes RR{s.rescue_scratch, c->n_rescue_warps, nullptr, 0};
        cudaStream_t rs = c->rescue_inline ? cs : side;
        CK(cudaStreamWaitEvent(rs, s.ev_k2, 0));
        tc.stream = rs;
        e = launch_rescue(c->ix, P, s.batch, pr, o, c->rescue_inline ? R : RR, rs, c->sm_count, &tr);
        if (c->rescue_inline) CK(cudaEventRecord(s.ev_k2, cs));
        if (e < 0) return fail(c, URMB_E_CUDA, std::string("rescue launch: ") + cudaGetErrorString((cudaError_t)-e));
        c->launches += (uint64_t)e;
        if (s.big_scratch) {
            // Reads over a per-mate capacity of the fast kernels are searched again by the big-capacity build on the slot's
            // high-priority stream: a first pass as soon as the search kernels are done (beside the mate rescue), a second
            // one after the mate rescue for the reads it added to the list (usually none).
            cudaStream_t bs = c->rescue_inline ? cs : s.big;
            for (int pass = 0; pass < 2; ++pass) {
                if (!c->rescue_inline) {
                    if (pass == 0) CK(cudaStreamWaitEvent(bs, s.ev_k2, 0));
                    else {
                        CK(cudaEventRecord(s.ev_side, rs));
                        CK(cudaStreamWaitEvent(bs, s.ev_side, 0));
                    }
                } else if (pass == 0) continue;   // inline: everything is on one stream, one pass at the end is enough
                e = urmb_big_rerun_listed(&c->ix, &P, &s.batch, &pr, &o, s.big_scratch, kBigWarps, bs, c->sm_count);
                if (e < 0) return fail(c, URMB_E_CUDA, std::string("big-capacity rerun launch: ") + cudaGetErrorString((cudaError_t)-e));
                c->launches += (uint64_t)e;
            }
            if (c->rescue_inline) CK(cudaEventRecord(s.ev_k2, cs));
            else {   // the batch is done when both streams are
                CK(cudaEventRecord(s.ev_big, bs));
                CK(cudaStreamWaitEvent(rs, s.ev_big, 0));
            }
        }
        if (tc.err != cudaSuccess) return fail(c, URMB_E_CUDA, std::string("event record: ") + cudaGetErrorString(tc.err));
        rescued = true;   // the side stream has work of this batch (or, inline, waits for the re-recorded ev_k2 below)
        if (c->rescue_inline) rescued = false;
    } else {
        CK(cudaEventRecord(s.ev_k1, cs));
        CK(cudaEventRecord(s.ev_k2, cs));
    }
    if (!rescued) CK(cudaStreamWaitEvent(side, s.ev_k2, 0));
    CK(cudaEventRecord(s.ev_rescue, side));
    s.launched = true;
    s.downloaded = false;
    return URMB_OK;
}

extern "C" int urmb_mark(urmb_ctx *c, int which) {
    if (!c || which < 0 || which > 1) return URMB_E_ARG;
    CK(cudaSetDevice(c->device));
    for (auto &s : c->slots)   // a mark comes after the side-stream work of every batch launched so far
        if (s.launched) CK(cudaStreamWaitEvent(c->compute, s.ev_rescue, 0));
    CK(cudaEventRecord(c->ev_lane, c->compute2));   // ... and after the second compute lane; which then waits for the mark
    CK(cudaStreamWaitEvent(c->compute, c->ev_lane, 0));
    CK(cudaEventRecord(c->ev_mark[which], c->compute));
    CK(cudaStreamWaitEvent(c->compute2, c->ev_mark[which], 0));
    return URMB_OK;
}

extern "C" int urmb_mark_elapsed(urmb_ctx *c, float *ms) {
    if (!c || !ms) return URMB_E_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaEventSynchronize(c->ev_mark[1]));
    CK(cudaEventElapsedTime(ms, c->ev_mark[0], c->ev_mark[1]));
    return URMB_OK;
}

extern "C" int urmb_download(urmb_ctx *c, int si) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    Slot &s = c->slots[si];
    if (!s.launched) return fail(c, URMB_E_ARG, "slot not launched");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamWaitEvent(s.copy, s.ev_k2, 0));
    CK(cudaStreamWaitEvent(s.copy, s.ev_rescue, 0));
    CK(cudaMemcpyAsync(s.h_counters, s.d_counters, CT_COUNT * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.copy));
    CK(cudaMemcpyAsync(s.h_res, s.d_res, (size_t)s.batch.n_reads * sizeof(urmb_result), cudaMemcpyDeviceToHost, s.copy));
    if (c->params.want_second && s.batch.paired && s.batch.n_reads)
        CK(cudaMemcpyAsync(s.h_second, s.d_second, (size_t)s.batch.n_reads * sizeof(urmb_second), cudaMemcpyDeviceToHost, s.copy));
    // Paths are few and short: copy the whole pool prefix a typical batch uses, the rest on demand in wait.
    s.downloaded = true;
    return URMB_OK;
}

extern "C" int urmb_host_alloc(size_t bytes, void **out) {
    if (!out) return URMB_E_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        set_global_error(std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
        cudaGetLastError();
        return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? URMB_E_NODEVICE : URMB_E_CUDA;
    }
    return URMB_OK;
}

extern "C" void urmb_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" int urmb_submit(urmb_ctx *c, int si, const urmb_batch *r1, const urmb_batch *r2) {
    int rc = urmb_upload(c, si, r1, r2);
    if (rc) return rc;
    rc = urmb_launch(c, si);
    if (rc) return rc;
    return urmb_download(c, si);
}

// Reads whose search overflowed a per-mate capacity of the fast build (urmb_result.flags bit 7) are mapped again, still on
// the GPU, by the same kernels compiled with capacities no read can exceed (urmb_big.cu); their records, path runs and second
// hits replace the overflowed ones.  Runs on its own stream (the other slots' batches keep flowing); pieces of 1024 units.
static int rerun_overflowed(urmb_ctx *c, Slot &s, uint32_t &used) {
    const uint32_t n = s.batch.n_units, nreads = s.batch.n_reads;
    const bool paired = s.batch.paired != 0;
    std::vector<uint32_t> sel;
    for (uint32_t u = 0; u < n; ++u)
        if ((s.h_res[u].flags & 0x80) || (paired && (s.h_res[n + u].flags & 0x80))) sel.push_back(u);
    if (sel.empty()) return URMB_OK;
    urmb_ctx::Big &g = c->big;
    const uint32_t KU = urmb_ctx::Big::kUnits, KR = 2 * KU;
    const bool second = c->params.want_second && paired;
    if (!g.ready) {
        int plo = 0, phi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&plo, &phi));
        CK(cudaStreamCreateWithPriority(&g.stream, cudaStreamNonBlocking, phi));   // its few blocks go first when an SM frees up
        CK(cudaMalloc(&g.d_offs, (KR + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&g.d_counters, CT_COUNT * sizeof(uint32_t)));
        CK(cudaMalloc(&g.d_todo, (KU + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&g.d_rescue, (KU + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&g.d_res, (KR + 1) * sizeof(urmb_result)));
        CK(cudaMalloc(&g.d_second, (KR + 1) * sizeof(urmb_second)));
        g.runs_cap = (size_t)KR * 512 + 4096;
        CK(cudaMalloc(&g.d_runs, g.runs_cap * sizeof(uint16_t)));
        CK(cudaMalloc(&g.scratch, urmb_big_scratch_bytes() * (size_t)urmb_ctx::Big::kWarps));
        CK(cudaMalloc(&g.pool, urmb_big_save_bytes() * 2 * 256));
        CK(cudaHostAlloc(&g.h_res, (KR + 1) * sizeof(urmb_result), cudaHostAllocDefault));
        CK(cudaHostAlloc(&g.h_second, (KR + 1) * sizeof(urmb_second), cudaHostAllocDefault));
        CK(cudaHostAlloc(&g.h_runs, g.runs_cap * sizeof(uint16_t), cudaHostAllocDefault));
        CK(cudaHostAlloc(&g.h_counters, CT_COUNT * sizeof(uint32_t), cudaHostAllocDefault));
        CK(cudaHostAlloc(&g.h_offs, (KR + 1) * sizeof(uint32_t), cudaHostAllocDefault));
        g.ready = true;
    }
    int rc;
    const size_t seq_need = (size_t)KR * s.batch.seqcap + 64, probe_need = (size_t)KR * 2 * s.batch.qcap;
    const size_t view_need = (size_t)KR * view_stride_for(s.batch.seqcap) + 64;
    if ((rc = grow_dev(c, g.d_seqs, g.seq_cap, seq_need))) return rc;
    if ((rc = grow_dev(c, g.d_view, g.view_cap, view_need))) return rc;
    if (probe_need > g.probe_cap) {
        cudaFree(g.d_tally); cudaFree(g.d_pos); cudaFree(g.d_ext);
        g.d_tally = nullptr; g.d_pos = nullptr; g.d_ext = nullptr;
        g.probe_cap = 0;
        CK(cudaMalloc(&g.d_tally, probe_need));
        CK(cudaMalloc(&g.d_pos, probe_need * 4));
        CK(cudaMalloc(&g.d_ext, probe_need * 4));
        g.probe_cap = probe_need;
    }
    uint32_t still = 0;
    const auto t_begin = std::chrono::steady_clock::now();
    uint32_t hs[5] = {0, 0, 0, 0, 0};
    for (size_t p0 = 0; p0 < sel.size(); p0 += KU) {
        const uint32_t m = (uint32_t)std::min<size_t>(KU, sel.size() - p0), sub = paired ? 2 * m : m;
        uint32_t o = 0;
        for (uint32_t j = 0; j < sub; ++j) {   // sub-batch read j: mate 1 of unit sel[p0 + j], then the mates 2
            const uint32_t k = (j < m) ? sel[p0 + j] : n + sel[p0 + j - m];
            const uint32_t len = s.h_offs[k + 1] - s.h_offs[k];
            g.h_offs[j] = o;
            if (len) CK(cudaMemcpyAsync(g.d_seqs + o, s.d_seqs + s.h_offs[k], len, cudaMemcpyDeviceToDevice, g.stream));
            o += len;
        }
        g.h_offs[sub] = o;
        CK(cudaMemcpyAsync(g.d_offs, g.h_offs, (sub + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, g.stream));
        CK(cudaMemsetAsync(g.d_counters, 0, CT_COUNT * sizeof(uint32_t), g.stream));
        if (second) CK(cudaMemsetAsync(g.d_second, 0, (size_t)sub * sizeof(urmb_second), g.stream));
        DevBatch b = s.batch;
        b.seqs = g.d_seqs;
        b.offs = g.d_offs;
        b.n_reads = sub;
        b.n_units = m;
        DevProbe pr{g.d_tally, g.d_pos, g.d_ext, g.d_view, view_stride_for(b.seqcap)};
        DevOut out{g.d_res, g.d_runs, (uint32_t)g.runs_cap, g.d_counters, g.d_todo, g.d_rescue, second ? g.d_second : nullptr,
                   nullptr, 0u, {nullptr, nullptr}, nullptr, 0u, g.d_rescue};
        const int e = urmb_big_map(&c->ix, &c->P, &b, &pr, &out, g.scratch, urmb_ctx::Big::kWarps, g.pool, 256, g.stream, c->sm_count);
        if (e < 0) return fail(c, URMB_E_CUDA, std::string("big-capacity rerun: ") + cudaGetErrorString((cudaError_t)-e));
        c->launches += (uint64_t)e;
        CK(cudaMemcpyAsync(g.h_counters, g.d_counters, CT_COUNT * sizeof(uint32_t), cudaMemcpyDeviceToHost, g.stream));
        CK(cudaMemcpyAsync(g.h_res, g.d_res, (size_t)sub * sizeof(urmb_result), cudaMemcpyDeviceToHost, g.stream));
        if (second) CK(cudaMemcpyAsync(g.h_second, g.d_second, (size_t)sub * sizeof(urmb_second), cudaMemcpyDeviceToHost, g.stream));
        CK(cudaStreamSynchronize(g.stream));
        const uint32_t bused = std::min<uint32_t>(g.h_counters[CT_RUNS], (uint32_t)g.runs_cap);
        if (bused) {
            CK(cudaMemcpyAsync(g.h_runs, g.d_runs, (size_t)bused * 2, cudaMemcpyDeviceToHost, g.stream));
            CK(cudaStreamSynchronize(g.stream));
            if ((size_t)used + bused > s.h_runs_cap) {   // grow the slot's host run pool, keeping its contents
                uint16_t *nr = nullptr;
                const size_t ncap = ((size_t)used + bused) * 2 + 4096;
                CK(cudaHostAlloc(&nr, ncap * sizeof(uint16_t), cudaHostAllocDefault));
                if (used) memcpy(nr, s.h_runs, (size_t)used * 2);
                cudaFreeHost(s.h_runs);
                s.h_runs = nr;
                s.h_runs_cap = ncap;
            }
            memcpy(s.h_runs + used, g.h_runs, (size_t)bused * 2);
        }
        for (uint32_t j = 0; j < sub; ++j) {
            const uint32_t k = (j < m) ? sel[p0 + j] : n + sel[p0 + j - m];
            urmb_result r = g.h_res[j];
            if (r.path_runs) r.path_off += used;
            if (r.flags & 0x80) ++still;
            s.h_res[k] = r;
            if (second) s.h_second[k] = g.h_second[j];
        }
        used += bused;
        c->rerun_total += sub;
        for (int k = 0; k < 4; ++k) hs[k] += g.h_counters[CT_DBG_HSPS + k];
        hs[4] = std::max(hs[4], g.h_counters[CT_DBG_MAXHSP]);
    }
    if (getenv("URMB_DEBUG"))
        fprintf(stderr, "[urmb] big-capacity rerun of %zu unit(s): %.2f ms on the host; reads by HSP count (<=256, <=512, <=1024, more): %u %u %u %u, max %u\n",
                sel.size(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(), hs[0], hs[1], hs[2], hs[3], hs[4]);
    s.h_counters[CT_OVERFLOW] = still;
    (void)nreads;
    return URMB_OK;
}

extern "C" int urmb_wait(urmb_ctx *c, int si, const urmb_result **res1, const urmb_result **res2, const uint16_t **runs,
                         uint32_t *runs_used) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    Slot &s = c->slots[si];
    if (!s.launched) return fail(c, URMB_E_ARG, "slot not launched");
    CK(cudaSetDevice(c->device));
    if (!s.downloaded) {
        int rc = urmb_download(c, si);
        if (rc) return rc;
    }
    CK(cudaStreamSynchronize(s.copy));
    uint32_t used = s.h_counters[0];
    if (used > s.d_runs_cap) {
        // The runs pool was too small for this batch: grow it and run the batch again (still on the GPU).
        int rc;
        if ((rc = grow_dev(c, s.d_runs, s.d_runs_cap, (size_t)used + 4096))) return rc;
        if ((rc = grow_host(c, s.h_runs, s.h_runs_cap, s.d_runs_cap))) return rc;
        if ((rc = urmb_launch(c, si))) return rc;
        if ((rc = urmb_download(c, si))) return rc;
        CK(cudaStreamSynchronize(s.copy));
        used = s.h_counters[0];
    }
    if (used) {
        CK(cudaMemcpyAsync(s.h_runs, s.d_runs, (size_t)used * 2, cudaMemcpyDeviceToHost, s.copy));
    }
    CK(cudaEventRecord(s.ev_d2h, s.copy));
    CK(cudaStreamSynchronize(s.copy));
    if (c->force_rerun && !s.counted) {   // test hook: every force_rerun-th unit takes the big-capacity path as well
        for (uint32_t u = 0; u < s.batch.n_units; u += c->force_rerun) s.h_res[u].flags |= 0x80;
        s.h_counters[CT_OVERFLOW] += (s.batch.n_units + c->force_rerun - 1) / c->force_rerun;
    }
    if (s.h_counters[CT_OVERFLOW] != 0 && !s.counted && !getenv("URMB_NO_RERUN")) {
        const uint32_t before = s.h_counters[CT_OVERFLOW];
        int rc = rerun_overflowed(c, s, used);
        if (rc) return rc;
        if (getenv("URMB_DEBUG")) fprintf(stderr, "[urmb] slot %d: %u read(s) over a per-mate capacity (hits %u, path runs %u, run pool %u, HSPs %u, path assembly %u) mapped again by the big-capacity build, %u still over\n", si, before, s.h_counters[CT_DBG_OVF], s.h_counters[CT_DBG_OVF + 1], s.h_counters[CT_DBG_OVF + 2], s.h_counters[CT_DBG_OVF + 3], s.h_counters[CT_DBG_OVF + 4], s.h_counters[CT_OVERFLOW]);
    }
    if (getenv("URMB_DEBUG")) fprintf(stderr, "[urmb] slot %d: %u units, %u finished by the first look, %u in the second pass, %u rescued (%u by the legacy kernel, %u full-window DPs), %u path runs\n", si, s.batch.n_units, s.h_counters[CT_FIRST_LOOK], s.h_counters[CT_TODO_TOTAL], s.h_counters[CT_RESCUE], s.h_counters[CT_RESCUE_LEGACY], s.h_counters[CT_RESCUE_DPS], used);
    if (getenv("URMB_DEBUG") && s.batch.paired) {
        fprintf(stderr, "[urmb] slot %d: rescue rounds, pairs stopped at a full-window DP:", si);
        for (int r = 1; r <= kRescueRounds + 1; ++r) fprintf(stderr, " %u", s.h_counters[CT_RQ_COUNT + r]);
        fprintf(stderr, "; pairs by scan windows (<=4, <=16, <=64, <=256, more): %u %u %u %u %u; longest pair %.2f Mticks (%u windows, round %u)\n",
                s.h_counters[CT_DBG_WIN], s.h_counters[CT_DBG_WIN + 1], s.h_counters[CT_DBG_WIN + 2], s.h_counters[CT_DBG_WIN + 3],
                s.h_counters[CT_DBG_WIN + 4], s.h_counters[CT_DBG_MAXT] * 1024.0 / 1e6, s.h_counters[CT_DBG_MAXW] & 0xFFFFFFu,
                s.h_counters[CT_DBG_MAXW] >> 24);
        fprintf(stderr, "[urmb] slot %d: launches of the last step (class:ms):", si);
        for (size_t i = 0; i < s.nkev; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, s.kev[2 * i], s.kev[2 * i + 1]) == cudaSuccess) fprintf(stderr, " %d:%.2f", s.kclass[i], ms);
        }
        cudaGetLastError();
        fprintf(stderr, "\n");
    }
    if (res1) *res1 = s.h_res;
    if (res2) *res2 = s.batch.paired ? s.h_res + s.batch.n_units : nullptr;
    if (runs) *runs = s.h_runs;
    if (runs_used) *runs_used = used;
    for (uint32_t r : s.too_long) s.h_res[r].flags |= 0x40;   // unmapped because the read (or its mate) is too long
    if (!s.counted) { c->unsupported_total += s.too_long.size(); c->overflow_total += s.h_counters[CT_OVERFLOW]; c->first_look_total += s.h_counters[CT_FIRST_LOOK]; s.counted = true; }
    // Reads that exceeded a per-read capacity carry bit 7 in urmb_result.flags and are counted (urmb_overflow_count): the
    // batch itself is valid, so this is not an error (the reference grows its lists without bound, state1.cpp:190).
    return URMB_OK;
}

extern "C" int urmb_unsupported_count(urmb_ctx *c, int si, uint32_t *last, uint64_t *total) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    if (last) *last = (uint32_t)c->slots[si].too_long.size();
    if (total) *total = c->unsupported_total;
    return URMB_OK;
}

extern "C" int urmb_overflow_count(urmb_ctx *c, int si, uint32_t *last, uint64_t *total) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    if (last) *last = c->slots[si].h_counters ? c->slots[si].h_counters[CT_OVERFLOW] : 0;
    if (total) *total = c->overflow_total;
    return URMB_OK;
}

extern "C" int urmb_first_look_count(urmb_ctx *c, int si, uint32_t *last, uint64_t *total) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    if (last) *last = c->slots[si].h_counters ? c->slots[si].h_counters[CT_FIRST_LOOK] : 0;
    if (total) *total = c->first_look_total;
    return URMB_OK;
}

extern "C" int urmb_second_hits(urmb_ctx *c, int si, const urmb_second **s1, const urmb_second **s2) {
    if (!c || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    Slot &s = c->slots[si];
    if (!c->params.want_second) return fail(c, URMB_E_ARG, "context created without want_second");
    if (!s.launched || !s.downloaded || !s.batch.paired) return fail(c, URMB_E_ARG, "no finished paired-end batch in this slot");
    if (s1) *s1 = s.h_second;
    if (s2) *s2 = s.h_second + s.batch.n_units;
    return URMB_OK;
}

extern "C" int urmb_timing_last(urmb_ctx *c, int si, urmb_timing *t) {
    if (!c || !t || si < 0 || si >= URMB_SLOTS) return URMB_E_ARG;
    Slot &s = c->slots[si];
    memset(t, 0, sizeof *t);
    if (!s.launched) return fail(c, URMB_E_ARG, "slot not launched");
    CK(cudaSetDevice(c->device));   // a process that drives several contexts may have another device current
    CK(cudaEventSynchronize(s.ev_k2));
    CK(cudaEventSynchronize(s.ev_rescue));
    cudaEventElapsedTime(&t->probe_ms, s.ev_k0, s.ev_k1);
    cudaEventElapsedTime(&t->search_ms, s.ev_k1, s.ev_k2);
    for (size_t i = 0; i < s.nkev; ++i) {
        float ms = 0.f;
        const int k = s.kclass[i];
        if (k < 0 || k >= URMB_KCLASSES) continue;
        if (cudaEventElapsedTime(&ms, s.kev[2 * i], s.kev[2 * i + 1]) == cudaSuccess) {
            t->kernel_ms[k] += ms;
            t->kernel_launches[k] += 1;
        }
    }
    t->rescue_ms = t->kernel_ms[6] + t->kernel_ms[8] + t->kernel_ms[9] + t->kernel_ms[10];
    if (cudaEventQuery(s.ev_h2d) == cudaSuccess) cudaEventElapsedTime(&t->h2d_ms, s.ev_h2d0, s.ev_h2d);
    if (cudaEventQuery(s.ev_d2h) == cudaSuccess && cudaEventQuery(s.ev_k2) == cudaSuccess)
        cudaEventElapsedTime(&t->d2h_ms, s.ev_k2, s.ev_d2h);
    cudaGetLastError();
    return URMB_OK;
}

extern "C" uint64_t urmb_launch_count(const urmb_ctx *c) { return c ? c->launches : 0; }

static int copy_out(urmb_ctx *c, uint32_t n, const urmb_result *r, urmb_result *out) {
    if (n && out) memcpy(out, r, (size_t)n * sizeof(urmb_result));
    return URMB_OK;
}

extern "C" int urmb_map_se(urmb_ctx *c, const urmb_batch *in, urmb_result *out, uint16_t *runs, uint32_t runs_cap,
                           uint32_t *runs_used) {
    int rc = urmb_submit(c, 0, in, nullptr);
    if (rc) return rc;
    const urmb_result *r1;
    const uint16_t *rr;
    uint32_t used = 0;
    rc = urmb_wait(c, 0, &r1, nullptr, &rr, &used);
    if (rc) return rc;
    copy_out(c, in->n, r1, out);
    if (runs_used) *runs_used = used;
    if (used > runs_cap) return fail(c, URMB_E_OVERFLOW, "caller's runs buffer too small");
    if (used && runs) memcpy(runs, rr, (size_t)used * 2);
    return rc;
}

extern "C" int urmb_map_pe(urmb_ctx *c, const urmb_batch *r1, const urmb_batch *r2, urmb_result *out1, urmb_result *out2,
                           uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used) {
    if (!r2) return URMB_E_ARG;
    int rc = urmb_submit(c, 0, r1, r2);
    if (rc) return rc;
    const urmb_result *a, *b;
    const uint16_t *rr;
    uint32_t used = 0;
    rc = urmb_wait(c, 0, &a, &b, &rr, &used);
    if (rc) return rc;
    copy_out(c, r1->n, a, out1);
    copy_out(c, r1->n, b, out2);
    if (runs_used) *runs_used = used;
    if (used > runs_cap) return fail(c, URMB_E_OVERFLOW, "caller's runs buffer too small");
    if (used && runs) memcpy(runs, rr, (size_t)used * 2);
    return rc;
}
