// urmb_fasta.cu -- FASTA bytes -> SeqData on the device: the concatenated, upper-cased records with 32 '-' bytes between
// them (ufindex.cpp:462-510), byte-identical to UfiBuilder::ReadFasta of urmb_host.cpp (fastaseqsource.cpp:26-112):
//   - lines end at '\n'; every '\r' is dropped;
//   - a header is a line whose first non-'\r' byte is '>'; its label runs from after '>' ('\r' removed) to the first space
//     byte (' ', '\t' ... '\r' -- isspace in the C locale);
//   - before the first header only lines that are empty after '\r' removal may appear ("expected '>' in line N");
//   - a sequence byte is kept when it is an ASCII letter and upper-cased; every other byte is dropped;
//   - records with no kept byte are dropped; the others are joined with 32 '-' bytes, none after the last.
//
// A stream compaction over the raw bytes, one warp per 16 KB tile (32 steps of 32 lanes x 16-byte loads), no atomics and no
// block-wide barriers (so that the warp emulator of tests/emu runs the same kernels):
//   hdr     : header starts per tile (a '>' with only '\r' between it and the previous '\n' or the file start; the look-back
//             may cross the tile border), scanned, then written in file order
//   hdr_end : each header's line end (first '\n' at or after it, or the file length)
//   count   : kept bytes per tile outside the header lines, and for every header the kept bytes of its tile before it
//   scan    : exclusive scan of the tile counts -> K(h_k), the kept bytes before header k: record k keeps K(h_k+1) - K(h_k)
//   (host)  : record table, empty records dropped; nstart[m] = K of the m-th kept record
//   scatter : kept byte number G goes to SeqData[G + 32 m] (m: its kept record), staged per step in shared memory so that
//             the warp writes contiguous bytes
//   pads    : the 32 '-' bytes in front of every kept record but the first
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

#include "urmb_internal.h"

namespace urmb {

#ifndef URMB_LAUNCH
#define URMB_LAUNCH(kern, grid, block, smem, stream, ...) \
    kern<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
#endif

constexpr uint32_t kFaStep = 512;                     // bytes of one warp step (32 lanes x 16)
constexpr uint32_t kFaSteps = 32;
constexpr uint64_t kFaTile = (uint64_t)kFaStep * kFaSteps;   // bytes per warp
constexpr int kFaWarps = 4;                           // warps per block

// Raw bytes are read in whole tiles: the buffer holds len bytes and zero bytes up to fasta_padded_len(len).
inline uint64_t fasta_tiles(uint64_t len) { return (len + kFaTile - 1) / kFaTile; }
uint64_t fasta_padded_len(uint64_t len) { return fasta_tiles(len) * kFaTile + 16; }

struct FastaArgs {
    const uint8_t *fa;    // raw bytes (+ zero padding)
    uint64_t len;
    uint64_t ntiles;
    uint64_t nrec;        // header starts (R); set after the header scan
    uint32_t *tcount;     // [ntiles] per-tile counts (header starts, then kept bytes)
    uint64_t *tscan;      // [ntiles + 1] exclusive scan of tcount
    uint64_t *h;          // [R + 1] header starts, h[R] = len
    uint64_t *e;          // [R] header line ends ('\n' or len)
    uint64_t *hk;         // [R + 1] kept bytes before header k (first within its tile, then file-wide); hk[R] = total
    const uint64_t *nstart;   // [M] kept-byte index of the first byte of each kept record
    uint64_t nkept_rec;   // M
    uint8_t *out;         // SeqData
};

__device__ __forceinline__ void fa_load16(const uint8_t *p, uint32_t w[4]) {
#ifdef URMB_EMU
    memcpy(w, p, 16);
#else
    const uint4 v = __ldg((const uint4 *)p);
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
#endif
}
__device__ __forceinline__ uint32_t fa_byte(const uint32_t w[4], int j) { return (w[j >> 2] >> (8 * (j & 3))) & 0xFFu; }
__device__ __forceinline__ bool fa_alpha(uint32_t c) { return (uint32_t)((c | 0x20u) - 'a') < 26u; }

// '>' at i starts a header: only '\r' lies between it and the previous '\n' or the start of the file
__device__ __forceinline__ bool fa_header_at(const uint8_t *fa, uint64_t i) {
    uint64_t j = i;
    while (j > 0 && fa[j - 1] == '\r') --j;
    return j == 0 || fa[j - 1] == '\n';
}

__device__ __forceinline__ uint32_t fa_warp_incl_scan(uint32_t v, int lane) {
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += u;
    }
    return v;
}

// Pass 1: header starts per tile (WRITE = false), then their positions in file order (WRITE = true).
template <bool WRITE>
__global__ void __launch_bounds__(32 * kFaWarps) fa_hdr_kernel(FastaArgs a) {
    const int lane = (int)(threadIdx.x & 31);
    const uint64_t t = (uint64_t)blockIdx.x * kFaWarps + threadIdx.x / 32;
    if (t >= a.ntiles) return;
    uint64_t rank = WRITE ? a.tscan[t] : 0;
    for (uint32_t s = 0; s < kFaSteps; ++s) {
        const uint64_t p = t * kFaTile + (uint64_t)s * kFaStep + 16u * lane;
        uint32_t w[4];
        fa_load16(a.fa + p, w);
        uint32_t starts = 0;
        for (int j = 0; j < 16; ++j)
            if (fa_byte(w, j) == '>' && p + j < a.len && fa_header_at(a.fa, p + j)) starts |= 1u << j;
        const uint32_t n = (uint32_t)__popc(starts);
        const uint32_t incl = fa_warp_incl_scan(n, lane);
        if (WRITE) {
            uint64_t r = rank + incl - n;
            for (uint32_t m = starts; m; m &= m - 1) a.h[r++] = p + (uint64_t)(__ffs(m) - 1);
        }
        rank += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (!WRITE && lane == 0) a.tcount[t] = (uint32_t)rank;
}

// Line end of every header; h[R] = len closes the last record.
__global__ void fa_hdr_end_kernel(FastaArgs a) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k == a.nrec) a.h[k] = a.len;
    if (k >= a.nrec) return;
    uint64_t i = a.h[k];
    while (i < a.len && a.fa[i] != '\n') ++i;
    a.e[k] = i;
}

// Kept-byte mask of the 16 bytes at p.  k: first header whose line ends at or after p (advanced here; monotone per lane).
// h0: the first header (bytes before it are never kept).
__device__ __forceinline__ uint32_t fa_kept_mask(const FastaArgs &a, const uint32_t w[4], uint64_t p, uint64_t h0, uint64_t &k,
                                                 uint64_t &hs, uint64_t &he) {
    uint32_t mask = 0;
    for (int j = 0; j < 16; ++j) {
        const uint64_t i = p + j;
        while (i > he && k < a.nrec) {   // past the current header line: on to the next
            ++k;
            hs = a.h[k];
            he = k < a.nrec ? a.e[k] : ~0ull;
        }
        const bool in_hdr = i >= hs && i <= he;
        if (fa_alpha(fa_byte(w, j)) && !in_hdr && i >= h0 && i < a.len) mask |= 1u << j;
    }
    return mask;
}

// First header whose line ends at or after p (lower bound over e).
__device__ __forceinline__ uint64_t fa_first_header(const FastaArgs &a, uint64_t p) {
    uint64_t lo = 0, hi = a.nrec;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) / 2;
        if (a.e[mid] < p) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Pass 2: kept bytes per tile; hk[k] = kept bytes of the tile before header k.
__global__ void __launch_bounds__(32 * kFaWarps) fa_count_kernel(FastaArgs a) {
    const int lane = (int)(threadIdx.x & 31);
    const uint64_t t = (uint64_t)blockIdx.x * kFaWarps + threadIdx.x / 32;
    if (t >= a.ntiles) return;
    uint64_t k = fa_first_header(a, t * kFaTile);
    uint64_t hs = a.h[k], he = k < a.nrec ? a.e[k] : ~0ull;
    const uint64_t h0 = a.h[0];
    uint32_t run = 0;
    for (uint32_t s = 0; s < kFaSteps; ++s) {
        const uint64_t p = t * kFaTile + (uint64_t)s * kFaStep + 16u * lane;
        uint32_t w[4];
        fa_load16(a.fa + p, w);
        const uint64_t k0 = k;
        const uint32_t mask = fa_kept_mask(a, w, p, h0, k, hs, he);
        const uint32_t n = (uint32_t)__popc(mask);
        const uint32_t incl = fa_warp_incl_scan(n, lane);
        for (uint64_t q = k0; q < a.nrec && a.h[q] < p + 16; ++q)   // headers that start in these 16 bytes
            if (a.h[q] >= p) a.hk[q] = run + incl - n + (uint32_t)__popc(mask & ((1u << (a.h[q] - p)) - 1u));
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) a.tcount[t] = run;
}

// Exclusive scan of n counts by one warp: out[i] = in[0] + ... + in[i-1], out[n] = total.
__global__ void fa_scan_kernel(const uint32_t *in, uint64_t *out, uint64_t n) {
    const int lane = (int)(threadIdx.x & 31);
    uint64_t base = 0;
    for (uint64_t o = 0; o < n; o += 32 * 4) {
        uint32_t v[4], sum = 0;
        for (int j = 0; j < 4; ++j) {
            const uint64_t i = o + 4u * lane + j;
            v[j] = i < n ? in[i] : 0u;
            sum += v[j];
        }
        const uint32_t incl = fa_warp_incl_scan(sum, lane);   // < 2^32: 128 tiles of 16 KB
        uint64_t run = base + incl - sum;
        for (int j = 0; j < 4; ++j) {
            const uint64_t i = o + 4u * lane + j;
            if (i < n) out[i] = run;
            run += v[j];
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) out[n] = base;
}

// K(h_k): kept bytes before header k, file-wide; hk[R] = all kept bytes.
__global__ void fa_rec_kernel(FastaArgs a) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < a.nrec) a.hk[k] += a.tscan[a.h[k] / kFaTile];
    if (k == a.nrec) a.hk[k] = a.tscan[a.ntiles];
}

// Pass 3: kept byte number G (upper-cased) goes to out[G + 32 m], m = the kept record it belongs to.
__global__ void __launch_bounds__(32 * kFaWarps) fa_scatter_kernel(FastaArgs a) {
    __shared__ uint8_t stage[kFaWarps][kFaStep];
    const int lane = (int)(threadIdx.x & 31), wib = (int)(threadIdx.x / 32);
    const uint64_t t = (uint64_t)blockIdx.x * kFaWarps + wib;
    if (t >= a.ntiles) return;
    uint8_t *st = stage[wib];
    uint64_t k = fa_first_header(a, t * kFaTile);
    uint64_t hs = a.h[k], he = k < a.nrec ? a.e[k] : ~0ull;
    const uint64_t h0 = a.h[0];
    uint64_t G = a.tscan[t];
    uint64_t m = 0;   // last kept record whose first kept byte is at or before G
    {
        uint64_t lo = 0, hi = a.nkept_rec;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) / 2;
            if (a.nstart[mid] <= G) lo = mid + 1;
            else hi = mid;
        }
        m = lo ? lo - 1 : 0;
    }
    for (uint32_t s = 0; s < kFaSteps; ++s) {
        const uint64_t p = t * kFaTile + (uint64_t)s * kFaStep + 16u * lane;
        uint32_t w[4];
        fa_load16(a.fa + p, w);
        const uint32_t mask = fa_kept_mask(a, w, p, h0, k, hs, he);
        const uint32_t n = (uint32_t)__popc(mask);
        const uint32_t incl = fa_warp_incl_scan(n, lane);
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t o = incl - n;
        for (uint32_t b = mask; b; b &= b - 1) st[o++] = (uint8_t)(fa_byte(w, __ffs(b) - 1) & 0xDFu);
        __syncwarp();
        for (uint32_t j = lane; j < total; j += 32) {
            const uint64_t g = G + j;
            while (m + 1 < a.nkept_rec && a.nstart[m + 1] <= g) ++m;
            a.out[g + 32 * m] = st[j];
        }
        __syncwarp();
        G += total;
    }
}

// The 32 '-' bytes in front of kept record m >= 1.
__global__ void fa_pad_kernel(FastaArgs a) {
    const uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m == 0 || m >= a.nkept_rec) return;
    memset(a.out + a.nstart[m] + 32 * m - 32, '-', 32);
}

// ---- host side, shared by the device path (urmb_api.cu) and the emulator (tests/emu) ----

static inline bool fa_space(uint8_t c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// Lines before the first header (at first) must be empty after '\r' removal: "" or the message of the host parser.
std::string fasta_check_head(const uint8_t *fa, uint64_t first) {
    uint64_t line = 1;
    for (uint64_t i = 0; i < first; ++i) {
        if (fa[i] == '\n') ++line;
        else if (fa[i] != '\r') return "expected '>' in line " + std::to_string(line);
    }
    return std::string();
}

// h[0..R] (h[R] = len), e[0..R), K[0..R] (K[R] = all kept bytes) -> table; "" or an error message.
std::string fasta_table(const uint8_t *fa, const uint64_t *h, const uint64_t *e, const uint64_t *K, uint64_t R,
                               FastaTable &t) {
    t = FastaTable();
    for (uint64_t k = 0; k < R; ++k) {
        std::string lab;
        for (uint64_t i = h[k] + 1; i < e[k]; ++i) {
            if (fa[i] == '\r') continue;
            if (fa_space(fa[i])) break;
            lab.push_back((char)fa[i]);
        }
        const uint64_t n = K[k + 1] - K[k];
        if (n == 0) { t.dropped.push_back(lab); continue; }
        if (!t.nstart.empty()) t.seq_size += 32;
        if (t.seq_size + n > (uint64_t)UINT32_MAX - URMB_SEQ_PAD) return "genome larger than SeqData can address (4 GB)";
        t.labels.push_back(lab);
        t.lengths.push_back((uint32_t)n);
        t.offsets.push_back((uint32_t)t.seq_size);
        t.nstart.push_back(K[k]);
        t.seq_size += n;
    }
    return std::string();
}

}  // namespace urmb

#ifndef URMB_EMU
namespace urmb {

int fasta_parse_device(const uint8_t *d_fa, const uint8_t *h_fa, uint64_t len, void *stream, void **d_seq, FastaTable &tab,
                       float *kernel_ms, std::string &err) {
    cudaStream_t st = (cudaStream_t)stream;
    *d_seq = nullptr;
    FastaArgs a{};
    a.fa = d_fa;
    a.len = len;
    a.ntiles = fasta_tiles(len);
    cudaEvent_t ev[2] = {nullptr, nullptr};
    std::vector<uint64_t> h, e, K;
    int rc = URMB_E_CUDA;
    const unsigned blocks = (unsigned)((a.ntiles + kFaWarps - 1) / kFaWarps);
    auto grid = [](uint64_t n) { return (unsigned)(n / 256 + 1); };
    cudaError_t ce = cudaSuccess;
#define FCK(call)                                                                           \
    do {                                                                                    \
        if ((ce = (call)) != cudaSuccess) { err = std::string(#call) + ": " + cudaGetErrorString(ce); goto done; } \
    } while (0)
    FCK(cudaEventCreate(&ev[0]));
    FCK(cudaEventCreate(&ev[1]));
    FCK(cudaEventRecord(ev[0], st));
    FCK(cudaMalloc(&a.tcount, (a.ntiles + 1) * 4));
    FCK(cudaMalloc(&a.tscan, (a.ntiles + 1) * 8));
    if (a.ntiles) URMB_LAUNCH(fa_hdr_kernel<false>, blocks, 32 * kFaWarps, 0, st, a);
    URMB_LAUNCH(fa_scan_kernel, 1, 32, 0, st, a.tcount, a.tscan, a.ntiles);
    FCK(cudaGetLastError());
    FCK(cudaMemcpyAsync(&a.nrec, a.tscan + a.ntiles, 8, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    FCK(cudaMalloc(&a.h, (a.nrec + 1) * 8));
    FCK(cudaMalloc(&a.e, (a.nrec + 1) * 8));
    FCK(cudaMalloc(&a.hk, (a.nrec + 1) * 8));
    if (a.ntiles) URMB_LAUNCH(fa_hdr_kernel<true>, blocks, 32 * kFaWarps, 0, st, a);
    URMB_LAUNCH(fa_hdr_end_kernel, grid(a.nrec), 256, 0, st, a);
    if (a.ntiles) URMB_LAUNCH(fa_count_kernel, blocks, 32 * kFaWarps, 0, st, a);
    URMB_LAUNCH(fa_scan_kernel, 1, 32, 0, st, a.tcount, a.tscan, a.ntiles);
    URMB_LAUNCH(fa_rec_kernel, grid(a.nrec), 256, 0, st, a);
    FCK(cudaGetLastError());
    h.resize(a.nrec + 1);
    e.resize(a.nrec + 1);
    K.resize(a.nrec + 1);
    FCK(cudaMemcpyAsync(h.data(), a.h, (a.nrec + 1) * 8, cudaMemcpyDeviceToHost, st));
    FCK(cudaMemcpyAsync(e.data(), a.e, a.nrec * 8, cudaMemcpyDeviceToHost, st));
    FCK(cudaMemcpyAsync(K.data(), a.hk, (a.nrec + 1) * 8, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    err = fasta_check_head(h_fa, h[0]);
    if (!err.empty()) { rc = URMB_E_IO; goto done; }
    err = fasta_table(h_fa, h.data(), e.data(), K.data(), a.nrec, tab);
    if (!err.empty()) { rc = URMB_E_UNSUPPORTED; goto done; }
    if (tab.nstart.empty()) { err = "no sequence in the FASTA data"; rc = URMB_E_IO; goto done; }
    a.nkept_rec = tab.nstart.size();
    {
        uint64_t *d_nstart = nullptr;
        FCK(cudaMalloc(&d_nstart, a.nkept_rec * 8));
        a.nstart = d_nstart;
        FCK(cudaMemcpyAsync(d_nstart, tab.nstart.data(), a.nkept_rec * 8, cudaMemcpyHostToDevice, st));
        FCK(cudaMalloc(d_seq, tab.seq_size + URMB_SEQ_PAD));
        a.out = (uint8_t *)*d_seq;
        FCK(cudaMemsetAsync(a.out + tab.seq_size, 0, URMB_SEQ_PAD, st));
        if (a.ntiles) URMB_LAUNCH(fa_scatter_kernel, blocks, 32 * kFaWarps, 0, st, a);
        URMB_LAUNCH(fa_pad_kernel, grid(a.nkept_rec), 256, 0, st, a);
        FCK(cudaGetLastError());
        FCK(cudaEventRecord(ev[1], st));
        FCK(cudaEventSynchronize(ev[1]));
        if (kernel_ms) cudaEventElapsedTime(kernel_ms, ev[0], ev[1]);
    }
    rc = URMB_OK;
done:
#undef FCK
    if (rc != URMB_OK && ce != cudaSuccess) rc = ce == cudaErrorMemoryAllocation ? URMB_E_NOMEM : URMB_E_CUDA;
    cudaStreamSynchronize(st);
    cudaFree(a.tcount); cudaFree(a.tscan); cudaFree(a.h); cudaFree(a.e); cudaFree(a.hk); cudaFree((void *)a.nstart);
    if (rc != URMB_OK) { cudaFree(*d_seq); *d_seq = nullptr; }
    for (cudaEvent_t x : ev) if (x) cudaEventDestroy(x);
    return rc;
}

}  // namespace urmb
#endif
