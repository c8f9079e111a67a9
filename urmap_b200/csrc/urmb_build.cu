// urmb_build.cu -- device-side UFI index construction (the "-make_ufi on GPU" row of SURVEY.md §8f).
//
// The reference builder (UFIndex::MakeIndex, ufindex.cpp:83-151) is sequential: k-mers are inserted in genome
// order and overflow list elements go to the first free never-owned slot after the end of their list
// (FindFreeSlot, ufindex.cpp:987), so *where* overflow elements land depends on insertion order.  What a
// mapper can observe, however, is only (a) each owned slot's head tally class (BOTH1 / PLUS1 / list) and
// (b) the positions of its list in genome order (GetRow_Blob, ufindex.cpp:883); slots that merely store
// another slot's overflow read as "other" and FREE slots read as FREE, and both are skipped identically
// (search1m6.cpp:172, getseed.cpp:22).  This builder reproduces (a) and (b) exactly -- same counts
// (CountSlots / CountSlots_Minus, ufindex.cpp:338,373), same "indexed iff 1<=n<=MaxIx and m<=MaxIx" rule
// (UpdateSlot, ufindex.cpp:208), same list order, same link encoding incl. long links -- but places overflow
// elements by parallel claiming, so the blob is functionally equivalent, not byte-identical.  The
// byte-identical sequential builder lives in the host CLI (urmb_host.cpp).
//
// Passes (all thread-per-element, HBM-bound):
//   init   : every slot := {FREE, 0xFFFFFFFF}
//   count  : saturating 8-bit counts per slot for plus- and minus-strand k-mers (CAS on packed bytes)
//   scan   : exclusive prefix sum of list lengths over indexed slots -> pool offsets (two-level)
//   scatter: positions of indexed k-mers -> pool[base[slot] + ticket]
//   heads  : per indexed slot: sort its <= MaxIx positions (genome order), write the head record
//   carry  : q(s) by a two-level max-plus scan -> bitmap of segment borders (q(s) == 0)
//   segment: one thread per segment replays UpdateSlot (ufindex.cpp:194-322) for its overflow elements in genome order
//   repair : segments that need a long link, replayed with the segments they spill into
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "urmb_internal.h"

namespace urmb {

#ifndef URMB_EMU
#define URMB_LAUNCH(kern, grid, block, smem, stream, ...) \
    kern<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
#endif

constexpr uint8_t BT_FREE = 0, BT_END = 127, BT_MY_BIT = 128, BT_PLUS1 = 254, BT_BOTH1 = 255, BT_LONG = 125;
constexpr uint32_t BT_MAX_NEXT = 124, BT_MAX_LINK = 0xffff;

struct BuildArgs {
    const uint8_t *seq;     // upper-case genome incl. '-' pads
    uint64_t seq_size;
    uint64_t slot_count, magic, shift_mask;
    uint32_t word_len, max_ix;
    uint8_t *blob;
    uint32_t *cntP, *cntM;  // packed 8-bit saturating counters
    uint32_t *fill;         // packed 8-bit tickets
    uint32_t *base;         // pool offset per slot
    uint64_t *blocksum;     // per scan block
    uint32_t *pool;
    uint8_t *qzero;         // bit s: q(s) == 0, nothing is carried from slot s to slot s+1 (segment border)
    int64_t *blockA, *blockB;   // per scan block: composite f(q) = max(A, q + B) of its slots
    int64_t *blockQ;        // q entering each scan block
    uint32_t *errors;       // [0] segments handed to the repair pass, [1] pool overflow, [2] truncated lists / repair gave up,
                            // [3] segments beyond the capacity of the repair list (the blob is then not valid either)
    uint64_t *flagged;      // start slots of the segments handed to the repair pass
    uint32_t flagged_cap;
};

__device__ __forceinline__ uint32_t bletter(uint32_t c) {  // genome is already upper case (ufindex.cpp:466)
    uint32_t u = c & 0xDFu, r = 0xFFu;
    if (u == 'A') r = 0;
    else if (u == 'C') r = 1;
    else if (u == 'G') r = 2;
    else if (u == 'T' || u == 'U') r = 3;
    return r;
}
__device__ __forceinline__ uint64_t bmurmur(uint64_t h) {
    h ^= (h >> 33); h *= 0xff51afd7ed558ccdULL; h ^= (h >> 33); h *= 0xc4ceb9fe1a85ec53ULL; h ^= (h >> 33);
    return h;
}
__device__ __forceinline__ uint64_t bslot(uint64_t word, const BuildArgs &a) {
    uint64_t h = bmurmur(word & a.shift_mask);
    uint64_t q = __umul64hi(h, a.magic);
    uint64_t r = h - q * a.slot_count;
    if (r >= a.slot_count) r -= a.slot_count;
    return r;
}
__device__ __forceinline__ uint32_t cnt_get(const uint32_t *c, uint64_t s) { return (c[s >> 2] >> ((s & 3) * 8)) & 255u; }

__device__ __forceinline__ void sat_inc(uint32_t *c, uint64_t s) {
    uint32_t *w = c + (s >> 2);
    const uint32_t sh = (uint32_t)(s & 3) * 8;
    uint32_t old = *w;
    for (;;) {
        if (((old >> sh) & 255u) == 255u) return;
        uint32_t assumed = old;
        old = atomicCAS(w, assumed, assumed + (1u << sh));
        if (old == assumed) return;
    }
}

// words of the k-mer starting at p on both strands; false if any letter is invalid
__device__ __forceinline__ bool kmer_words(const BuildArgs &a, uint64_t p, uint64_t &fw, uint64_t &rc) {
    fw = 0;
    rc = 0;
    const uint32_t W = a.word_len;
    for (uint32_t t = 0; t < W; ++t) {
        uint32_t l = bletter(a.seq[p + t]);
        if (l > 3) return false;
        fw = (fw << 2) | l;
        rc |= (uint64_t)(3u - l) << (2 * t);
    }
    return true;
}

__global__ void build_init_kernel(BuildArgs a) {
    // 4 records (20 bytes = 5 words) per thread
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t ngroups = (a.slot_count + 3) / 4;
    if (g >= ngroups) return;
    const uint64_t nbytes = 5 * a.slot_count;
    uint8_t *p = a.blob + g * 20;
    if (g * 20 + 20 <= nbytes) {
        uint32_t *w = reinterpret_cast<uint32_t *>(p);
        w[0] = 0xFFFFFF00u; w[1] = 0xFFFF00FFu; w[2] = 0xFF00FFFFu; w[3] = 0x00FFFFFFu; w[4] = 0xFFFFFFFFu;
    } else {
        for (uint64_t i = g * 20; i < nbytes; ++i) a.blob[i] = (i % 5 == 0) ? 0 : 0xFF;
    }
}

__global__ void build_count_kernel(BuildArgs a) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p + a.word_len > a.seq_size) return;
    uint64_t fw, rc;
    if (!kmer_words(a, p, fw, rc)) return;
    sat_inc(a.cntP, bslot(fw, a));
    sat_inc(a.cntM, bslot(rc, a));
}

__device__ __forceinline__ uint32_t list_len(const BuildArgs &a, uint64_t s) {  // 0 if the slot is not indexed
    uint32_t n = cnt_get(a.cntP, s), m = cnt_get(a.cntM, s);
    return (n >= 1 && n <= a.max_ix && m <= a.max_ix) ? n : 0;
}

constexpr int kScanBlock = 2048;  // slots per scan block, 256 threads x 8

__global__ void build_blocksum_kernel(BuildArgs a) {
    __shared__ uint32_t red[256];
    const uint64_t s0 = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)threadIdx.x * 8;
    uint32_t sum = 0;
    for (int k = 0; k < 8; ++k) {
        uint64_t s = s0 + k;
        if (s < a.slot_count) sum += list_len(a, s);
    }
    red[threadIdx.x] = sum;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
        if ((int)threadIdx.x < st) red[threadIdx.x] += red[threadIdx.x + st];
        __syncthreads();
    }
    if (threadIdx.x == 0) a.blocksum[blockIdx.x] = red[0];
}

// single CTA: exclusive scan of blocksum in place
__global__ void build_scan_blocksums_kernel(BuildArgs a, uint64_t nblocks) {
    __shared__ uint64_t part[1024];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint64_t b0 = 0; b0 < nblocks; b0 += 1024) {
        uint64_t i = b0 + threadIdx.x;
        uint64_t v = (i < nblocks) ? a.blocksum[i] : 0;
        part[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            uint64_t t = ((int)threadIdx.x >= off) ? part[threadIdx.x - off] : 0;
            __syncthreads();
            part[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nblocks) a.blocksum[i] = carry + part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += part[1023];
        __syncthreads();
    }
}

__global__ void build_base_kernel(BuildArgs a) {
    __shared__ uint32_t part[256];
    const uint64_t s0 = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)threadIdx.x * 8;
    uint32_t len[8], sum = 0;
    for (int k = 0; k < 8; ++k) {
        uint64_t s = s0 + k;
        len[k] = (s < a.slot_count) ? list_len(a, s) : 0;
        sum += len[k];
    }
    part[threadIdx.x] = sum;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {
        uint32_t t = ((int)threadIdx.x >= off) ? part[threadIdx.x - off] : 0;
        __syncthreads();
        part[threadIdx.x] += t;
        __syncthreads();
    }
    uint64_t run = a.blocksum[blockIdx.x] + part[threadIdx.x] - sum;
    for (int k = 0; k < 8; ++k) {
        uint64_t s = s0 + k;
        if (s < a.slot_count) a.base[s] = (uint32_t)run;
        run += len[k];
    }
}

__global__ void build_scatter_kernel(BuildArgs a) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p + a.word_len > a.seq_size) return;
    uint64_t fw, rc;
    if (!kmer_words(a, p, fw, rc)) return;
    const uint64_t s = bslot(fw, a);
    const uint32_t n = list_len(a, s);
    if (n == 0) return;
    const uint32_t sh = (uint32_t)(s & 3) * 8;
    const uint32_t old = atomicAdd(a.fill + (s >> 2), 1u << sh);
    const uint32_t r = (old >> sh) & 255u;
    if (r >= n) { atomicAdd(a.errors + 1, 1u); return; }
    a.pool[(uint64_t)a.base[s] + r] = (uint32_t)p;
}

__device__ __forceinline__ void put_rec(uint8_t *blob, uint64_t slot, uint8_t tally, uint32_t pos) {
    uint8_t *p = blob + 5 * slot;
    p[0] = tally;
    p[1] = (uint8_t)pos; p[2] = (uint8_t)(pos >> 8); p[3] = (uint8_t)(pos >> 16); p[4] = (uint8_t)(pos >> 24);
}

__device__ __forceinline__ uint32_t get_tally(const uint8_t *blob, uint64_t slot) { return blob[5 * slot]; }
__device__ __forceinline__ uint32_t get_pos(const uint8_t *blob, uint64_t slot) {
    const uint8_t *p = blob + 5 * slot;
    return (uint32_t)p[1] | ((uint32_t)p[2] << 8) | ((uint32_t)p[3] << 16) | ((uint32_t)p[4] << 24);
}
__device__ __forceinline__ bool in_U(const BuildArgs &a, uint64_t s) {   // FindFreeSlot's "will never be owned"
    const uint32_t n = cnt_get(a.cntP, s);
    return !(n > 0 && n <= a.max_ix);
}
__device__ __forceinline__ uint32_t arrivals(const BuildArgs &a, uint64_t s) {
    const uint32_t n = list_len(a, s);
    return n >= 2 ? n - 1 : 0;
}

// heads: sort the slot's positions into genome order (UpdateSlot is called in genome order) and write the head record
// (ufindex.cpp:217-234); the ticket byte is turned into "elements still to insert".
__global__ void build_heads_kernel(BuildArgs a) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.slot_count) return;
    const uint32_t n = list_len(a, s);
    if (n == 0) return;
    const uint64_t b = a.base[s];
    uint32_t first;
    if (n <= 32) {
        uint32_t pos[32];
        for (uint32_t i = 0; i < n; ++i) {
            uint32_t v = a.pool[b + i];
            int j = (int)i - 1;
            while (j >= 0 && pos[j] > v) { pos[j + 1] = pos[j]; --j; }
            pos[j + 1] = v;
        }
        for (uint32_t i = 0; i < n; ++i) a.pool[b + i] = pos[i];
        first = pos[0];
    } else {   // -maxix above 32: sorted in place
        uint32_t *pos = a.pool + b;
        for (uint32_t i = 1; i < n; ++i) {
            const uint32_t v = pos[i];
            int j = (int)i - 1;
            while (j >= 0 && pos[j] > v) { pos[j + 1] = pos[j]; --j; }
            pos[j + 1] = v;
        }
        first = pos[0];
    }
    put_rec(a.blob, s, (n == 1 && cnt_get(a.cntM, s) == 0) ? BT_BOTH1 : BT_PLUS1, first);
    atomicSub(a.fill + (s >> 2), 1u << ((uint32_t)(s & 3) * 8));
}

// carry, level 1: composite of one scan block.  f_s(q) = max(0, q - u(s)) + a(s) = max(a(s), q + a(s) - u(s)).
constexpr int64_t kNegInf = -(1ll << 60);
struct MaxPlus { int64_t A, B; };
__device__ __forceinline__ MaxPlus mp_then(const MaxPlus &f, const MaxPlus &g) {   // apply f, then g
    MaxPlus r;
    const int64_t t = f.A + g.B;
    r.A = g.A > t ? g.A : t;
    r.B = f.B + g.B;
    return r;
}
__device__ __forceinline__ MaxPlus mp_slot(const BuildArgs &a, uint64_t s) {
    const int64_t ar = arrivals(a, s), u = in_U(a, s) ? 1 : 0;
    return MaxPlus{ar, ar - u};
}
#ifndef URMB_EMU
__global__ void build_carry_block_kernel(BuildArgs a) {
    __shared__ MaxPlus red[256];
    const uint64_t s0 = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)threadIdx.x * 8;
    MaxPlus f{kNegInf, 0};
    for (int k = 0; k < 8; ++k)
        if (s0 + k < a.slot_count) f = mp_then(f, mp_slot(a, s0 + k));
    red[threadIdx.x] = f;
    __syncthreads();
    for (int st = 1; st < 256; st <<= 1) {   // ordered tree: thread i (multiple of 2*st) absorbs its right neighbour
        if ((threadIdx.x & (2 * st - 1)) == 0) red[threadIdx.x] = mp_then(red[threadIdx.x], red[threadIdx.x + st]);
        __syncthreads();
    }
    if (threadIdx.x == 0) { a.blockA[blockIdx.x] = red[0].A; a.blockB[blockIdx.x] = red[0].B; }
}
// carry, level 2 (one CTA): q entering every scan block.  Each thread composes a contiguous range of block composites,
// thread 0 chains the 1024 range composites -- twice, because the table is a ring: the second round starts from the
// carry that leaves the last block -- and every thread then walks its range again with its entry value.
__global__ void __launch_bounds__(1024) build_carry_top_kernel(BuildArgs a, uint64_t nblocks) {
    __shared__ MaxPlus part[1024];
    __shared__ int64_t entry[1024];
    const uint64_t per = (nblocks + 1023) / 1024;
    const uint64_t lo = (uint64_t)threadIdx.x * per, hi = lo + per < nblocks ? lo + per : nblocks;
    MaxPlus f{kNegInf, 0};
    for (uint64_t b = lo; b < hi; ++b) f = mp_then(f, MaxPlus{a.blockA[b], a.blockB[b]});
    part[threadIdx.x] = f;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t q = 0;
        for (int round = 0; round < 2; ++round)
            for (int t = 0; t < 1024; ++t) {
                entry[t] = q;
                const int64_t v = q + part[t].B;
                q = part[t].A > v ? part[t].A : v;
            }
    }
    __syncthreads();
    int64_t q = entry[threadIdx.x];
    for (uint64_t b = lo; b < hi; ++b) {
        a.blockQ[b] = q;
        const int64_t v = q + a.blockB[b];
        q = a.blockA[b] > v ? a.blockA[b] : v;
    }
}
// carry, level 3: q at every slot -> border bitmap (one byte per thread: its 8 slots)
__global__ void build_carry_apply_kernel(BuildArgs a) {
    __shared__ MaxPlus sc[256];
    const uint64_t s0 = (uint64_t)blockIdx.x * kScanBlock + (uint64_t)threadIdx.x * 8;
    MaxPlus f{kNegInf, 0};
    for (int k = 0; k < 8; ++k)
        if (s0 + k < a.slot_count) f = mp_then(f, mp_slot(a, s0 + k));
    sc[threadIdx.x] = f;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {   // inclusive scan of the composites, left to right
        MaxPlus t = sc[threadIdx.x];
        if ((int)threadIdx.x >= off) t = mp_then(sc[threadIdx.x - off], t);
        __syncthreads();
        sc[threadIdx.x] = t;
        __syncthreads();
    }
    int64_t q = a.blockQ[blockIdx.x];
    if (threadIdx.x > 0) {
        const MaxPlus p = sc[threadIdx.x - 1];
        const int64_t t = q + p.B;
        q = p.A > t ? p.A : t;
    }
    uint32_t bits = 0;
    for (int k = 0; k < 8; ++k) {
        const uint64_t s = s0 + k;
        if (s >= a.slot_count) break;
        const MaxPlus m = mp_slot(a, s);
        const int64_t t = q + m.B;
        q = m.A > t ? m.A : t;
        if (q == 0) bits |= 1u << k;
    }
    if (s0 < a.slot_count) a.qzero[s0 >> 3] = (uint8_t)bits;
}
#endif

__device__ __forceinline__ bool q_is_zero(const BuildArgs &a, uint64_t s) { return (a.qzero[s >> 3] >> (s & 7)) & 1u; }
__device__ __forceinline__ uint64_t next_slot(const BuildArgs &a, uint64_t s) { return s + 1 == a.slot_count ? 0 : s + 1; }

__device__ __forceinline__ void flag_segment(const BuildArgs &a, uint64_t s) {
    const uint32_t i = atomicAdd(a.errors, 1u);
    if (i < a.flagged_cap) a.flagged[i] = s;
    else atomicAdd(a.errors + 3, 1u);   // flag buffer full: not a truncation -- its own count and message
}

// segment: thread s owns the segment that starts at s when s has overflow elements and nothing is carried into s.
// It replays UFIndex::UpdateSlot (ufindex.cpp:194-322) for the overflow elements of every list whose head lies in
// the segment, in genome order, with FindEndOfList (ufindex.cpp:945-985) and FindFreeSlot (:987-1000) on the blob.
__global__ void build_segment_kernel(BuildArgs a) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.slot_count) return;
    if (arrivals(a, s) == 0) return;
    if (!q_is_zero(a, s == 0 ? a.slot_count - 1 : s - 1)) return;
    // extent: up to and including the first slot e with q(e) == 0 (a whole ring of carried elements cannot happen:
    // then no slot would start a segment)
    uint64_t len = 1;
    for (uint64_t t = s; !q_is_zero(a, t); t = next_slot(a, t)) ++len;
    for (;;) {
        // the list with the smallest next genome position
        uint64_t best = 0, t = s;
        uint32_t bestpos = 0xFFFFFFFFu;
        bool any = false;
        for (uint64_t i = 0; i < len; ++i, t = next_slot(a, t)) {
            const uint32_t n = list_len(a, t);
            if (n < 2) continue;
            const uint32_t left = (a.fill[t >> 2] >> ((uint32_t)(t & 3) * 8)) & 255u;
            if (left == 0) continue;
            const uint32_t p = a.pool[(uint64_t)a.base[t] + (n - left)];
            if (!any || p < bestpos) { any = true; best = t; bestpos = p; }
        }
        if (!any) return;
        atomicSub(a.fill + (best >> 2), 1u << ((uint32_t)(best & 3) * 8));
        // FindEndOfList
        uint64_t eol = best;
        for (;;) {
            const uint32_t T = get_tally(a.blob, eol);
            if (T == BT_PLUS1 || T == BT_BOTH1 || T == BT_END) break;
            if (T == 253 || T == BT_LONG) { flag_segment(a, s); return; }   // long link: the repair pass handles it
            eol += T & 127u;
            if (eol >= a.slot_count) eol -= a.slot_count;
        }
        // FindFreeSlot, bounded by the segment (beyond it the one-slot-per-element count would be violated)
        uint64_t fs = eol;
        uint32_t step = 0;
        bool border = q_is_zero(a, eol);   // nothing may be carried out of the segment's last slot
        for (;;) {
            if (border) { flag_segment(a, s); return; }
            fs = next_slot(a, fs);
            ++step;
            if (in_U(a, fs) && get_tally(a.blob, fs) == BT_FREE) break;
            border = q_is_zero(a, fs);
        }
        if (step > BT_MAX_NEXT) { flag_segment(a, s); return; }   // a long link takes two U-slots: repair pass
        // ufindex.cpp:303-313
        a.blob[5 * eol] = (uint8_t)((get_tally(a.blob, eol) & BT_MY_BIT) | step);
        put_rec(a.blob, fs, BT_END, bestpos);
    }
}

// repair: the few segments in which an element needs a LONG LINK (probe distance > 124: two U-slots, ufindex.cpp:256-300).
// The extra slot breaks the one-slot-per-element count, so such a segment may spill over its border.  One thread takes
// the flagged segments in slot order: the region (whole segments, starting with the flagged one) is reset to its heads
// and replayed with the complete UpdateSlot; whenever a probe would leave the region, the next segment is added and the
// region is replayed again.  Lists that would have to be truncated (no free slot within 65534) are counted in errors[2].
__device__ uint64_t segment_end(const BuildArgs &a, uint64_t t) {
    while (!q_is_zero(a, t)) t = next_slot(a, t);
    return t;
}
__device__ __forceinline__ void set_left(const BuildArgs &a, uint64_t t, uint32_t v) {
    uint32_t *w = a.fill + (t >> 2);
    const uint32_t sh = (uint32_t)(t & 3) * 8;
    *w = (*w & ~(255u << sh)) | (v << sh);
}
// FindFreeSlot from `from`; returns the step or 0 (none within 65534) and sets `left_region` when the walk would pass `end`
__device__ uint32_t repair_find_free(const BuildArgs &a, uint64_t from, uint64_t end, uint64_t &slot_out, bool &left_region) {
    uint64_t t = from;
    for (uint32_t step = 1; step < BT_MAX_LINK; ++step) {
        if (t == end) { left_region = true; return 0; }
        t = next_slot(a, t);
        if (in_U(a, t) && get_tally(a.blob, t) == BT_FREE) { slot_out = t; return step; }
    }
    return 0;
}
__global__ void build_repair_kernel(BuildArgs a) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    uint32_t nf = a.errors[0];
    if (nf > a.flagged_cap) nf = a.flagged_cap;
    for (uint32_t i = 1; i < nf; ++i) {   // slot order
        const uint64_t v = a.flagged[i];
        int j = (int)i - 1;
        while (j >= 0 && a.flagged[j] > v) { a.flagged[j + 1] = a.flagged[j]; --j; }
        a.flagged[j + 1] = v;
    }
    uint64_t done_from = 0, done_to = 0;
    bool have_done = false;
    for (uint32_t f = 0; f < nf; ++f) {
        const uint64_t s = a.flagged[f];
        if (have_done && done_from <= done_to && s >= done_from && s <= done_to) continue;   // inside a repaired region
        uint64_t end = segment_end(a, s);
        for (;;) {   // (re)play the region [s .. end]
            for (uint64_t t = s;; t = next_slot(a, t)) {   // reset to the state after the heads pass
                const uint32_t n = list_len(a, t);
                if (in_U(a, t)) put_rec(a.blob, t, BT_FREE, 0xFFFFFFFFu);
                else if (n > 0) {
                    put_rec(a.blob, t, (n == 1 && cnt_get(a.cntM, t) == 0) ? BT_BOTH1 : BT_PLUS1, a.pool[a.base[t]]);
                    set_left(a, t, n - 1);
                }
                if (t == end) break;
            }
            bool grow = false, give_up = false;
            for (;;) {
                uint64_t best = 0;
                uint32_t bestpos = 0xFFFFFFFFu;
                bool any = false;
                for (uint64_t t = s;; t = next_slot(a, t)) {
                    const uint32_t n = list_len(a, t);
                    if (n >= 2) {
                        const uint32_t left = (a.fill[t >> 2] >> ((uint32_t)(t & 3) * 8)) & 255u;
                        if (left) {
                            const uint32_t p = a.pool[(uint64_t)a.base[t] + (n - left)];
                            if (!any || p < bestpos) { any = true; best = t; bestpos = p; }
                        }
                    }
                    if (t == end) break;
                }
                if (!any) break;
                uint64_t eol = best;   // FindEndOfList, ufindex.cpp:945-985
                for (;;) {
                    const uint32_t T = get_tally(a.blob, eol);
                    if (T == BT_PLUS1 || T == BT_BOTH1 || T == BT_END) break;
                    if (T == 253 || T == BT_LONG) {
                        const uint32_t P = get_pos(a.blob, eol);
                        eol = (eol + (P & 0xffffu)) % a.slot_count;
                        eol = (eol + (P >> 16)) % a.slot_count;
                    } else
                        eol = (eol + (T & 127u)) % a.slot_count;
                }
                uint64_t fs = 0, fs2 = 0;
                const uint32_t step = repair_find_free(a, eol, end, fs, grow);
                if (grow) break;
                if (step == 0) { give_up = true; break; }
                if (step > BT_MAX_NEXT) {   // ufindex.cpp:256-300
                    const uint32_t step2 = repair_find_free(a, fs, end, fs2, grow);
                    if (grow) break;
                    if (step2 == 0) { give_up = true; break; }
                    const uint32_t eolpos = get_pos(a.blob, eol);
                    put_rec(a.blob, eol, (uint8_t)((get_tally(a.blob, eol) & BT_MY_BIT) | BT_LONG), step | (step2 << 16));
                    put_rec(a.blob, fs, BT_LONG, eolpos);
                    put_rec(a.blob, fs2, BT_END, bestpos);
                } else {   // ufindex.cpp:303-313
                    a.blob[5 * eol] = (uint8_t)((get_tally(a.blob, eol) & BT_MY_BIT) | step);
                    put_rec(a.blob, fs, BT_END, bestpos);
                }
                set_left(a, best, ((a.fill[best >> 2] >> ((uint32_t)(best & 3) * 8)) & 255u) - 1);
            }
            if (give_up) { atomicAdd(a.errors + 2, 1u); break; }   // TruncateSlot (ufindex.cpp:153-192) is not reproduced
            if (!grow) break;
            end = segment_end(a, next_slot(a, end));   // the region swallows the next segment and is replayed
        }
        done_from = s;
        done_to = end;
        have_done = true;
    }
}

static std::string g_build_err;

#define BCK(call)                                                                          \
    do {                                                                                   \
        cudaError_t e_ = (cudaError_t)(call);                                              \
        if (e_ != cudaSuccess) {                                                           \
            g_build_err = std::string(#call) + ": " + cudaGetErrorString(e_);              \
            goto fail;                                                                     \
        }                                                                                  \
    } while (0)

}  // namespace urmb

using namespace urmb;

#ifndef URMB_EMU
extern "C" const char *urmb_build_last_error() { return g_build_err.c_str(); }

// d_seq: seq_data_size bytes on the current device; d_blob: 5*slot_count+URMB_BLOB_PAD bytes (written).
// stats[0] = indexed positions, stats[1] = lists the reference would truncate (the blob is then NOT valid),
// stats[2] = microseconds.
extern "C" int urmb_build_index_device(const void *d_seq, uint64_t seq_data_size, uint64_t slot_count,
                                       uint32_t word_length, uint32_t max_ix, void *d_blob, uint64_t *stats) {
    // the slot counts saturate at 255 as the reference's (ufindex.cpp:338-408): lists of up to 254 positions are exact here
    if (!d_seq || !d_blob || slot_count < 2 || word_length < 8 || word_length > 32 || max_ix < 1) return URMB_E_ARG;
    if (max_ix > 254) { g_build_err = "-maxix above 254 (saturated slot counts)"; return URMB_E_UNSUPPORTED; }
    BuildArgs a{};
    a.seq = (const uint8_t *)d_seq;
    a.seq_size = seq_data_size;
    a.slot_count = slot_count;
    a.magic = barrett_magic(slot_count);
    a.shift_mask = (word_length >= 32) ? ~0ull : ((1ull << (2 * word_length)) - 1);
    a.word_len = word_length;
    a.max_ix = max_ix;
    a.blob = (uint8_t *)d_blob;
    const uint64_t cwords = (slot_count + 3) / 4 + 1;
    const uint64_t nblocks = (slot_count + kScanBlock - 1) / kScanBlock;
    uint64_t total = 0;
    uint32_t herr[4] = {0, 0, 0, 0};
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    float ms = 0;
    const int T = 256;
    const uint64_t gpos = (seq_data_size + T - 1) / T, gslot = (slot_count + T - 1) / T;
    BCK(cudaEventCreate(&e0));
    BCK(cudaEventCreate(&e1));
    BCK(cudaEventRecord(e0));
    BCK(cudaMalloc(&a.cntP, cwords * 4));
    BCK(cudaMalloc(&a.cntM, cwords * 4));
    BCK(cudaMalloc(&a.fill, cwords * 4));
    BCK(cudaMalloc(&a.base, slot_count * 4));
    BCK(cudaMalloc(&a.blocksum, (nblocks + 1) * 8));
    BCK(cudaMalloc(&a.qzero, slot_count / 8 + 16));
    BCK(cudaMalloc(&a.blockA, (nblocks + 1) * 8));
    BCK(cudaMalloc(&a.blockB, (nblocks + 1) * 8));
    BCK(cudaMalloc(&a.blockQ, (nblocks + 1) * 8));
    BCK(cudaMalloc(&a.errors, 16));
    a.flagged_cap = 1u << 18;   // appended in nearly increasing slot order, so the repair pass's insertion sort stays cheap
    BCK(cudaMalloc(&a.flagged, (size_t)a.flagged_cap * 8));
    BCK(cudaMemset(a.cntP, 0, cwords * 4));
    BCK(cudaMemset(a.cntM, 0, cwords * 4));
    BCK(cudaMemset(a.fill, 0, cwords * 4));
    BCK(cudaMemset(a.qzero, 0, slot_count / 8 + 16));
    BCK(cudaMemset(a.errors, 0, 16));
    BCK(cudaMemset(a.blocksum, 0, (nblocks + 1) * 8));
    BCK(cudaMemset((uint8_t *)d_blob + 5 * slot_count, 0, URMB_BLOB_PAD));
    build_init_kernel<<<(unsigned)(((slot_count + 3) / 4 + T - 1) / T), T>>>(a);
    build_count_kernel<<<(unsigned)gpos, T>>>(a);
    build_blocksum_kernel<<<(unsigned)nblocks, 256>>>(a);
    build_scan_blocksums_kernel<<<1, 1024>>>(a, nblocks + 1);   // entry [nblocks] (zero) becomes the grand total
    BCK(cudaGetLastError());
    BCK(cudaMemcpy(&total, a.blocksum + nblocks, 8, cudaMemcpyDeviceToHost));
    BCK(cudaMalloc(&a.pool, (total + 1) * 4));
    build_base_kernel<<<(unsigned)nblocks, 256>>>(a);
    build_scatter_kernel<<<(unsigned)gpos, T>>>(a);
    build_heads_kernel<<<(unsigned)gslot, T>>>(a);
    build_carry_block_kernel<<<(unsigned)nblocks, 256>>>(a);
    build_carry_top_kernel<<<1, 1024>>>(a, nblocks);
    build_carry_apply_kernel<<<(unsigned)nblocks, 256>>>(a);
    build_segment_kernel<<<(unsigned)gslot, T>>>(a);
    build_repair_kernel<<<1, 32>>>(a);
    BCK(cudaGetLastError());
    BCK(cudaMemcpy(herr, a.errors, 16, cudaMemcpyDeviceToHost));
    BCK(cudaEventRecord(e1));
    BCK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms, e0, e1);
    if (stats) {
        stats[0] = total;
        stats[1] = herr[2];
        stats[2] = (uint64_t)(ms * 1000.0f);
    }
    cudaFree(a.cntP); cudaFree(a.cntM); cudaFree(a.fill); cudaFree(a.base); cudaFree(a.blocksum);
    cudaFree(a.qzero); cudaFree(a.blockA); cudaFree(a.blockB); cudaFree(a.blockQ); cudaFree(a.errors); cudaFree(a.flagged); cudaFree(a.pool);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (herr[1]) { g_build_err = "pool overflow (internal error)"; return URMB_E_OVERFLOW; }
    if (herr[3]) {   // a very dense table (one segment in ten needs the sequential repair pass at load factor 0.95)
        g_build_err = std::to_string(a.flagged_cap + herr[3]) + " segments need the sequential repair pass (more than its list of " +
                      std::to_string(a.flagged_cap) + " holds: dense table)";
        return URMB_E_OVERFLOW;
    }
    return URMB_OK;
fail:
    cudaFree(a.cntP); cudaFree(a.cntM); cudaFree(a.fill); cudaFree(a.base); cudaFree(a.blocksum);
    cudaFree(a.qzero); cudaFree(a.blockA); cudaFree(a.blockB); cudaFree(a.blockQ); cudaFree(a.errors); cudaFree(a.flagged); cudaFree(a.pool);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    return URMB_E_CUDA;
}

// Host-buffer convenience used by `urmap_b200 -make_ufi ... -gpu_build`.
extern "C" int urmb_host_gpu_build(const uint8_t *seq, uint64_t n, uint64_t slots, uint32_t W, uint32_t maxix,
                                   uint8_t *blob) {
    void *d_seq = nullptr, *d_blob = nullptr;
    int rc = URMB_E_CUDA;
    uint64_t stats[3] = {0, 0, 0};
    if (cudaMalloc(&d_seq, n + 64) != cudaSuccess) { g_build_err = "cudaMalloc(seq) failed (no CUDA device?)"; return URMB_E_NODEVICE; }
    if (cudaMalloc(&d_blob, 5 * slots + URMB_BLOB_PAD) != cudaSuccess) { g_build_err = "cudaMalloc(blob) failed"; goto out; }
    if (cudaMemset((uint8_t *)d_seq + n, 0, 64) != cudaSuccess) goto out;
    if (cudaMemcpy(d_seq, seq, n, cudaMemcpyHostToDevice) != cudaSuccess) goto out;
    rc = urmb_build_index_device(d_seq, n, slots, W, maxix, d_blob, stats);
    if (rc == 0 && stats[1] != 0) {
        g_build_err = std::to_string(stats[1]) + " list(s) would have to be truncated";
        rc = URMB_E_OVERFLOW;
    }
    if (rc == 0 && cudaMemcpy(blob, d_blob, 5 * slots, cudaMemcpyDeviceToHost) != cudaSuccess) rc = URMB_E_CUDA;
out:
    cudaFree(d_seq);
    cudaFree(d_blob);
    return rc;
}
#endif
