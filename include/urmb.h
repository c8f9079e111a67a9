/* include/urmb.h -- C ABI of the B200-native URMAP mapping engine (liburmb.so).
 *
 * URMAP has no plugin / FFI interface of its own (SURVEY.md §8b); the in-process boundary a
 * drop-in replacement slots under is the one its worker threads use:
 *
 *     MapThread      /root/reference/src/map.cpp:11-25    State1::SetUFI, State1::Search, Output1
 *     UFIMapThread   /root/reference/src/map2.cpp:11-37   State2::SetUFI, State2::Search
 *     UFIndex::FromFile  /root/reference/src/ufindexio.cpp:60-115
 *
 * Each entry point below names the reference interface it replaces.  Plain pointers and
 * sizes only; no C++ or torch types.  All functions return 0 on success, a negative URMB_E_*
 * code on failure (never exit()); urmb_last_error() gives the message (the reference instead
 * terminates the process through Die(), myutils.cpp:915).
 *
 * Threading: one urmb_ctx per GPU; a ctx may be driven by one host thread at a time.  A ctx
 * owns URMB_SLOTS batch slots so that the H2D copy of batch k+1, the kernels of batch k and
 * the D2H copy of batch k-1 overlap on separate CUDA streams.
 */
#ifndef URMB_H
#define URMB_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define URMB_OK 0
#define URMB_E_ARG (-1)       /* bad argument */
#define URMB_E_IO (-2)        /* file error / bad UFI magic */
#define URMB_E_CUDA (-3)      /* CUDA runtime error */
#define URMB_E_NOMEM (-4)
#define URMB_E_OVERFLOW (-5)  /* the caller's runs buffer is too small (urmb_map_se / urmb_map_pe) */
#define URMB_E_UNSUPPORTED (-6) /* word length > 32, batch of more than 4 GB of bases, ... */
#define URMB_E_NODEVICE (-7)  /* no CUDA device: there is NO CPU fallback */

#define URMB_SLOTS 8
#define URMB_MAX_READ_LEN 256
#define URMB_MAX_IX 1024 /* largest MaxIx of an index (-maxix, ufindexio.cpp:135-136; the reference's default is 32) */

typedef struct urmb_index_host urmb_index_host; /* parsed UFI file in (pinned) host memory */
typedef struct urmb_ctx urmb_ctx;               /* per-GPU context */

/* Scoring "method" (State1::SetMethod, state1.cpp:147-183; map.cpp:34-37; map2.cpp:15-21,46-48). */
typedef struct urmb_params {
    int32_t method;      /* 6 = default, 7 = -map -veryfast */
    int32_t pe_method;   /* 4 = default -map2 (Search4), 5 = -map2 -veryfast (Search5) */
    int32_t band_radius; /* <0: method default (12 / 8; Search5 uses 4) */
    int32_t minq;        /* statistics only (map2.cpp:75) */
    int32_t want_second; /* != 0: paired-end searches also report State2's second pair (urmb_second_hits; -tabbedout) */
} urmb_params;

/* A batch of reads: concatenated ASCII bases + n+1 offsets (what FASTQSeqSource::GetNext,
 * fastqseqsource.cpp:9, hands to State1::Search one read at a time). Labels and qualities
 * stay on the host. */
typedef struct urmb_batch {
    uint32_t n;
    const uint8_t *seqs;
    const uint32_t *offs;
} urmb_batch;

/* Per-read result: exactly the fields State1::SetSAM / State2::SetSAM2 consume
 * (m_TopHit->{m_DBStartPos,m_Plus,m_Score,m_Path}, m_Mapq; setsam.cpp:75, output2.cpp:71). */
typedef struct urmb_result {
    uint32_t db_pos;    /* m_TopHit->m_DBStartPos, 0xFFFFFFFF when there is no top hit */
    uint32_t path_off;  /* first run of the path in the runs pool */
    uint16_t path_runs; /* 0 => empty path (gapless hit, CIGAR "<QL>M") */
    int16_t score;      /* m_TopHit->m_Score */
    int16_t best;       /* m_BestScore */
    int16_t second;     /* m_SecondBestScore */
    uint8_t mapq;       /* m_Mapq */
    uint8_t flags;      /* bit0 plus strand, bit1 has top hit, bit6 not searched (read or mate longer than
                           URMB_MAX_READ_LEN), bit7 capacity overflow */
    uint8_t hit_count;
    uint8_t hsp_count;
} urmb_result;
/* Second pair of a paired-end search: m_UD_Fwd/Rev.m_SecondHit as AdjustTopHitsAndMapqs leaves them (search2.cpp:49-56),
 * which is what State2::OutputTab2 prints (outputtab2.cpp:85-119).  flags bit1 clear = no second hit. */
typedef struct urmb_second {
    uint32_t db_pos; /* m_SecondHit->m_DBStartPos */
    int16_t score;   /* m_SecondHit->m_Score */
    uint8_t flags;   /* bit0 plus strand, bit1 has second hit */
    uint8_t pad;
} urmb_second;
/* path run: u16 = (len << 2) | op, op 0='M' 1='D' 2='I' in the reference's PATH alphabet
 * (D consumes the read, I consumes the genome; PathToCIGAR, cigar.cpp:22-25, swaps them). */

typedef struct urmb_contig {
    uint32_t length;
    uint32_t offset; /* into the concatenated sequence data */
    const char *label;
} urmb_contig;

/* Device-resident index description for urmb_index_attach (e.g. buffers that arrived by an
 * NCCL broadcast). d_blob must hold 5*slot_count+16 bytes, d_seq seq_data_size+URMB_SEQ_PAD
 * bytes with the padding zero-filled. */
#define URMB_SEQ_PAD 4096
#define URMB_BLOB_PAD 16
typedef struct urmb_index_desc {
    uint32_t word_length;
    uint32_t max_ix;
    uint32_t seq_data_size;
    uint32_t reserved;
    uint64_t slot_count;
    const void *d_blob;
    const void *d_seq;
} urmb_index_desc;

/* Kernel timings of the last launch on a slot (CUDA events on the launching streams). */
#define URMB_KCLASSES 12 /* 0 probe, 1 seed pairing (PE) / seeds (SE), 2 first HSP alignment, 3 rows (short rows), 4 final
                            HSP alignment, 5 pair finishing, 6 mate rescue: window scans continued from the saved pair states,
                            7 deferred long rows, 8 mate rescue: full-window DPs, 9 mate rescue: legacy kernel (pairs beyond
                            the rescue pool, searched again from scratch), 10 mate rescue: last round (stragglers finished in
                            place), 11 reserved */
typedef struct urmb_timing {
    float probe_ms;  /* slot-probe / gather kernel */
    float search_ms; /* all search kernels on the compute stream (seed pairing, alignment, rows, finishing) */
    float h2d_ms;
    float d2h_ms;
    float rescue_ms; /* mate-rescue kernel: runs on a side stream and overlaps the next batch */
    float kernel_ms[URMB_KCLASSES];      /* summed launch durations per kernel class */
    uint32_t kernel_launches[URMB_KCLASSES];
} urmb_timing;

/* ---- index: replaces UFIndex::FromFile (ufindexio.cpp:51,60-115) ---- */
int urmb_index_load_host(const char *ufi_path, urmb_index_host **out);
void urmb_index_free_host(urmb_index_host *h);
int urmb_index_info(const urmb_index_host *h, urmb_index_desc *desc /* d_* = host pointers */,
                    uint32_t *n_contigs);
int urmb_index_contig(const urmb_index_host *h, uint32_t i, urmb_contig *out);

/* ---- context: replaces the per-thread State1 / State2 objects (map.cpp:13, map2.cpp:14) ---- */
int urmb_ctx_create(int device, const urmb_params *p, urmb_ctx **out);
void urmb_ctx_destroy(urmb_ctx *c);
const char *urmb_last_error(const urmb_ctx *c); /* c may be NULL: last global error */

/* ---- State1::SetUFI / State2::SetUFI (state1.cpp:185, state2.cpp:14) ---- */
int urmb_index_upload(urmb_ctx *c, const urmb_index_host *h);   /* H2D copy, ctx owns the buffers */
int urmb_index_attach(urmb_ctx *c, const urmb_index_desc *d);   /* caller-owned device buffers */
int urmb_index_broadcast(urmb_ctx **ctxs, int n, const urmb_index_host *h); /* one process, n GPUs */
int urmb_index_device_desc(const urmb_ctx *c, urmb_index_desc *out);

/* ---- mapping: State1::Search (search1.cpp:7) / State2::Search (search2.cpp:59) ---- */
/* Synchronous convenience calls on slot 0: host buffers in, host buffers out. */
int urmb_map_se(urmb_ctx *c, const urmb_batch *in, urmb_result *out, uint16_t *runs, uint32_t runs_cap,
                uint32_t *runs_used);
int urmb_map_pe(urmb_ctx *c, const urmb_batch *r1, const urmb_batch *r2, urmb_result *out1,
                urmb_result *out2, uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used);

/* Pipelined calls: stage -> (upload, launch, download are enqueued on the slot's stream) -> wait.
 * r2 == NULL selects single-end.  After urmb_wait the results of the slot stay valid in pinned
 * host memory until the slot is staged again. */
int urmb_submit(urmb_ctx *c, int slot, const urmb_batch *r1, const urmb_batch *r2);
int urmb_wait(urmb_ctx *c, int slot, const urmb_result **res1, const urmb_result **res2,
              const uint16_t **runs, uint32_t *runs_used);
/* Reads whose search exceeded a per-read capacity of the kernels (256 hits, 256 HSPs, 64 path runs per alignment; the
 * reference grows these lists without bound, state1.cpp:190) are still reported, with bit 7 set in urmb_result.flags, and
 * counted here: *last = such reads in the batch urmb_wait last returned for this slot, *total = over all batches of the
 * context.  Their records may differ from the reference's; it is not an error of the batch. */
int urmb_overflow_count(urmb_ctx *c, int slot, uint32_t *last, uint64_t *total);
/* Reads longer than URMB_MAX_READ_LEN are not searched (the reference maps reads up to 4096 bases, xdpmem.h:6): they and
 * their mates are reported unmapped with bit 6 set in urmb_result.flags; every other read of the batch is mapped as usual.
 * Counts as for urmb_overflow_count. */
int urmb_unsupported_count(urmb_ctx *c, int slot, uint32_t *last, uint64_t *total);
/* Pairs that left State2::Search4/5 inside its seed loop (search2m4.cpp:79-142: MAPQ 40/40 exit) on the probe kernel's first
 * look at the first 8 steps of both seed iterators, and therefore skipped the complete probe and the search kernels
 * (statistics; counts as for urmb_overflow_count). */
int urmb_first_look_count(urmb_ctx *c, int slot, uint32_t *last, uint64_t *total);
/* After urmb_wait on a paired-end slot of a context created with want_second: the second hits of mate 1 / mate 2. */
int urmb_second_hits(urmb_ctx *c, int slot, const urmb_second **s1, const urmb_second **s2);
/* Finer-grained steps (bench.py uses them to time the kernels with inputs resident in HBM). */
int urmb_upload(urmb_ctx *c, int slot, const urmb_batch *r1, const urmb_batch *r2);
int urmb_launch(urmb_ctx *c, int slot);
int urmb_download(urmb_ctx *c, int slot);
int urmb_timing_last(urmb_ctx *c, int slot, urmb_timing *t);
/* Number of kernels launched by this ctx so far. */
uint64_t urmb_launch_count(const urmb_ctx *c);
/* Context-wide time marks for timing several launches issued back to back: a mark is a CUDA event recorded after all
 * work submitted so far on both the compute and the rescue stream.  urmb_mark_elapsed synchronises on mark 1 and
 * returns the device time between mark 0 and mark 1. */
int urmb_mark(urmb_ctx *c, int which /* 0 | 1 */);
int urmb_mark_elapsed(urmb_ctx *c, float *ms);

/* ---- index construction on the device (SURVEY.md §8f rank 2; replaces UFIndex::MakeIndex, ufindex.cpp:83-151).
 * The blob is BYTE-IDENTICAL to the reference's: the order-dependent placement of overflow list elements
 * (UpdateSlot / FindFreeSlot, ufindex.cpp:194-322, 987-1000) is reproduced by cutting the table into independent
 * segments with a max-plus carry scan and replaying the reference's insertions inside each segment in genome order;
 * segments in which an element needs a long link (probe distance > 124) are replayed once more, merged with the
 * segments they spill into (urmb_build.cu).  Only lists that the reference would TRUNCATE (no free slot within 65534)
 * are not reproduced: stats[1] counts them, the blob is then not valid and the caller must use the sequential builder
 * (`urmap_b200 -make_ufi -gpu_build` does that by itself).
 * d_seq: seq_data_size bytes of upper-case sequence data on the current device; d_blob: 5*slot_count+URMB_BLOB_PAD
 * bytes (written).  stats[0] = indexed positions, stats[1] = lists that would be truncated, stats[2] = microseconds. */
int urmb_build_index_device(const void *d_seq, uint64_t seq_data_size, uint64_t slot_count, uint32_t word_length,
                            uint32_t max_ix, void *d_blob, uint64_t *stats);
const char *urmb_build_last_error(void);

/* Index of a FASTA file built on the device(s) of n contexts: the table `-make_ufi` writes for the same word length,
 * max_ix and slot count, without a file.  fa: the raw (decompressed) FASTA bytes on the host.  *header receives the
 * contig table (labels, lengths, offsets); its blob / seq pointers are NULL.  The contexts own the device buffers.
 * The bytes are parsed on every device (urmb_fasta.cu) into exactly the SeqData of UfiBuilder::ReadFasta (urmb_host.cpp,
 * fastaseqsource.cpp:26-112).  Errors: URMB_E_IO for a bad FASTA ("expected '>' in line N", as -make_ufi) or one without
 * sequence; URMB_E_UNSUPPORTED for a genome larger than SeqData can address; the builder's own code and message when it
 * refuses the table (URMB_E_OVERFLOW: a list the reference would truncate, a full repair list; URMB_E_UNSUPPORTED: max_ix
 * above 254) -- `-make_ufi` builds those tables on the host. */
int urmb_index_from_fasta(urmb_ctx **ctxs, int n, const uint8_t *fa, uint64_t fa_len, uint32_t word_length,
                          uint32_t max_ix, uint64_t slot_count, urmb_index_host **header);
/* Labels of the FASTA records that had no sequence and were dropped (for the warnings -make_ufi prints); URMB_E_ARG past the
 * last one. */
int urmb_index_dropped(const urmb_index_host *h, uint32_t i, const char **label);
/* Seconds spent by urmb_index_from_fasta (host clock around device work that ends in a synchronise; the slowest GPU):
 * t[0] upload of the raw bytes, t[1] parse, t[2] table build, t[3] packed genome, t[4] device time of the parse kernels. */
int urmb_index_fasta_times(const urmb_index_host *h, double t[5]);

/* Optional: size all slots for batches of n_units reads (pairs when paired != 0) of up to max_read_len bases ahead of
 * the first urmb_submit.  It touches the slots only and may run on another thread while urmb_index_upload /
 * urmb_index_broadcast of the same context is still copying; word_length is the index's (UFI header). */
int urmb_reserve(urmb_ctx *c, uint32_t n_units, uint32_t max_read_len, int paired, uint32_t word_length);

/* ---- page-locked host memory for read batches.  When the `seqs` pointers of a batch handed to urmb_submit / urmb_upload
 * lie in page-locked memory (from urmb_host_alloc, cudaHostAlloc / cudaHostRegister, a pinned torch tensor ...) the bases
 * are copied to the device straight from there, without the staging copy; such a batch must then stay unchanged until
 * urmb_wait has returned for that slot.  Pageable batches are staged as before and may be reused right after the call. */
int urmb_host_alloc(size_t bytes, void **out);
void urmb_host_free(void *p);

/* ---- measured roofline denominators (SURVEY.md §8d: "a 32-byte random-gather micro-benchmark on the 27 GB blob" and
 * "measured int32 ALU op/s from a micro-benchmark on the same box").  No reference counterpart; bench.py calls them.
 * urmb_peak_gather: n_access random reads of access_bytes (4 | 8 | 16) at 32-byte-aligned addresses uniform over
 * d_buf[0, n_bytes) (32-byte aligned device pointer, current device); *ms = device time of the best of two timed passes.
 * urmb_peak_alu: independent LOP3/IADD3/SHF chains, ops_per_thread per thread on SMs x 8 blocks x 256 threads;
 * *total_ops = 32-bit integer operations executed in *ms. */
int urmb_peak_gather(const void *d_buf, uint64_t n_bytes, uint32_t access_bytes, uint64_t n_access, float *ms);
int urmb_peak_alu(uint64_t ops_per_thread, float *ms, double *total_ops);

#ifdef __cplusplus
}
#endif
#endif /* URMB_H */
