/* oracle/urmap_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * C entry points of the CPU restatement of URMAP's mapping hot path (SURVEY.md §8a).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library; the product (urmap_b200/) never links or calls it.
 *
 * Parity status: PINNED -- tests/test_oracle_vs_reference.py checks the SAM text this
 * restatement produces against the SAM of the unmodified reference binary
 * (oracle/_ref/urmap, compiled from /root/reference/src by oracle/Makefile) and against
 * the committed golden SAM fixtures in tests/golden/ made by the same binary.
 */
#ifndef URMAP_ORACLE_H
#define URMAP_ORACLE_H
#include <stdint.h>
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct uo_index uo_index;

typedef struct uo_params {
    int32_t method;      /* State1::SetMethod: 6 (default) or 7 (-map -veryfast)  state1.cpp:147 */
    int32_t pe_method;   /* State2::m_Method: 4 (default) or 5 (-map2 -veryfast)   map2.cpp:46   */
    int32_t band_radius; /* <0: method default (12 / 8); map2 -veryfast forces 4   map2.cpp:17   */
    int32_t minq;        /* only used by the hit statistics                         map2.cpp:75   */
} uo_params;

/* Same layout as urmb_result (include/urmb.h). */
typedef struct uo_result {
    uint32_t db_pos;     /* m_TopHit->m_DBStartPos, 0xFFFFFFFF when m_TopHit == 0 */
    uint32_t path_off;   /* first run of the top hit's path in the runs pool */
    uint16_t path_runs;  /* 0 => empty path (gapless, CIGAR <QL>M) */
    int16_t  score;      /* m_TopHit->m_Score (0 if none) */
    int16_t  best;       /* m_BestScore */
    int16_t  second;     /* m_SecondBestScore */
    uint8_t  mapq;       /* m_Mapq */
    uint8_t  flags;      /* bit0: plus strand; bit1: has top hit */
    uint8_t  hit_count;  /* min(m_HitCount,255) */
    uint8_t  hsp_count;  /* min(m_HSPCount,255) */
} uo_result;

/* Work counters that define the algorithmic bytes / cells of SURVEY.md §8d. */
typedef struct uo_stats {
    uint64_t reads;
    uint64_t probes;        /* P: GetBlob calls                          */
    uint64_t row_calls;     /* GetRow_Blob calls                          */
    uint64_t row_hops;      /* H: list elements fetched beyond the head   */
    uint64_t extend_calls;  /* ExtendPen + ExtendScan calls               */
    uint64_t compare_bytes; /* C: genome bytes compared / scanned         */
    uint64_t slot_hashes;   /* S                                          */
    uint64_t dp_calls;
    uint64_t dp_cells;      /* inner-loop trip count of viterbi.cpp:122   */
    uint64_t scan_calls;
    uint64_t tb_poison_reads; /* traceback reads of cells the current call never wrote */
    uint64_t compare_bytes_rows; /* part of C spent on positions that came out of GetRow_Blob */
    uint64_t row_hops_long;      /* part of H spent on the second visit of rows longer than 2 (phase 5 / pending round 2) */
    uint64_t compare_bytes_rows_long; /* part of compare_bytes_rows spent there */
    uint64_t dp_cells_scan;      /* part of dp_cells spent in State1::Scan's full-window Viterbi (mate rescue) */
} uo_stats;

uo_index *uo_index_open(const char *ufi_path);   /* mmap, ufindexio.cpp:60-115 */
void uo_index_close(uo_index *ix);
uint64_t uo_index_slot_count(const uo_index *ix);
uint32_t uo_index_seq_size(const uo_index *ix);
uint32_t uo_index_word_length(const uo_index *ix);
uint32_t uo_index_max_ix(const uo_index *ix);
uint32_t uo_index_contig_count(const uo_index *ix);
const uint8_t *uo_index_blob(const uo_index *ix);
const uint8_t *uo_index_seq(const uo_index *ix);

/* runs: u16 = (len << 2) | op, op 0='M' 1='D' 2='I' in the reference's PATH alphabet
 * (D consumes the read only, I consumes the genome only; PathToCIGAR swaps them). */
int uo_map_se(const uo_index *ix, const uo_params *p, const uint8_t *seqs, const uint32_t *offs,
              uint32_t n, uo_result *res, uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used,
              uo_stats *stats, int threads);
int uo_map_pe(const uo_index *ix, const uo_params *p, const uint8_t *seqs1, const uint32_t *offs1,
              const uint8_t *seqs2, const uint32_t *offs2, uint32_t n, uo_result *res1,
              uo_result *res2, uint16_t *runs, uint32_t runs_cap, uint32_t *runs_used,
              uo_stats *stats, int threads);

/* SAM text (setsam.cpp, output1.cpp, output2.cpp, state1.cpp:736). Returned buffers are
 * malloc'd; release with uo_free.  labels/quals are concatenated with the given offsets;
 * quals may be NULL. */
char *uo_sam_header(const uo_index *ix, const char *version, const char *cmdline, size_t *len);
char *uo_sam_se(const uo_index *ix, uint32_t n, const uint8_t *seqs, const uint32_t *offs,
                const uint8_t *quals, const uint8_t *labels, const uint32_t *label_offs,
                const uo_result *res, const uint16_t *runs, size_t *len);
char *uo_sam_pe(const uo_index *ix, uint32_t n, const uint8_t *seqs1, const uint32_t *offs1,
                const uint8_t *quals1, const uint8_t *labels1, const uint32_t *label_offs1,
                const uint8_t *seqs2, const uint32_t *offs2, const uint8_t *quals2,
                const uint8_t *labels2, const uint32_t *label_offs2, const uo_result *res1,
                const uo_result *res2, const uint16_t *runs, size_t *len);
void uo_free(void *p);

/* Unit-level entry points for kernel parity tests. */
void uo_slots(const uo_index *ix, const uint8_t *seq, uint32_t L, uint64_t *plus, uint64_t *minus);
void uo_revcomp(const uint8_t *seq, uint32_t L, uint8_t *out);
/* returns score; path (NUL-terminated, reference path alphabet) must hold LA+LB+2 bytes */
float uo_viterbi(const uo_params *p, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB,
                 int left, int right, char *path);
/* uo_viterbi plus the number of traceback reads of cells the call never wrote (uo_stats::tb_poison_reads): where it
 * is not zero the reference reads stale bytes there and its result is undefined */
float uo_viterbi_ex(const uo_params *p, const uint8_t *A, uint32_t LA, const uint8_t *B, uint32_t LB,
                    int left, int right, char *path, uint64_t *tb_poison_reads);
/* path -> CIGAR incl. the dangling-M polish (cigar.cpp:4,141); out must hold 12*strlen(path)+16 */
void uo_path_to_cigar(const char *path, uint32_t QL, char *out);
uint64_t uo_get_prime(uint64_t n);
/* number of slots whose observable content (head class + GetRow_Blob list) differs; ~0 if incomparable */
uint64_t uo_index_functional_diff(const uo_index *a, const uo_index *b, uint64_t *first_bad);               /* prime.cpp:11 + primes.h */

#ifdef __cplusplus
}
#endif
#endif
