/*
 * psa.h -- C-ABI of the B200-native pairwise-alignment hot path (libpsa.so).
 *
 * This is the drop-in boundary for the reference's DP fill + traceback.  The reference has no
 * FFI layer; its seam is the free function
 *     int main_alignment_function(char* A, char* B, size_t m, size_t n, size_t p, double g, double h)
 *         (/root/reference/alignment_algorithm/main_alignment.h:38, body main_alignment.cpp:353-410)
 * and, one level down, class Subproblem (alignment_algorithm/subproblem_alignment.h:16-97).
 * Each entry point below names the reference interface it replaces.  All pointers are plain host
 * pointers unless the name says _device; no C++/torch types cross this boundary; every function
 * returns 0 on success or a negative psa_status.  There is NO CPU fallback: without a usable
 * CUDA device every compute call fails with PSA_ERR_CUDA.
 *
 * Conventions
 *   - sequences are passed as pointers to base 1 (a[0] is the reference's A[1]) plus lengths;
 *     raw bytes, any alphabet, compared with == (subproblem_alignment.h:83-88)
 *   - scoring: match +1, mismatch 0, a gap of length k costs h + g*k; g,h integers >= 0
 *   - table values are int32; PSA_NEG_INF stands for the reference's -infinity
 *   - states: 1 = diagonal (A[i] over B[j]), 2 = gap in A (consumes B[j]), 3 = gap in B
 *     (consumes A[i])  -- struct alignment_point.t, subproblem_alignment.h:8-13
 */
#ifndef PSA_H
#define PSA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSA_NEG_INF (INT32_MIN / 2)

typedef enum {
    PSA_OK = 0,
    PSA_ERR_ARG = -1,          /* null pointer, negative size, non-integral/negative g or h        */
    PSA_ERR_RANGE = -2,        /* score range does not fit the kernel's lanes / a size limit        */
    PSA_ERR_CUDA = -3,         /* any CUDA failure, including "no device" (never falls back to CPU)  */
    PSA_ERR_NOMEM = -4,
    PSA_ERR_CAPACITY = -5      /* caller-provided output buffer too small                            */
} psa_status;

typedef enum { PSA_GLOBAL = 0, PSA_LOCAL = 1 } psa_mode;

/* what to compute */
#define PSA_WANT_SCORE     1u  /* corner values (global) / best score + end cell (local)            */
#define PSA_WANT_TRACEBACK 2u  /* + alignment path                                                   */
#define PSA_OPS_COMPACT    4u  /* psa_align_batch_packed: op words back to back instead of fixed stride */

typedef struct psa_ctx psa_ctx;

/* One context per (host thread, device).  Owns a stream and reusable device/pinned scratch.
 * Replaces: nothing in the reference (it keeps no state); plays the role of the per-call
 * Subproblem tables (subproblem_alignment.h:66-73) but never holds an O(mn) table. */
int psa_ctx_create(int device, psa_ctx** out);
void psa_ctx_destroy(psa_ctx* ctx);
/* Last error text of this context (never NULL). psa_ctx_create failures: pass NULL. */
const char* psa_last_error(const psa_ctx* ctx);
/* Number of kernel launches issued through this context so far (bench.py's gpu_launches). */
int64_t psa_launch_count(const psa_ctx* ctx);

/* ---- single pair ------------------------------------------------------------------------
 * Replaces Subproblem::compute_tables() + Subproblem::find_alignment()
 * (subproblem_alignment.cpp:329-355, :105-172) for start_type = end_type = -1, the only live
 * case (main_alignment.cpp:396-407), and print_seq's rows (main_alignment.cpp:32-55). */
typedef struct {
    int32_t t1, t2, t3;        /* global: T1/T2/T3[m][n]; local: t1 = score, t2 = t3 = PSA_NEG_INF  */
    int32_t score;             /* global: max(t1,t2,t3); local: best T1                              */
    int32_t end_state;         /* state the traceback starts in                                      */
    int64_t end_i, end_j;      /* global: m, n; local: end cell (1-based; 0,0 when score == 0)      */
    int64_t start_i, start_j;  /* first emitted cell (1-based; 0,0 when nothing is emitted)         */
    int64_t aln_len;           /* emitted columns; 0 without PSA_WANT_TRACEBACK                      */
    uint8_t* ops;              /* aln_len states (1/2/3) in forward order; library-owned             */
    char* row_a;               /* aln_len chars + NUL: A[i] or '-' (print_seq line 1)                */
    char* row_b;               /* aln_len chars + NUL: B[j] or '-' (print_seq line 2)                */
} psa_result;

int psa_align_pair(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int mode, int g, int h,
                   unsigned flags, psa_result* out);
void psa_result_free(psa_result* r);

/* sequence_similarity (test_functions/pull_data.cpp:97-127) for a batch of pairs in the psa_align_batch
 * layout: out[k] = #{ i < min(len_a,len_b) : a[i] == b[i] } / max(len_a,len_b)  (0 for an empty pair).
 * The host form copies in and out and returns when the results are in `out`; the device form is
 * asynchronous on the given stream (max_len = upper bound of every length, picks the launch shape). */
int psa_similarity_batch(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                         const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                         size_t bytes_a, size_t bytes_b, double* out);
int psa_similarity_batch_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                int max_len, double* d_out, void* cuda_stream);

/* The other border variants of the reference's Subproblem (start_type / end_type in
 * {-1,-2,-3,1,2,3}: subproblem_alignment.cpp:212-227 and :259-292 for the borders, :112-146 for
 * the forced / credited end state) -- what optimal_alignment (main_alignment.cpp:250-251) would
 * pass for the pieces of a partitioned alignment.  Global mode.  Pieces with n <= 256 take the short-pair
 * kernel, larger ones the long-pair kernels (checkpointed traceback, lengths < 2^21 - 1). */
int psa_align_pair_typed(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int start_type, int end_type,
                         int g, int h, unsigned flags, psa_result* out);

/* optimal_alignment over a partition (main_alignment.cpp:202-350): bp[0..n_bp) are the partition
 * points (i, j, t) -- the `align` nodes of subproblem_alignment.h:8-13 -- in non-decreasing order;
 * piece k spans A(bp[k].i, bp[k+1].i] x B(bp[k].j, bp[k+1].j] with start type bp[k].t and end type
 * -bp[k+1].t (:248-251).  All pieces are solved by ONE batched launch and their alignments linked in
 * order.  The reference solves them in three thread waves and links all but the last piece
 * (:343, `i < num_subproblems-1`); here every piece is linked.  The live configuration is the
 * two-point partition {(0,0,-1), (m,n,1)} (:392-398), for which this equals psa_align_pair.
 * out: ops/rows/aln_len of the linked alignment, start cell of its first column, t1..t3/end_state
 * of the last piece, score = score of the linked alignment as printed.  If every piece is at most 256
 * columns wide they all run in one launch; otherwise a handful of pieces run one after the other, each on
 * the whole GPU, and more of them run as one batch of long pairs (one warp per piece, as psa_align_batch). */
typedef struct psa_bp {
    int64_t i, j;
    int32_t t;
    int32_t reserved;
} psa_bp;
int psa_align_partition(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, const psa_bp* bp, size_t n_bp,
                        int g, int h, psa_result* out);

/* Partition finder + stitched alignment (SURVEY 8 f-3): what sequence_alignment/partial.cpp:81-163 (best crossing
 * cell per special row from a forward and a reverse table, combine rule :101-108) and optimal_alignment
 * (main_alignment.cpp:202-351) were meant to do together.  A forward and a reverse score-only sweep on the GPU
 * keep H and T3 on every 128th row (O((m/128) n) memory instead of six O(mn) int tables); the best crossing of up
 * to pieces-1 evenly spread special rows is max_j max(Hf+Hr, T3f+T3r+h), smallest j first; the pieces between the
 * crossings are solved as independent typed subproblems (a crossing inside a vertical gap ends the piece above in
 * T3 and lets the piece below continue the gap) and stitched.  The stitched alignment is COMPLETE -- it includes
 * the border gap run find_alignment drops (subproblem_alignment.cpp:170) -- and is verified to re-score to the
 * optimum before it is returned (if tied co-optimal paths make two crossings incompatible the call falls back to
 * fewer pieces).  out: ops / rows / aln_len of the whole alignment, score = max(T1,T2,T3)[m][n];
 * bp_out (optional, capacity bp_cap): the crossings used, (i, j, t) with t = 1 node / 3 inside a vertical gap.
 * Global mode, start / end type -1; lengths < 2^21 - 1. */
int psa_align_long_partitioned(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int g, int h, int pieces,
                               psa_result* out, psa_bp* bp_out, size_t bp_cap, size_t* n_bp);

/* ---- batches of independent pairs -------------------------------------------------------
 * Replaces the harness' pair-parallel callers: hardware_concurrency() host threads each calling
 * main_alignment_function on its own pairs (test_functions/testing.cpp:145-152, :269-276,
 * :352-358).  Sequences are stored back to back in one byte array per side; pair k uses
 * bases_a[off_a[k] .. off_a[k]+len_a[k]) and likewise for b. */
typedef struct {
    int32_t t1, t2, t3;        /* as psa_result                                                      */
    int32_t score;
    int32_t end_state;
    int32_t end_i, end_j;
    int32_t start_i, start_j;
    int32_t aln_len;
} psa_batch_item;              /* 40 bytes */

/* ops, if requested, are 2-bit codes (1/2/3; 0 = unused), 16 per uint32 starting at bit 0, in
 * TRACEBACK order (first code = the end cell), ops_stride_words words per pair; the caller must
 * give ops_stride_words >= ceil((max m + max n) / 16), for short and long pairs alike.  Words past
 * ceil(aln_len / 16) of a pair are not written.  psa_ops_unpack turns one pair's words into
 * forward-order bytes.
 * Long pairs (wider than 256 columns) with PSA_WANT_TRACEBACK: a few pairs run one after the other, each
 * over the whole GPU (psa_align_long_device); larger batches run one warp per pair -- a fill that keeps
 * tile-boundary checkpoints, then a walk that recomputes only the tiles the path crosses -- in chunks
 * sized by the device memory free at call time.  Lengths < 2^21 - 1. */
int psa_align_batch(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                    const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                    size_t bytes_a, size_t bytes_b, int mode, int g, int h, unsigned flags,
                    psa_batch_item* items, uint32_t* ops, size_t ops_stride_words);

/* Same computation with every buffer already resident in device memory (the caller's
 * allocations, e.g. torch tensors) on the given cudaStream_t (NULL = the context's stream);
 * asynchronous: the caller synchronises.  max_len_a/max_len_b bound the lengths in the batch.
 * Long pairs accept PSA_WANT_TRACEBACK: always the one-warp-per-pair batch path (checkpointed fill +
 * batched walk), planned from n_pairs, max_len_a and max_len_b alone, so nothing is read back and the
 * call stays asynchronous; results are identical to psa_align_pair on each pair. */
int psa_align_batch_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                           const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b,
                           size_t n_pairs, int max_len_a, int max_len_b, int mode, int g, int h, unsigned flags,
                           psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream);

/* ---- banded batches ------------------------------------------------------------------------
 * psa_align_batch / psa_align_batch_device restricted to a diagonal band of half-width `band` >= 0: for a pair of
 * lengths m, n >= 1, cell (i, j) exists iff |j - floor(i*n/m)| <= band (the band around the line from (0,0) to (m,n));
 * every other cell is -infinity.  Inside the band the recurrence, borders, scoring, end cell, tie rules and traceback
 * order are psa_align_batch's, in both modes (a local alignment may start at any cell of the band).  Cell (m, n) is
 * always in the band; if the band admits no complete global path the record reports PSA_NEG_INF corners and score,
 * end state 1, aln_len 0, and no op words are written.  Members with m = 0 or n = 0 get psa_align_batch's record.
 * With band >= max(m, n) every cell is in the band and the results equal psa_align_batch's exactly.
 * For similar sequences (reads against their source window, overlaps, polishing) the fill and the traceback
 * checkpoints shrink from m*n to about m*(2*band + 1) cells.  Same buffer layouts, op-word format and capacity rule as
 * psa_align_batch; flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only (anything else: PSA_ERR_ARG); lengths < 2^21 - 1.
 * Score range: a band can force a gap opening on every row, so a global call with band < max(M, N) and M, N >= 1
 * (M, N = the largest lengths of the call) needs g(M+N+2) + h(min(M, N) + 3) + M + N < 2^28, else PSA_ERR_RANGE
 * ("banded score range exceeds int32 lanes").  Local calls and bands >= max(M, N) keep psa_align_batch's
 * g(M+N+2) + 2h + M + N < 2^28.  At g = 0 a 1 Mbp x 1 Mbp global pair admits h <= 266.
 * Every pair runs on the banded long-pair kernels, one warp per pair: short pairs are correct but gain nothing from
 * the band over psa_align_batch.  The device form is asynchronous on cuda_stream (NULL = the context's stream) and
 * plans its work from n_pairs, max_len_a, max_len_b and band alone. */
int psa_align_batch_banded(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                           const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                           size_t bytes_a, size_t bytes_b, int mode, int g, int h, int band, unsigned flags,
                           psa_batch_item* items, uint32_t* ops, size_t ops_stride_words);
int psa_align_batch_banded_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                  const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                  int max_len_a, int max_len_b, int mode, int g, int h, int band, unsigned flags,
                                  psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream);

/* ---- fixed-stride batches of 2-bit packed DNA reads ----------------------------------------
 * The short-read shape of config 2 as a production caller would hold it: every pair is len_a x len_b
 * (len_a <= 512, len_b <= 256), both sides packed 16 bases per 32-bit word (base r of a sequence in
 * bits 2*(r%16) of its word r/16; A=0 C=1 T=2 G=3 = (ascii >> 1) & 3), each sequence starting on a word
 * boundary: pair k's A is a2[k*ceil(len_a/16) ...].  No offset or length arrays, a quarter of the bytes
 * over PCIe, 16-byte result records; only plain upper-case ACGT can be represented -- anything else takes
 * psa_align_batch (raw bytes, any alphabet).  Same kernels, same results as psa_align_batch on the
 * unpacked reads.  Replaces the same callers (testing.cpp:120-152 builds one char buffer per read).
 * With PSA_OPS_COMPACT the op words come back to back in pair order: pair k's ceil(aln_len/16) words start at the
 * running sum of the earlier pairs' word counts (`ops` must still hold n_pairs * ops_stride_words words, the worst
 * case).  The words are packed on the GPU -- written straight into `ops` as whole 128-byte lines when `ops` is
 * page-locked, copied out once at the end otherwise -- so only words that carry ops cross PCIe: a 150 bp read
 * pair uses 6 - 11 of its 20-word stride. */
typedef struct {
    int32_t score;             /* local: best T1; global: max(T1,T2,T3)[m][n]                          */
    uint16_t end_i, end_j;     /* as psa_batch_item                                                    */
    uint16_t start_i, start_j;
    uint16_t aln_len;
    uint16_t end_state;
} psa_packed_item;             /* 16 bytes */

/* Host helper: packs n bytes of upper-case ACGT into ceil(n/16) words; returns the number of bytes that are
 * NOT one of A, C, G, T (0 = the sequence is representable; such bytes are packed as their (c>>1)&3). */
size_t psa_pack_bases(const uint8_t* bases, size_t n, uint32_t* packed);

/* Batch form for fixed-length reads held as ASCII (what pull_data.cpp:18-95 leaves in memory, testing.cpp:120-128
 * copies per pair): read k = bases[k*src_stride .. k*src_stride + len) -> packed[k*ceil(len/16) ...], i.e. exactly the
 * a2 / b2 layout of psa_align_batch_packed.  8 bases per 64-bit operation, n_threads host threads (0 = all hardware
 * threads).  Returns the total number of bytes that are not A, C, G or T (as psa_pack_bases does per sequence). */
size_t psa_pack_reads(const uint8_t* bases, size_t n_reads, size_t len, size_t src_stride, uint32_t* packed, int n_threads);

int psa_align_batch_packed(psa_ctx* ctx, const uint32_t* a2, const uint32_t* b2, size_t n_pairs, int len_a, int len_b,
                           int mode, int g, int h, unsigned flags, psa_packed_item* items, uint32_t* ops,
                           size_t ops_stride_words);

/* One long pair, sequences resident in device memory (configs 3 and 4): intra-pair wavefront
 * over all SMs; with PSA_WANT_TRACEBACK the fill keeps tile-boundary checkpoints and the path is
 * recovered by per-tile recompute -- never an O(mn) table.  Replaces compute_tables() +
 * find_alignment() for pairs the reference cannot even allocate (24 B/cell,
 * subproblem_alignment.h:66-73).  Asynchronous on cuda_stream; lengths < 2^21 - 1. */
int psa_align_long_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int mode, int g,
                          int h, unsigned flags, psa_batch_item* d_item, uint32_t* d_ops, size_t ops_words,
                          void* cuda_stream);

/* ---- one banded pair over the whole GPU ------------------------------------------------------
 * One pair inside the diagonal band of psa_align_batch_banded (|j - floor(i*n/m)| <= band), computed by every SM: the
 * row blocks of the banded tile kernels run as a wavefront over all resident warps (progress counters per strip), and
 * the traceback walk is fed by a parallel recompute of the band tiles it can still reach.  Results are a one-pair
 * psa_align_batch_banded's, byte for byte: the same record and op words, the same no-path record in global mode
 * (PSA_NEG_INF corners, end state 1, aln_len 0, no op words written), and with band >= max(m, n) those of
 * psa_align_pair / psa_align_long_device.  flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only; band < 0 or any other
 * flag is PSA_ERR_ARG; lengths >= 2^21 - 1 are PSA_ERR_RANGE, and so are (g, h) outside psa_align_batch_banded's score
 * range rule (global with band < max(m, n): g(m+n+2) + h(min(m, n) + 3) + m + n < 2^28).  With traceback the fill keeps tile checkpoints of at most
 * 3 KiB x min(NB*S, (n + 2*bw*NB)/256 + 2*NB) bytes (NB = ceil(m/128), S = ceil(n/256), bw = min(band, m + n)) plus a
 * code buffer of at most 256 MiB; if they exceed half of the free device memory the call fails with PSA_ERR_NOMEM.
 *
 * psa_align_pair_banded: host strings; fills *out as psa_align_pair does (m = 0 or n = 0: psa_align_pair's record).
 * psa_align_long_banded_device: sequences in device memory, m, n >= 1, psa_align_long_device's null / capacity rules
 * (ops_words >= ceil((m+n)/16) with traceback).  Asynchronous on cuda_stream (NULL = the context's stream); the plan
 * is a function of (m, n, band, mode, flags) alone, nothing is read back, and the call issues
 *     score only:  2 kernel launches (fill, record)
 *     traceback:   2 + 2 * ceil(NB / rpw) launches (tile offsets, fill, then a recompute and a walk per window), with
 *                  rpw = min(NB, max(1, floor(2^28 / (tpr * 16384)))),
 *                  tpr = min(S, floor((2*bw + floor(128*n/m) + 2) / 256) + 2). */
int psa_align_pair_banded(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int mode, int g, int h,
                          int band, unsigned flags, psa_result* out);
int psa_align_long_banded_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int mode,
                                 int g, int h, int band, unsigned flags, psa_batch_item* d_item, uint32_t* d_ops,
                                 size_t ops_words, void* cuda_stream);

/* ---- banded alignment along an anchor chain -------------------------------------------------------
 * The band of psa_align_batch_banded / psa_align_pair_banded, centred on a caller-supplied chain of anchors instead of
 * the straight line from (0,0) to (m,n): what a mapper knows after seeding and chaining.  An anchor (i, j) is the
 * boundary point after A[1..i] and B[1..j], the coordinates of the DP cells: a seed match of length L at 0-based
 * positions x in A and y in B gives the anchors (x, y) and (x+L, y+L).
 * For a pair with m, n >= 1 and anchors P_1 .. P_K the guide is the polyline P_0 = (0,0), P_1, ..., P_K, P_{K+1} = (m,n).
 *   valid chain:  0 <= i_k <= m and 0 <= j_k <= n, both coordinates non-decreasing along the chain (equal points,
 *                 horizontal runs (equal i) and vertical runs (equal j) are allowed)
 *   guide columns of row i, [cmin(i), cmax(i)]: if chain points lie on row i, the j of the first and the j of the last
 *                 of them; otherwise i lies strictly inside one segment P_k -> P_{k+1} (i_k < i < i_{k+1}) and
 *                 cmin(i) = cmax(i) = j_k + floor((i - i_k)(j_{k+1} - j_k) / (i_{k+1} - i_k))
 *   band:         lo(i) = max(0, cmin(i) - band), hi(i) = min(n, cmax(i) + band); cell (i, j) exists iff lo(i) <= j <= hi(i)
 * Everything else is psa_align_batch_banded's: out-of-band cells, borders (row 0's gap border up to hi(0), column 0's
 * where lo(i) = 0), both modes, tie rules, traceback order, op words, the no-path record (PSA_NEG_INF corners and score,
 * end state 1, aln_len 0, no op words) and, for m = 0 or n = 0, psa_align_batch's record.  An empty chain (K = 0) is
 * the diagonal band: results byte-identical to psa_align_batch_banded / psa_align_pair_banded.  A horizontal run widens
 * its row to cover the jump, so an insertion of any size is representable at any band; with band >= max(m, n) every
 * cell exists and the results equal psa_align_batch's whatever the chain.  Flags, band >= 0, lengths < 2^21 - 1, buffer
 * layouts, the capacity rule and the score-range rule (global with band < max(M, N): g(M+N+2) + h(min(M, N) + 3) + M + N
 * < 2^28) are psa_align_batch_banded's.  Checkpoint memory keeps that entry's bound for every valid chain.
 *
 * psa_align_batch_guided: host buffers; pair k uses anchors[off_anc[k] .. off_anc[k] + n_anc[k]).  Every chain is
 *   checked on the host (n_anc[k] >= 0, off_anc[k] >= 0, off_anc[k] + n_anc[k] <= total_anc, a valid chain for the
 *   pair's lengths, m = 0 or n = 0 included); a failure is PSA_ERR_ARG naming the pair and the anchor.
 * psa_align_batch_guided_device: every array in device memory (d_anchors, d_off_anc and d_n_anc non-null), asynchronous
 *   on cuda_stream, planned from n_pairs, max_len_a, max_len_b and band alone.  It cannot return a chain error: a pair
 *   whose chain is invalid gets the REJECTED record -- t1 = t2 = t3 = score = PSA_NEG_INF, end_state 0 (which no other
 *   record has), end / start cells 0, aln_len 0, no op words written -- and reads or writes nothing of the other pairs.
 * psa_align_pair_guided: host strings, fills *out as psa_align_pair_banded does, on the same whole-GPU kernels; the
 *   chain is checked on the host (PSA_ERR_ARG naming the anchor; anchors may be NULL when n_anchors = 0) and plans the
 *   call exactly.  The call issues
 *     score only:  2 kernel launches (fill, record)
 *     traceback:   2 + 2 * ceil(NB / rpw) launches, rpw = min(NB, max(1, floor(2^28 / (tpr * 16384)))), NB = ceil(m/128),
 *                  with tpr = psa_align_pair_banded's for an empty chain and otherwise the largest number of 256-column
 *                  tiles a row block touches: the maximum over row blocks (rows i0+1 .. i0+r, r = min(128, m - i0)) of
 *                  s_hi - s_lo + 1, s_lo = floor((max(1, lo(i0+1)) - 1) / 256), s_hi = max(s_lo, floor((max(1, hi(i0+r)) - 1) / 256)).
 *   PSA_ERR_NOMEM as psa_align_pair_banded: if checkpoints and codes exceed half of the free device memory. */
typedef struct {
    int32_t i, j;
} psa_anchor;

int psa_align_batch_guided(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                           const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                           size_t bytes_a, size_t bytes_b, const psa_anchor* anchors, const int64_t* off_anc,
                           const int32_t* n_anc, size_t total_anc, int mode, int g, int h, int band, unsigned flags,
                           psa_batch_item* items, uint32_t* ops, size_t ops_stride_words);
int psa_align_batch_guided_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                  const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                  int max_len_a, int max_len_b, const psa_anchor* d_anchors, const int64_t* d_off_anc,
                                  const int32_t* d_n_anc, int mode, int g, int h, int band, unsigned flags,
                                  psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream);
int psa_align_pair_guided(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, const psa_anchor* anchors,
                          size_t n_anchors, int mode, int g, int h, int band, unsigned flags, psa_result* out);

/* ---- one long pair over several GPUs (config 4) ---------------------------------------------
 * Score-only fill of ONE pair by the column-stationary systolic kernel: the matrix is cut into panels of
 * panel_strips * psa_long_strip_columns() columns (one warp per strip -- 256 columns, 8 per lane -- every strip
 * of a panel resident at once, all m rows),
 * and the panels are dealt out block-cyclically: panel q belongs to rank q mod world (one process per GPU).  The
 * last strip of a panel streams its boundary column -- 8 bytes per row, validity tag in-band -- straight into the
 * NEXT rank's ring buffer through a peer-mapped pointer (NVLink P2P, system-scope stores); the first strip of the
 * next panel consumes it a few dozen rows later, so all GPUs work on the same anti-diagonal wavefront.  No NCCL on
 * the data path, no barrier between calls (rows are numbered cumulatively; the rings are never cleared).
 *   psa_long_panel_strips : resident strips of this GPU = the largest panel_strips it accepts; every rank must
 *                           pass the SAME panel_strips (e.g. the minimum over ranks)
 *   psa_long_strip_columns: columns per strip (the unit of panel_strips)
 *   psa_xbuf_create       : allocate this rank's INCOMING boundary buffer for pairs of up to m_cap rows (it holds a
 *                           whole column: a rank's panels run one after the other, so the panel that feeds its NEXT
 *                           panel must be able to finish first) + its IPC handle; pass the same m_cap to the align call
 *   psa_xbuf_open         : map rank (r + 1) mod world's incoming ring -> usable as d_xout_peer
 * Every rank holds the whole of A and B.  Local mode: every rank reports the best cell of ITS panels (global
 * coordinates); the caller keeps the maximum (score, then smallest end_i, then smallest end_j).  Global mode: the
 * rank that owns the last panel reports T1/T2/T3[m][n], the others PSA_NEG_INF.  world == 1 needs no rings and
 * equals psa_align_long_device without traceback.  Replaces nothing in the reference (24 TB of tables at 1 Mbp). */
size_t psa_xbuf_bytes(size_t m_cap);
int psa_xbuf_create(psa_ctx* ctx, size_t m_cap, void** d_xbuf, unsigned char ipc_handle[64]);
int psa_xbuf_open(psa_ctx* ctx, const unsigned char ipc_handle[64], void** d_peer);
int psa_xbuf_close(psa_ctx* ctx, void* d_peer);
int psa_xbuf_destroy(psa_ctx* ctx, void* d_xbuf);
int psa_long_panel_strips(psa_ctx* ctx);
int psa_long_strip_columns(psa_ctx* ctx);
int psa_align_long_cyclic_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int rank,
                                 int world, int panel_strips, int mode, int g, int h, size_t m_cap, void* d_xin,
                                 void* d_xout_peer, psa_batch_item* d_item, void* cuda_stream);

void psa_ops_unpack(const uint32_t* words, int32_t aln_len, uint8_t* ops_forward);
/* print_seq (main_alignment.cpp:32-55): expand forward ops into the two rows (no terminator). */
void psa_render_rows(const char* a, const char* b, const uint8_t* ops_forward, int64_t aln_len, int64_t start_i,
                     int64_t start_j, char* row_a, char* row_b);

/* ---- integer-pipe roofline microbenchmark (SURVEY 8d) -----------------------------------
 * Measures sustained warp-instruction issue of the cell-update instruction mix.
 * kind: 0 = VIADDMNMX+VIMNMX3 int32 mix, 1 = the same .S16x2, 2 = IADD3 only, 3 = IMAD only,
 *       4 = ALU+FMA interleaved, 5 = PRMT, 6 = IDP.4A
 * Returns lane-operations per second over the whole GPU in *lane_ops_per_s. */
int psa_peak_int_ops(psa_ctx* ctx, int kind, double* lane_ops_per_s, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* PSA_H */
