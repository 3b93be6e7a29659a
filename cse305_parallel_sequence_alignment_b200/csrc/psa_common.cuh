// psa_common.cuh -- shared definitions of libpsa (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <algorithm>
#include <string>

#include "../../include/psa.h"

// In-kernel stand-in for the reference's -infinity (subproblem_alignment.cpp:214-223).  Far
// enough from INT32_MIN that a few "- g - h" never wrap, far enough from real scores that it
// never wins a max.  Converted to PSA_NEG_INF at the API boundary (out_value, psa_result.cuh).
#define PSA_KNEG (-(1 << 29))

// Per-context tuning and measurement options (psa_internal.h: psa_ctx_set_option).  The shipped
// behaviour is the default value of every field; nothing on a launch path reads the environment.
struct psa_options {
    int pack = 1;                 // 0: never use the packed (.S16x2) kernels
    int pipeline = 1;             // 0: psa_align_batch copies everything first instead of the chunked pipeline
    int pack_traceback = 0;       // 0: per-cell direction codes in a recycled global ring (faster: DESIGN.md section 4);
                                  // 1: tile-boundary checkpoints + per-tile recompute (no code stream at all)
    int pack_skip_walk = 0;       // measurement only: fill launches without the traceback walk (results lack ops)
    int pack_ctas_per_sm = 0;     // > 0: cap of resident CTAs per SM of the packed fill kernel
    long long pack_chunk = 131072;
    int pack_serial_fills = 0;    // 1: host pipelines start fill(c) when fill(c-1) has finished, so chunks complete evenly spaced, in
                                  // order (0: the four in-flight fills share the SMs and finish together, their D2H in one burst)
    int pack_long_k = 0;          // 8 / 16: force the lane width of the packed long-batch kernel
    int long_geometry = -1;       // >= 0: force the tile geometry of the single long pair kernel (score only)
    int long_ctas_per_sm = 0;
    int long_band = 1;            // 0: no ahead-of-time band recompute before the checkpointed traceback walk
    long long long_tb_chunk = 0;  // > 0: cap of the pairs per chunk of a long traceback batch (tests: several chunks in one call)
    int long_systolic = -1;       // -1 auto, 0 never, 1 always: column-stationary systolic kernel for one long pair (score only)
    int systolic_warps_per_sm = 0;   // resident strips per SM (default 8)
    int systolic_kc = 8;          // columns per lane of the systolic kernel (4 or 8): 8 measured faster on 1 and on 8 GPUs (fewer strips = a
                                  // shorter pipeline ramp, at most one strip per warp scheduler of an 8-GPU share; DESIGN.md section 5)
    int systolic_rb = 4;          // rows per lane and step (1, 2 or 4)
    int timing = 0;               // 1: host-side phase timings on stderr; 2: + per-chunk GPU timeline
};

struct psa_ctx {
    int device = 0;
    psa_options opt;
    int smem_optin = 0;          // cudaDevAttrMaxSharedMemoryPerBlockOptin
    // stream ordering of the shared scratch: asynchronous device calls on different user streams are chained
    cudaEvent_t last_event = nullptr;
    cudaStream_t last_stream = nullptr;
    bool last_valid = false;
    cudaStream_t stream = nullptr;
    int sm_count = 0;
    int64_t launches = 0;
    int epoch = 0;               // internal call counter for epoch-biased progress counters
    std::string err;
    // reusable device scratch for the host-buffer entry points
    void* d_scratch = nullptr;
    size_t d_scratch_bytes = 0;
    void* h_pinned = nullptr;
    size_t h_pinned_bytes = 0;
    // boundary rows / checkpoints / flags of the long-pair kernels
    void* d_work = nullptr;
    size_t d_work_bytes = 0;
    // persistent state of the systolic kernel (rings + cumulative row counters; psa_systolic.cu)
    void* d_sys = nullptr;
    int sys_strips = 0;
    size_t sys_self_rows = 0;
    // internal streams/events: chunked fill/traceback overlap of the packed kernel
    cudaStream_t aux_stream[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t aux_event[3] = {nullptr, nullptr, nullptr};
    cudaStream_t post_stream = nullptr;     // compaction of the op words, chunk after chunk, off the fill streams (psa_pack_pipeline_packed)
};

inline int psa_fail(psa_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return code;
}

#define PSA_CUDA_OK(ctx, expr)                                                                       \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess)                                                                       \
            return psa_fail((ctx), PSA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

// Raises the dynamic shared-memory limit of `kern` to the device's opt-in maximum, once per (kernel, device)
// for the life of the process.  The attribute is per function, not per context: setting it to a call-specific
// size on every launch let concurrent host threads lower it under each other (round-1 failure).
int psa_kernel_optin_smem(psa_ctx* ctx, const void* kern);
// Stream ordering of ctx-owned scratch (d_work, aux streams): call at the start / end of every asynchronous
// device entry point.  A call on a different stream than the previous one first waits for that one's end.
int psa_stream_enter(psa_ctx* ctx, cudaStream_t st);
int psa_stream_leave(psa_ctx* ctx, cudaStream_t st);

// device-side description of one batch call
// Border variant of the pieces of one call (subproblem_alignment.cpp:212-227, :259-292, :112-146): one pair of types for
// all of them, or a host array with one byte per pair, (start_type + 3) | (end_type + 3) << 4.
struct psa_piece_types {
    int start_type = -1, end_type = -1;
    const uint8_t* per_pair = nullptr;
    bool any() const { return start_type != -1 || end_type != -1 || per_pair != nullptr; }
};

struct psa_batch_args {
    const uint8_t* bases_a;
    const int64_t* off_a;
    const int32_t* len_a;
    const uint8_t* bases_b;
    const int64_t* off_b;
    const int32_t* len_b;
    int64_t n_pairs;
    int g, h;
    psa_batch_item* items;
    uint32_t* ops;              // may be null (score only)
    int64_t ops_stride_words;
    // Subproblem border variants (subproblem_alignment.cpp:212-227, :259-292, :112-146); -1/-1 = the live case.
    // Implemented by the generic int32 short-pair kernel and the long-pair kernels.
    int start_type = -1;
    int end_type = -1;
    // 2-bit packed fixed-stride input (psa_align_batch_packed): bases_* / off_* / len_* are null; pair k's A is the
    // words a2[k*wa .. (k+1)*wa), base r in bits 2*(r%16) of word r/16 (A=0 C=1 T=2 G=3), every pair fixed_m x fixed_n
    const uint32_t* a2 = nullptr;
    const uint32_t* b2 = nullptr;
    int wa = 0, wb = 0;
    int fixed_m = 0, fixed_n = 0;
    const int* flagged_count = nullptr;   // optional, with a flag array: number of flagged pairs (0 = nothing to do, the flagged launch returns at once)
    const uint8_t* types = nullptr;   // optional, per pair: (start_type + 3) | (end_type + 3) << 4; overrides the two above
};

// Anchor chains of a guided batch (psa_align_batch_guided): pair k's chain is anchors[off[k] .. off[k] + n[k]).
struct psa_guide {
    const psa_anchor* anchors;
    const int64_t* off;
    const int32_t* n;
};

// launchers (each returns a psa_status and bumps ctx->launches)
int psa_launch_short(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                     cudaStream_t stream);
bool psa_short_supported(int max_m, int max_n, bool traceback);
// same kernel restricted to pairs whose flag byte is non-zero (device array, one byte per pair)
int psa_launch_short_flagged(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                             const uint8_t* d_flags, cudaStream_t stream);
bool psa_pack_supported(int max_m, int max_n, int mode, int g, int h);
int psa_launch_pack(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                    cudaStream_t stream);
// host-buffer pipelines over one chunk driver: per-chunk H2D -> fill -> traceback -> D2H, chunk c on aux stream c % 4
int psa_pack_pipeline(psa_ctx* ctx, const psa_batch_args& dev, const psa_batch_args& host, size_t bytes_a, size_t bytes_b,
                      int max_m, int max_n, int mode, bool traceback);
// the same pipeline for 2-bit packed fixed-stride input and 16-byte result records (psa_align_batch_packed)
int psa_pack_pipeline_packed(psa_ctx* ctx, const psa_batch_args& dev, const uint32_t* h_a2, const uint32_t* h_b2,
                             psa_packed_item* d_items16, psa_packed_item* h_items16, uint32_t* h_ops, int mode, bool traceback,
                             bool compact, uint8_t* d_compact);
int psa_launch_peak(psa_ctx* ctx, int kind, double* lane_ops_per_s, double* ms);
int psa_launch_similarity(psa_ctx* ctx, const psa_batch_args& args, int max_len, double* d_out, cudaStream_t st);
// column-stationary systolic kernel (psa_systolic.cu): the panels first_panel, first_panel + panel_step, ... of one pair
size_t psa_systolic_xbuf_bytes(size_t m_cap);
int psa_systolic_capacity(psa_ctx* ctx);
int psa_launch_systolic(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n_total, int mode, int g, int h,
                        int first_panel, int panel_step, int panel_strips, void* xin, void* xout, size_t x_m_cap,
                        psa_batch_item* d_item, cudaStream_t st);
int psa_launch_long_single(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h,
                           bool traceback, psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st,
                           int start_type = -1, int end_type = -1);
int psa_find_crossings(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, const uint8_t* d_ar, const uint8_t* d_br, int m, int n,
                       int g, int h, int max_rows, int* h_points, int* n_points, cudaStream_t st);
int psa_launch_long_batch(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st);
size_t psa_long_batch_scratch_bytes(psa_ctx* ctx, long long n_pairs, int max_n);
int psa_launch_long_batch_at(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode,
                             const uint8_t* d_flags, uint8_t* scratch, cudaStream_t st);
// Batch of long pairs with traceback: chunks of a checkpointed one-warp-per-pair fill + one-warp-per-pair walk (psa_long.cu).
// psa_long_batch_tb_chunk: pairs per chunk for this batch shape (0: one checkpoint slot exceeds the memory budget).
int psa_long_batch_tb_chunk(psa_ctx* ctx, long long n_pairs, int max_m, int max_n, int mode, long long* chunk);
int psa_launch_long_batch_tb(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st);
// Banded batch (psa_align_batch_banded): every pair on the banded tile kernels, one warp per pair (psa_long.cu).  With a
// guide (device arrays) each pair's band follows its anchor chain (psa_align_batch_guided[_device]).
int psa_launch_banded(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, int band, bool traceback,
                      cudaStream_t st, const psa_guide* guide = nullptr);
// One banded pair over the whole GPU (psa_align_pair_banded, psa_align_long_banded_device; psa_long.cu).
int psa_launch_banded_pair(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h, int band,
                           bool traceback, psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st);
// The same around a valid anchor chain (psa_align_pair_guided): planned from the host copy, run on the device copy.
int psa_launch_guided_pair(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h, int band,
                           const psa_anchor* h_anchors, const psa_anchor* d_anchors, int n_anchors, bool traceback,
                           psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st);
bool psa_pack_long_supported(int max_m, int max_n, int mode, int g, int h);
int psa_launch_pack_long(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st);
