// psa_capi.cu -- the extern "C" surface declared in include/psa.h.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>
#include <chrono>
#include <mutex>
#include <set>
#include <thread>
#include <utility>

#include "psa_common.cuh"
#include "psa_internal.h"

namespace {

thread_local std::string g_create_err;     // psa_last_error(NULL): the calling thread's last psa_ctx_create failure

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int ensure_scratch(psa_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->d_scratch_bytes) return PSA_OK;
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    ctx->d_scratch = nullptr;
    ctx->d_scratch_bytes = 0;
    bytes = align_up(bytes + bytes / 4, 1 << 20);
    if (cudaMalloc(&ctx->d_scratch, bytes) != cudaSuccess) {
        cudaGetLastError();
        return psa_fail(ctx, PSA_ERR_NOMEM, "cudaMalloc of batch scratch failed");
    }
    ctx->d_scratch_bytes = bytes;
    return PSA_OK;
}

int check_scoring(psa_ctx* ctx, int mode, int g, int h, int64_t max_m, int64_t max_n) {
    if (mode != PSA_GLOBAL && mode != PSA_LOCAL) return psa_fail(ctx, PSA_ERR_ARG, "mode must be PSA_GLOBAL or PSA_LOCAL");
    if (g < 0 || h < 0) return psa_fail(ctx, PSA_ERR_ARG, "g and h must be >= 0");
    const int64_t span = (int64_t)g * (max_m + max_n + 2) + 2 * (int64_t)h + max_m + max_n;
    if (span >= (1 << 28)) return psa_fail(ctx, PSA_ERR_RANGE, "score range exceeds int32 lanes");
    return PSA_OK;
}

// check_scoring for the banded entries.  Its bound counts three gap openings, which holds for the full matrix only: a
// band can force an opening on every row (n = 3m at band 1 needs a horizontal run of 2 per row).  An optimal path never
// puts a vertical run next to a horizontal one (one diagonal step replaces the corner, inside the band, for 2g less and
// a match or nothing), so its gap runs are separated by diagonals: at most min(m, n) + 1 of them, one more for a T2 / T3
// value that ends in a gap and one for the border run.  Global mode with band < max(m, n) therefore admits
// g(m+n+2) + h(min(m, n) + 3) + m + n < 2^28, which keeps out_value's threshold argument (psa_result.cuh) true.  Local
// values never fall below -(g+h), a band >= max(m, n) holds every cell and an empty side leaves no cell for the band
// to cut: those keep check_scoring's bound.  A batch is checked with its largest m and n.  The argument uses only that
// a corner's two end cells are in the band, so it covers the bands of anchor chains (psa_align_batch_guided) as well.
int check_banded_scoring(psa_ctx* ctx, int mode, int g, int h, int band, int64_t max_m, int64_t max_n) {
    int rc = check_scoring(ctx, mode, g, h, max_m, max_n);
    if (rc || mode != PSA_GLOBAL || band >= std::max(max_m, max_n) || std::min(max_m, max_n) == 0) return rc;
    const int64_t span = (int64_t)g * (max_m + max_n + 2) + (int64_t)h * (std::min(max_m, max_n) + 3) + max_m + max_n;
    if (span >= (1 << 28)) return psa_fail(ctx, PSA_ERR_RANGE, "banded score range exceeds int32 lanes");
    return PSA_OK;
}

// The host forms' chain check (psa_align_batch_guided, psa_align_pair_guided): pair k's anchors
// anchors[off[k] .. off[k] + cnt[k]) lie inside the array and form a valid chain for its lengths (include/psa.h).
int check_chains(psa_ctx* ctx, const psa_anchor* anchors, const int64_t* off, const int32_t* cnt, size_t total,
                 const int32_t* len_a, const int32_t* len_b, size_t n_pairs) {
    for (size_t k = 0; k < n_pairs; ++k) {
        const std::string pair = "pair " + std::to_string(k) + ": ";
        if (cnt[k] < 0 || off[k] < 0 || (uint64_t)off[k] + (uint64_t)cnt[k] > total)
            return psa_fail(ctx, PSA_ERR_ARG, pair + "anchor range outside the anchor array");
        const psa_anchor* c = anchors + off[k];
        for (int32_t q = 0; q < cnt[k]; ++q) {
            if (c[q].i < 0 || c[q].i > len_a[k] || c[q].j < 0 || c[q].j > len_b[k])
                return psa_fail(ctx, PSA_ERR_ARG, pair + "anchor " + std::to_string(q) + " outside the matrix");
            if (q > 0 && (c[q].i < c[q - 1].i || c[q].j < c[q - 1].j))
                return psa_fail(ctx, PSA_ERR_ARG, pair + "anchor " + std::to_string(q) + " decreases a coordinate of the chain");
        }
    }
    return PSA_OK;
}

int dispatch_batch(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, unsigned flags,
                   cudaStream_t stream) {
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && !args.ops) return psa_fail(ctx, PSA_ERR_ARG, "traceback requested without an ops buffer");
    if (tb && args.ops_stride_words * 16 < (int64_t)max_m + max_n)
        return psa_fail(ctx, PSA_ERR_CAPACITY, "ops_stride_words < ceil((max m + max n)/16)");
    if (args.start_type != -1 || args.end_type != -1 || args.types != nullptr) {
        if (mode != PSA_GLOBAL) return psa_fail(ctx, PSA_ERR_ARG, "start/end types apply to global alignment only");
        if (psa_short_supported(max_m, max_n, tb)) return psa_launch_short(ctx, args, max_m, max_n, mode, tb, stream);
        if (tb) return psa_launch_long_batch_tb(ctx, args, max_m, max_n, mode, stream);
        return psa_fail(ctx, PSA_ERR_RANGE, "typed subproblems wider than 256 columns need PSA_WANT_TRACEBACK on the device entry");
    }
    if (psa_short_supported(max_m, max_n, tb)) {
        // DNA fast path (two pairs per register, .S16x2); non-ACGT members fall through to the generic kernel inside
        if (args.n_pairs >= 64 && ctx->opt.pack && psa_pack_supported(max_m, max_n, mode, args.g, args.h))
            return psa_launch_pack(ctx, args, max_m, max_n, mode, tb, stream);
        return psa_launch_short(ctx, args, max_m, max_n, mode, tb, stream);
    }
    if (!tb) {
        if (args.n_pairs >= 2 && ctx->opt.pack && psa_pack_long_supported(max_m, max_n, mode, args.g, args.h))
            return psa_launch_pack_long(ctx, args, max_m, max_n, mode, stream);
        return psa_launch_long_batch(ctx, args, max_m, max_n, mode, stream);
    }
    return psa_launch_long_batch_tb(ctx, args, max_m, max_n, mode, stream);
}

}  // namespace

int psa_kernel_optin_smem(psa_ctx* ctx, const void* kern) {
    static std::mutex mu;
    static std::set<std::pair<const void*, int>> done;
    std::lock_guard<std::mutex> hold(mu);
    if (done.count({kern, ctx->device})) return PSA_OK;
    cudaFuncAttributes fa;
    PSA_CUDA_OK(ctx, cudaFuncGetAttributes(&fa, kern));
    // the opt-in maximum covers static + dynamic shared memory of a block
    PSA_CUDA_OK(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_optin - (int)fa.sharedSizeBytes));
    done.insert({kern, ctx->device});
    return PSA_OK;
}

int psa_stream_enter(psa_ctx* ctx, cudaStream_t st) {
    if (ctx->last_valid && ctx->last_stream != st) PSA_CUDA_OK(ctx, cudaStreamWaitEvent(st, ctx->last_event, 0));
    return PSA_OK;
}

int psa_stream_leave(psa_ctx* ctx, cudaStream_t st) {
    PSA_CUDA_OK(ctx, cudaEventRecord(ctx->last_event, st));
    ctx->last_stream = st;
    ctx->last_valid = true;
    return PSA_OK;
}

extern "C" {

int psa_ctx_set_option(psa_ctx* ctx, const char* name, long long value) {
    if (!ctx || !name) return PSA_ERR_ARG;
    psa_options& o = ctx->opt;
    const std::string k(name);
    if (k == "pack") o.pack = (int)value;
    else if (k == "pipeline") o.pipeline = (int)value;
    else if (k == "pack_traceback") o.pack_traceback = (int)value;
    else if (k == "pack_skip_walk") o.pack_skip_walk = (int)value;
    else if (k == "pack_ctas_per_sm") o.pack_ctas_per_sm = (int)value;
    else if (k == "pack_chunk") o.pack_chunk = value < 1024 ? 1024 : value;
    else if (k == "pack_serial_fills") o.pack_serial_fills = (int)value;
    else if (k == "pack_long_k") o.pack_long_k = (int)value;
    else if (k == "long_geometry") o.long_geometry = (int)value;
    else if (k == "long_ctas_per_sm") o.long_ctas_per_sm = (int)value;
    else if (k == "long_band") o.long_band = (int)value;
    else if (k == "long_tb_chunk") o.long_tb_chunk = value;
    else if (k == "long_systolic") o.long_systolic = (int)value;
    else if (k == "systolic_warps_per_sm") o.systolic_warps_per_sm = (int)value;
    else if (k == "systolic_kc") o.systolic_kc = (int)value;
    else if (k == "systolic_rb") o.systolic_rb = (int)value;
    else if (k == "timing") o.timing = (int)value;
    else return psa_fail(ctx, PSA_ERR_ARG, "psa_ctx_set_option: unknown option '" + k + "'");
    return PSA_OK;
}

int psa_ctx_create(int device, psa_ctx** out) {
    if (!out) return PSA_ERR_ARG;
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        g_create_err = std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0");
        cudaGetLastError();
        return PSA_ERR_CUDA;
    }
    if (device < 0 || device >= n_dev) { g_create_err = "device index out of range"; return PSA_ERR_ARG; }
    psa_ctx* ctx = new (std::nothrow) psa_ctx();
    if (!ctx) return PSA_ERR_NOMEM;
    ctx->device = device;
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&ctx->last_event, cudaEventDisableTiming)) != cudaSuccess) {
        g_create_err = std::string("context setup: ") + cudaGetErrorString(e);
        delete ctx;
        return PSA_ERR_CUDA;
    }
    if (prop.major < 10) {
        g_create_err = "libpsa is built for sm_100a only; device is sm_" + std::to_string(prop.major * 10 + prop.minor);
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return PSA_ERR_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    *out = ctx;
    return PSA_OK;
}

void psa_ctx_destroy(psa_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->d_work) cudaFree(ctx->d_work);
    if (ctx->d_sys) cudaFree(ctx->d_sys);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    for (int k = 0; k < 4; ++k) if (ctx->aux_stream[k]) cudaStreamDestroy(ctx->aux_stream[k]);
    if (ctx->post_stream) cudaStreamDestroy(ctx->post_stream);
    for (int k = 0; k < 3; ++k) if (ctx->aux_event[k]) cudaEventDestroy(ctx->aux_event[k]);
    if (ctx->last_event) cudaEventDestroy(ctx->last_event);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* psa_last_error(const psa_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int64_t psa_launch_count(const psa_ctx* ctx) { return ctx ? ctx->launches : 0; }

int psa_align_batch_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                           const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b,
                           size_t n_pairs, int max_len_a, int max_len_b, int mode, int g, int h, unsigned flags,
                           psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (n_pairs == 0) return PSA_OK;
    if (!d_bases_a || !d_bases_b || !d_off_a || !d_off_b || !d_len_a || !d_len_b || !d_items)
        return psa_fail(ctx, PSA_ERR_ARG, "null device pointer");
    if (max_len_a < 0 || max_len_b < 0) return psa_fail(ctx, PSA_ERR_ARG, "negative length bound");
    int rc = check_scoring(ctx, mode, g, h, max_len_a, max_len_b);
    if (rc) return rc;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    psa_batch_args args{d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, (int64_t)n_pairs, g, h,
                        d_items, d_ops, (int64_t)ops_stride_words};
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = dispatch_batch(ctx, args, max_len_a, max_len_b, mode, flags, st);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

}  // extern "C"

// Pairs of a host-buffer traceback batch of long pairs from which the batched path (one warp per pair) replaces the
// per-pair loop (each pair over the whole GPU).  Sweep of 1 - 64 pairs (profiles/r03_long_tb.json, same box): at 16 pairs
// the batch is at least as fast in every series (5 kbp local 38.6 vs 38.7 ms, global 28.9 vs 40.0; 1 kbp local 2.9 vs
// 8.1, global 1.4 vs 8.3); at 8 pairs the per-pair loop still wins at 5 kbp (19.4 vs 34.9 ms local, 20.0 vs 21.2 global).
constexpr int kLongTbBatchMin = 16;

// Host-buffer batch with an optional border variant per call or per pair; psa_align_batch is the -1/-1 case.
// band >= 0: psa_align_batch_banded (every pair on the banded kernels); with guide (host arrays of total_anc anchors)
// psa_align_batch_guided.
static int align_batch_host(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                            const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                            size_t bytes_a, size_t bytes_b, int mode, int g, int h, unsigned flags,
                            psa_batch_item* items, uint32_t* ops, size_t ops_stride_words, const psa_piece_types& ty,
                            int band = -1, const psa_guide* guide = nullptr, size_t total_anc = 0) {
    if (!ctx) return PSA_ERR_ARG;
    if (n_pairs == 0) return PSA_OK;
    if (!off_a || !off_b || !len_a || !len_b || !items || (!bases_a && bytes_a) || (!bases_b && bytes_b))
        return psa_fail(ctx, PSA_ERR_ARG, "null host pointer");
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && !ops) return psa_fail(ctx, PSA_ERR_ARG, "traceback requested without an ops buffer");
    const auto t_begin = std::chrono::steady_clock::now();
    int max_m = 0, max_n = 0;
    bool contiguous = true;      // offsets ascending, every sequence starting where the previous one ended
    {
        // branch-free pass, split over a few host threads: harness-sized batches have 10^6 pairs (24 MB of
        // offsets/lengths) and this scan sits inside the end-to-end time
        const int T = n_pairs >= (1u << 19) ? 8 : (n_pairs >= (1u << 17) ? 4 : 1);
        struct Part { int mm, mn, lo; int64_t off, bad, gap; } parts[8];
        auto scan = [&](int t) {
            const size_t k0 = n_pairs * t / T, k1 = n_pairs * (t + 1) / T;
            Part q{0, 0, 0, 0, 0, 0};
            for (size_t k = k0; k < k1; ++k) {
                q.mm = std::max(q.mm, len_a[k]);
                q.mn = std::max(q.mn, len_b[k]);
                q.lo = std::min(q.lo, std::min(len_a[k], len_b[k]));
                q.off = std::min(q.off, std::min(off_a[k], off_b[k]));
                q.bad |= (int64_t)((uint64_t)off_a[k] + (uint64_t)(uint32_t)len_a[k] > (uint64_t)bytes_a);
                q.bad |= (int64_t)((uint64_t)off_b[k] + (uint64_t)(uint32_t)len_b[k] > (uint64_t)bytes_b);
                if (k + 1 < n_pairs) q.gap |= (off_a[k + 1] - off_a[k] - len_a[k]) | (off_b[k + 1] - off_b[k] - len_b[k]);
            }
            parts[t] = q;
        };
        if (T == 1) scan(0);
        else {
            std::thread th[7];
            for (int t = 1; t < T; ++t) th[t - 1] = std::thread(scan, t);
            scan(0);
            for (int t = 1; t < T; ++t) th[t - 1].join();
        }
        int mn_len = 0;
        int64_t mn_off = 0, bad = 0, gap = 0;
        for (int t = 0; t < T; ++t) {
            max_m = std::max(max_m, parts[t].mm); max_n = std::max(max_n, parts[t].mn);
            mn_len = std::min(mn_len, parts[t].lo); mn_off = std::min(mn_off, parts[t].off);
            bad |= parts[t].bad; gap |= parts[t].gap;
        }
        contiguous = (gap == 0);
        if (mn_len < 0 || mn_off < 0 || bad) {
            for (size_t k = 0; k < n_pairs; ++k)
                if (len_a[k] < 0 || len_b[k] < 0 || off_a[k] < 0 || off_b[k] < 0 ||
                    (size_t)off_a[k] + (size_t)len_a[k] > bytes_a || (size_t)off_b[k] + (size_t)len_b[k] > bytes_b)
                    return psa_fail(ctx, PSA_ERR_ARG, "pair " + std::to_string(k) + ": offset/length outside the base arrays");
        }
    }
    int rc = band >= 0 ? check_banded_scoring(ctx, mode, g, h, band, max_m, max_n) : check_scoring(ctx, mode, g, h, max_m, max_n);
    if (rc) return rc;
    if (guide) {
        if (!guide->off || !guide->n || (!guide->anchors && total_anc)) return psa_fail(ctx, PSA_ERR_ARG, "null anchor array");
        rc = check_chains(ctx, guide->anchors, guide->off, guide->n, total_anc, len_a, len_b, n_pairs);
        if (rc) return rc;
    }
    if (tb && ops_stride_words * 16 < (size_t)max_m + max_n)
        return psa_fail(ctx, PSA_ERR_CAPACITY, "ops_stride_words < ceil((max m + max n)/16)");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    // an asynchronous device call of this context may still be using the shared scratch on a user stream
    if (ctx->last_valid) { PSA_CUDA_OK(ctx, cudaEventSynchronize(ctx->last_event)); ctx->last_valid = false; }

    // device layout: [bases_a | bases_b | off_a | off_b | len_a | len_b | items | ops]
    size_t o = 0;
    const size_t o_ba = o; o = align_up(o + std::max<size_t>(bytes_a, 1), 256);
    const size_t o_bb = o; o = align_up(o + std::max<size_t>(bytes_b, 1), 256);
    const size_t o_oa = o; o = align_up(o + n_pairs * 8, 256);
    const size_t o_ob = o; o = align_up(o + n_pairs * 8, 256);
    const size_t o_la = o; o = align_up(o + n_pairs * 4, 256);
    const size_t o_lb = o; o = align_up(o + n_pairs * 4, 256);
    const size_t o_it = o; o = align_up(o + n_pairs * sizeof(psa_batch_item), 256);
    const size_t o_op = o; o = align_up(o + (tb ? n_pairs * ops_stride_words * 4 : 0), 256);
    const size_t o_ty = o; o = align_up(o + (ty.per_pair ? n_pairs : 0), 256);
    // guided: [anchors | off_anc | n_anc]
    const size_t o_an = o; o = align_up(o + (guide ? total_anc * sizeof(psa_anchor) : 0), 256);
    const size_t o_ao = o; o = align_up(o + (guide ? n_pairs * 8 : 0), 256);
    const size_t o_ac = o; o = align_up(o + (guide ? n_pairs * 4 : 0), 256);
    rc = ensure_scratch(ctx, o);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_scratch;
    cudaStream_t st = ctx->stream;
    psa_batch_args args{d + o_ba, (const int64_t*)(d + o_oa), (const int32_t*)(d + o_la), d + o_bb,
                        (const int64_t*)(d + o_ob), (const int32_t*)(d + o_lb), (int64_t)n_pairs, g, h,
                        (psa_batch_item*)(d + o_it), tb ? (uint32_t*)(d + o_op) : nullptr, (int64_t)ops_stride_words};
    args.start_type = ty.start_type; args.end_type = ty.end_type;
    if (ty.per_pair) {
        args.types = d + o_ty;
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ty, ty.per_pair, n_pairs, cudaMemcpyHostToDevice, st));
    }
    const bool typed = ty.any();
    // large DNA batches laid out back to back: chunked copy/compute pipeline on the four aux streams
    if (band < 0 && !typed && contiguous && n_pairs > (size_t)ctx->opt.pack_chunk && psa_short_supported(max_m, max_n, tb) &&
        psa_pack_supported(max_m, max_n, mode, g, h) && ctx->opt.pack && ctx->opt.pipeline) {
        psa_batch_args host{bases_a, off_a, len_a, bases_b, off_b, len_b, (int64_t)n_pairs, g, h, items, ops,
                            (int64_t)ops_stride_words};
        const auto t_valid = std::chrono::steady_clock::now();
        rc = psa_pack_pipeline(ctx, args, host, bytes_a, bytes_b, max_m, max_n, mode, tb);
        if (ctx->opt.timing) {
            const auto t_end = std::chrono::steady_clock::now();
            fprintf(stderr, "psa_align_batch: validate %.3f ms, pipeline %.3f ms\n",
                    std::chrono::duration<double, std::milli>(t_valid - t_begin).count(),
                    std::chrono::duration<double, std::milli>(t_end - t_valid).count());
        }
        return rc;
    }
    if (bytes_a) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ba, bases_a, bytes_a, cudaMemcpyHostToDevice, st));
    if (bytes_b) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_bb, bases_b, bytes_b, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_oa, off_a, n_pairs * 8, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ob, off_b, n_pairs * 8, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_la, len_a, n_pairs * 4, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_lb, len_b, n_pairs * 4, cudaMemcpyHostToDevice, st));
    const psa_guide d_guide{(const psa_anchor*)(d + o_an), (const int64_t*)(d + o_ao), (const int32_t*)(d + o_ac)};
    if (guide) {
        if (total_anc) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_an, guide->anchors, total_anc * sizeof(psa_anchor), cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ao, guide->off, n_pairs * 8, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ac, guide->n, n_pairs * 4, cudaMemcpyHostToDevice, st));
    }
    const bool is_short = psa_short_supported(max_m, max_n, tb);
    if (typed && mode != PSA_GLOBAL) return psa_fail(ctx, PSA_ERR_ARG, "start/end types apply to global alignment only");
    // long pairs with traceback: from kLongTbBatchMin pairs on, one warp per pair (checkpointed batch fill + batched walk)
    // unless one pair's checkpoints exceed the memory budget
    long long tb_chunk = 0;
    if (band < 0 && !is_short && tb && n_pairs >= (size_t)kLongTbBatchMin) {
        rc = psa_long_batch_tb_chunk(ctx, (long long)n_pairs, max_m, max_n, mode, &tb_chunk);
        if (rc) return rc;
    }
    if (band >= 0) {
        rc = psa_launch_banded(ctx, args, max_m, max_n, mode, band, tb, st, guide ? &d_guide : nullptr);
        if (rc) return rc;
    } else if (is_short || (!typed && !tb && n_pairs > 8) || tb_chunk > 0) {
        rc = dispatch_batch(ctx, args, max_m, max_n, mode, flags, st);
        if (rc) return rc;
    } else {
        // long pairs (and typed pieces wider than the short kernel takes): each pair gets the whole GPU
        // (row-block wavefront across all SMs)
        for (size_t k = 0; k < n_pairs && rc == PSA_OK; ++k) {
            const int st_k = ty.per_pair ? (int)(ty.per_pair[k] & 15) - 3 : ty.start_type;
            const int et_k = ty.per_pair ? (int)(ty.per_pair[k] >> 4) - 3 : ty.end_type;
            psa_batch_item* d_item = (psa_batch_item*)(d + o_it) + k;
            uint32_t* d_ops_k = tb ? (uint32_t*)(d + o_op) + k * ops_stride_words : nullptr;
            if (len_a[k] == 0 || len_b[k] == 0) {     // borders only: the short kernel's degenerate branch
                psa_batch_args one = args;
                one.off_a += k; one.len_a += k; one.off_b += k; one.len_b += k; one.n_pairs = 1;
                one.items = d_item; one.ops = d_ops_k;
                if (one.types) one.types += k;
                rc = psa_launch_short(ctx, one, 1, 1, mode, tb, st);
            } else {
                rc = psa_launch_long_single(ctx, d + o_ba + off_a[k], d + o_bb + off_b[k], len_a[k], len_b[k], mode, g, h,
                                            tb, d_item, d_ops_k, st, st_k, et_k);
            }
        }
        if (rc) return rc;
    }
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(items, d + o_it, n_pairs * sizeof(psa_batch_item), cudaMemcpyDeviceToHost, st));
    if (tb) PSA_CUDA_OK(ctx, cudaMemcpyAsync(ops, d + o_op, n_pairs * ops_stride_words * 4, cudaMemcpyDeviceToHost, st));
    PSA_CUDA_OK(ctx, cudaStreamSynchronize(st));
    return PSA_OK;
}

extern "C" {

int psa_align_batch(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                    const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                    size_t bytes_a, size_t bytes_b, int mode, int g, int h, unsigned flags,
                    psa_batch_item* items, uint32_t* ops, size_t ops_stride_words) {
    return align_batch_host(ctx, bases_a, off_a, len_a, bases_b, off_b, len_b, n_pairs, bytes_a, bytes_b, mode, g, h, flags,
                            items, ops, ops_stride_words, psa_piece_types{});
}

int psa_align_batch_banded(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                           const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                           size_t bytes_a, size_t bytes_b, int mode, int g, int h, int band, unsigned flags,
                           psa_batch_item* items, uint32_t* ops, size_t ops_stride_words) {
    if (!ctx) return PSA_ERR_ARG;
    if (band < 0) return psa_fail(ctx, PSA_ERR_ARG, "band must be >= 0");
    if (flags & ~(PSA_WANT_SCORE | PSA_WANT_TRACEBACK)) return psa_fail(ctx, PSA_ERR_ARG, "flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only");
    return align_batch_host(ctx, bases_a, off_a, len_a, bases_b, off_b, len_b, n_pairs, bytes_a, bytes_b, mode, g, h, flags,
                            items, ops, ops_stride_words, psa_piece_types{}, band);
}

int psa_align_batch_banded_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                  const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                  int max_len_a, int max_len_b, int mode, int g, int h, int band, unsigned flags,
                                  psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (band < 0) return psa_fail(ctx, PSA_ERR_ARG, "band must be >= 0");
    if (flags & ~(PSA_WANT_SCORE | PSA_WANT_TRACEBACK)) return psa_fail(ctx, PSA_ERR_ARG, "flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only");
    if (n_pairs == 0) return PSA_OK;
    if (!d_bases_a || !d_bases_b || !d_off_a || !d_off_b || !d_len_a || !d_len_b || !d_items)
        return psa_fail(ctx, PSA_ERR_ARG, "null device pointer");
    if (max_len_a < 0 || max_len_b < 0) return psa_fail(ctx, PSA_ERR_ARG, "negative length bound");
    int rc = check_banded_scoring(ctx, mode, g, h, band, max_len_a, max_len_b);
    if (rc) return rc;
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && !d_ops) return psa_fail(ctx, PSA_ERR_ARG, "traceback requested without an ops buffer");
    if (tb && ops_stride_words * 16 < (size_t)max_len_a + max_len_b)
        return psa_fail(ctx, PSA_ERR_CAPACITY, "ops_stride_words < ceil((max m + max n)/16)");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    psa_batch_args args{d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, (int64_t)n_pairs, g, h,
                        d_items, tb ? d_ops : nullptr, (int64_t)ops_stride_words};
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = psa_launch_banded(ctx, args, max_len_a, max_len_b, mode, band, tb, st);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

int psa_align_batch_guided(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                           const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                           size_t bytes_a, size_t bytes_b, const psa_anchor* anchors, const int64_t* off_anc,
                           const int32_t* n_anc, size_t total_anc, int mode, int g, int h, int band, unsigned flags,
                           psa_batch_item* items, uint32_t* ops, size_t ops_stride_words) {
    if (!ctx) return PSA_ERR_ARG;
    if (band < 0) return psa_fail(ctx, PSA_ERR_ARG, "band must be >= 0");
    if (flags & ~(PSA_WANT_SCORE | PSA_WANT_TRACEBACK)) return psa_fail(ctx, PSA_ERR_ARG, "flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only");
    const psa_guide guide{anchors, off_anc, n_anc};
    return align_batch_host(ctx, bases_a, off_a, len_a, bases_b, off_b, len_b, n_pairs, bytes_a, bytes_b, mode, g, h, flags,
                            items, ops, ops_stride_words, psa_piece_types{}, band, &guide, total_anc);
}

int psa_align_batch_guided_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                  const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                  int max_len_a, int max_len_b, const psa_anchor* d_anchors, const int64_t* d_off_anc,
                                  const int32_t* d_n_anc, int mode, int g, int h, int band, unsigned flags,
                                  psa_batch_item* d_items, uint32_t* d_ops, size_t ops_stride_words, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (band < 0) return psa_fail(ctx, PSA_ERR_ARG, "band must be >= 0");
    if (flags & ~(PSA_WANT_SCORE | PSA_WANT_TRACEBACK)) return psa_fail(ctx, PSA_ERR_ARG, "flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only");
    if (n_pairs == 0) return PSA_OK;
    if (!d_bases_a || !d_bases_b || !d_off_a || !d_off_b || !d_len_a || !d_len_b || !d_items || !d_anchors || !d_off_anc || !d_n_anc)
        return psa_fail(ctx, PSA_ERR_ARG, "null device pointer");
    if (max_len_a < 0 || max_len_b < 0) return psa_fail(ctx, PSA_ERR_ARG, "negative length bound");
    int rc = check_banded_scoring(ctx, mode, g, h, band, max_len_a, max_len_b);
    if (rc) return rc;
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && !d_ops) return psa_fail(ctx, PSA_ERR_ARG, "traceback requested without an ops buffer");
    if (tb && ops_stride_words * 16 < (size_t)max_len_a + max_len_b)
        return psa_fail(ctx, PSA_ERR_CAPACITY, "ops_stride_words < ceil((max m + max n)/16)");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    psa_batch_args args{d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, (int64_t)n_pairs, g, h,
                        d_items, tb ? d_ops : nullptr, (int64_t)ops_stride_words};
    const psa_guide guide{d_anchors, d_off_anc, d_n_anc};
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = psa_launch_banded(ctx, args, max_len_a, max_len_b, mode, band, tb, st, &guide);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

// Argument rules shared by both forms of the one-pair banded entry (the host form handles m = 0 or n = 0 itself).
static int check_banded_pair(psa_ctx* ctx, size_t m, size_t n, int mode, int g, int h, int band, unsigned flags) {
    if (band < 0) return psa_fail(ctx, PSA_ERR_ARG, "band must be >= 0");
    if (flags & ~(PSA_WANT_SCORE | PSA_WANT_TRACEBACK)) return psa_fail(ctx, PSA_ERR_ARG, "flags: PSA_WANT_SCORE and PSA_WANT_TRACEBACK only");
    if (m >= 0x1FFFFF || n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    return check_banded_scoring(ctx, mode, g, h, band, (int64_t)m, (int64_t)n);
}

int psa_align_long_banded_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int mode, int g,
                                 int h, int band, unsigned flags, psa_batch_item* d_item, uint32_t* d_ops, size_t ops_words,
                                 void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (!d_a || !d_b || !d_item || m == 0 || n == 0) return psa_fail(ctx, PSA_ERR_ARG, "null pointer or empty sequence");
    int rc = check_banded_pair(ctx, m, n, mode, g, h, band, flags);
    if (rc) return rc;
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && (!d_ops || ops_words * 16 < m + n)) return psa_fail(ctx, PSA_ERR_CAPACITY, "ops buffer < ceil((m+n)/16) words");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = psa_launch_banded_pair(ctx, d_a, d_b, (int)m, (int)n, mode, g, h, band, tb, d_item, d_ops, st);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

int psa_align_long_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int mode, int g, int h,
                          unsigned flags, psa_batch_item* d_item, uint32_t* d_ops, size_t ops_words, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (!d_a || !d_b || !d_item || m == 0 || n == 0) return psa_fail(ctx, PSA_ERR_ARG, "null pointer or empty sequence");
    if (m > (size_t)INT32_MAX || n > (size_t)INT32_MAX) return psa_fail(ctx, PSA_ERR_RANGE, "length exceeds int32");
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && (!d_ops || ops_words * 16 < m + n)) return psa_fail(ctx, PSA_ERR_CAPACITY, "ops buffer < ceil((m+n)/16) words");
    int rc = check_scoring(ctx, mode, g, h, (int64_t)m, (int64_t)n);
    if (rc) return rc;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = psa_launch_long_single(ctx, d_a, d_b, (int)m, (int)n, mode, g, h, tb, d_item, d_ops, st);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

size_t psa_xbuf_bytes(size_t m_cap) { return psa_systolic_xbuf_bytes(m_cap); }

int psa_xbuf_create(psa_ctx* ctx, size_t m_cap, void** d_xbuf, unsigned char ipc_handle[64]) {
    if (!ctx || !d_xbuf || !ipc_handle || m_cap == 0) return psa_fail(ctx, PSA_ERR_ARG, "psa_xbuf_create: bad argument");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    void* p = nullptr;
    const size_t bytes = psa_systolic_xbuf_bytes(m_cap);
    if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return psa_fail(ctx, PSA_ERR_NOMEM, "psa_xbuf_create: cudaMalloc"); }
    PSA_CUDA_OK(ctx, cudaMemset(p, 0, bytes));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t hnd;
    PSA_CUDA_OK(ctx, cudaIpcGetMemHandle(&hnd, p));
    memcpy(ipc_handle, &hnd, 64);
    *d_xbuf = p;
    return PSA_OK;
}

int psa_xbuf_open(psa_ctx* ctx, const unsigned char ipc_handle[64], void** d_peer) {
    if (!ctx || !d_peer || !ipc_handle) return psa_fail(ctx, PSA_ERR_ARG, "psa_xbuf_open: bad argument");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, ipc_handle, 64);
    PSA_CUDA_OK(ctx, cudaIpcOpenMemHandle(d_peer, hnd, cudaIpcMemLazyEnablePeerAccess));
    return PSA_OK;
}

int psa_xbuf_close(psa_ctx* ctx, void* d_peer) {
    if (!ctx) return PSA_ERR_ARG;
    if (d_peer) PSA_CUDA_OK(ctx, cudaIpcCloseMemHandle(d_peer));
    return PSA_OK;
}

int psa_xbuf_destroy(psa_ctx* ctx, void* d_xbuf) {
    if (!ctx) return PSA_ERR_ARG;
    if (d_xbuf) PSA_CUDA_OK(ctx, cudaFree(d_xbuf));
    return PSA_OK;
}

int psa_long_panel_strips(psa_ctx* ctx) { return ctx ? psa_systolic_capacity(ctx) : 0; }
int psa_long_strip_columns(psa_ctx* ctx) { return ctx ? 32 * (ctx->opt.systolic_kc == 4 ? 4 : 8) : 0; }

int psa_align_long_cyclic_device(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, size_t m, size_t n, int rank,
                                 int world, int panel_strips, int mode, int g, int h, size_t m_cap, void* d_xin,
                                 void* d_xout_peer, psa_batch_item* d_item, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (!d_a || !d_b || !d_item || m == 0 || n == 0 || world < 1 || rank < 0 || rank >= world || panel_strips < 1)
        return psa_fail(ctx, PSA_ERR_ARG, "psa_align_long_cyclic_device: bad argument");
    if (world > 1 && (!d_xin || !d_xout_peer)) return psa_fail(ctx, PSA_ERR_ARG, "several ranks need the inter-GPU rings");
    if (m > (size_t)INT32_MAX || n > (size_t)INT32_MAX) return psa_fail(ctx, PSA_ERR_RANGE, "length exceeds int32");
    int rc = check_scoring(ctx, mode, g, h, (int64_t)m, (int64_t)n);
    if (rc) return rc;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    rc = psa_stream_enter(ctx, st);
    if (rc) return rc;
    rc = psa_launch_systolic(ctx, d_a, d_b, (int)m, (int)n, mode, g, h, rank, world, panel_strips,
                             world > 1 ? d_xin : nullptr, world > 1 ? d_xout_peer : nullptr, m_cap, d_item, st);
    if (rc) return rc;
    return psa_stream_leave(ctx, st);
}

size_t psa_pack_bases(const uint8_t* bases, size_t n, uint32_t* packed) {
    size_t bad = 0;
    for (size_t w = 0; w * 16 < n; ++w) {
        uint32_t v = 0;
        const size_t e = std::min<size_t>(16, n - w * 16);
        for (size_t x = 0; x < e; ++x) {
            const uint8_t c = bases[w * 16 + x];
            bad += !(c == 'A' || c == 'C' || c == 'G' || c == 'T');
            v |= (uint32_t)((c >> 1) & 3u) << (2 * x);
        }
        packed[w] = v;
    }
    return bad;
}

int psa_align_batch_packed(psa_ctx* ctx, const uint32_t* a2, const uint32_t* b2, size_t n_pairs, int len_a, int len_b,
                           int mode, int g, int h, unsigned flags, psa_packed_item* items, uint32_t* ops,
                           size_t ops_stride_words) {
    if (!ctx) return PSA_ERR_ARG;
    if (n_pairs == 0) return PSA_OK;
    if (!a2 || !b2 || !items || len_a < 1 || len_b < 1) return psa_fail(ctx, PSA_ERR_ARG, "psa_align_batch_packed: null pointer or empty reads");
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    if (tb && !ops) return psa_fail(ctx, PSA_ERR_ARG, "traceback requested without an ops buffer");
    if (tb && ops_stride_words * 16 < (size_t)len_a + len_b) return psa_fail(ctx, PSA_ERR_CAPACITY, "ops_stride_words < ceil((len_a + len_b)/16)");
    int rc = check_scoring(ctx, mode, g, h, len_a, len_b);
    if (rc) return rc;
    if (!psa_short_supported(len_a, len_b, tb) || !psa_pack_supported(len_a, len_b, mode, g, h))
        return psa_fail(ctx, PSA_ERR_RANGE, "psa_align_batch_packed serves reads up to 512 x 256 with h <= 2; use psa_align_batch");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    if (ctx->last_valid) { PSA_CUDA_OK(ctx, cudaEventSynchronize(ctx->last_event)); ctx->last_valid = false; }
    const int wa = (len_a + 15) / 16, wb = (len_b + 15) / 16;
    size_t o = 0;
    const size_t o_a = o; o = align_up(o + n_pairs * wa * 4, 256);
    const size_t o_b = o; o = align_up(o + n_pairs * wb * 4, 256);
    const size_t o_it = o; o = align_up(o + n_pairs * sizeof(psa_batch_item), 256);
    const size_t o_i16 = o; o = align_up(o + n_pairs * sizeof(psa_packed_item), 256);
    const size_t o_op = o; o = align_up(o + (tb ? n_pairs * ops_stride_words * 4 : 0), 256);
    // compact ops: scan scratch (offsets, CTA sums, chunk bases) and the device buffer the words are packed into
    const bool compact = tb && (flags & PSA_OPS_COMPACT) != 0;
    const size_t o_cp = o;
    if (compact) o = align_up(o + align_up(n_pairs, 256) * 4 + 4096 * 128 * 4 + 4096 * 8 + 256 + n_pairs * ops_stride_words * 4, 256);
    rc = ensure_scratch(ctx, o);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_scratch;
    psa_batch_args args{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, (int64_t)n_pairs, g, h,
                        (psa_batch_item*)(d + o_it), tb ? (uint32_t*)(d + o_op) : nullptr, (int64_t)ops_stride_words};
    args.a2 = (const uint32_t*)(d + o_a); args.b2 = (const uint32_t*)(d + o_b);
    args.wa = wa; args.wb = wb; args.fixed_m = len_a; args.fixed_n = len_b;
    return psa_pack_pipeline_packed(ctx, args, a2, b2, (psa_packed_item*)(d + o_i16), items, ops, mode, tb, compact, d + o_cp);
}

void psa_ops_unpack(const uint32_t* words, int32_t aln_len, uint8_t* ops_forward) {
    for (int32_t k = 0; k < aln_len; ++k)
        ops_forward[aln_len - 1 - k] = (uint8_t)((words[k >> 4] >> (2 * (k & 15))) & 3u);
}

void psa_render_rows(const char* a, const char* b, const uint8_t* ops, int64_t len, int64_t start_i, int64_t start_j,
                     char* row_a, char* row_b) {
    // print_seq (main_alignment.cpp:32-55): line 1 shows A[i] for states 1/3, line 2 B[j] for 1/2
    int64_t i = start_i, j = start_j;
    for (int64_t k = 0; k < len; ++k) {
        if (k > 0) {
            if (ops[k] != 2) ++i;
            if (ops[k] != 3) ++j;
        }
        row_a[k] = (ops[k] == 1 || ops[k] == 3) ? a[i - 1] : '-';
        row_b[k] = (ops[k] == 1 || ops[k] == 2) ? b[j - 1] : '-';
    }
}

}  // extern "C"

// Gives *out library-owned ops and rows for `len` alignment columns (rows NUL-terminated) and sets aln_len; the caller
// fills ops and renders the rows.  On allocation failure frees what was allocated.
static int alloc_alignment(psa_ctx* ctx, psa_result* out, int64_t len) {
    out->ops = (uint8_t*)malloc((size_t)len + 1);
    out->row_a = (char*)malloc((size_t)len + 1);
    out->row_b = (char*)malloc((size_t)len + 1);
    if (!out->ops || !out->row_a || !out->row_b) { psa_result_free(out); return psa_fail(ctx, PSA_ERR_NOMEM, "malloc"); }
    out->row_a[len] = 0; out->row_b[len] = 0;
    out->aln_len = len;
    return PSA_OK;
}

// *out from one pair's record and, with traceback (words != null), its op words: ops, then rows through psa_render_rows.
static int fill_result(psa_ctx* ctx, psa_result* out, const psa_batch_item& it, const uint32_t* words, const char* a, const char* b) {
    out->t1 = it.t1; out->t2 = it.t2; out->t3 = it.t3; out->score = it.score; out->end_state = it.end_state;
    out->end_i = it.end_i; out->end_j = it.end_j; out->start_i = it.start_i; out->start_j = it.start_j;
    out->aln_len = it.aln_len;
    if (words) {
        int rc = alloc_alignment(ctx, out, it.aln_len);
        if (rc) return rc;
        psa_ops_unpack(words, it.aln_len, out->ops);
        psa_render_rows(a, b, out->ops, it.aln_len, it.start_i, it.start_j, out->row_a, out->row_b);
    }
    return PSA_OK;
}

static bool ok_type(int t) { return t == -1 || t == -2 || t == -3 || t == 1 || t == 2 || t == 3; }

static int align_pair_impl(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int mode, int g, int h,
                           unsigned flags, psa_result* out, const psa_piece_types& ty) {
    if (!ctx) return PSA_ERR_ARG;
    if (!out || (!a && m) || (!b && n)) return psa_fail(ctx, PSA_ERR_ARG, "null pointer");
    if (m > (size_t)INT32_MAX || n > (size_t)INT32_MAX) return psa_fail(ctx, PSA_ERR_RANGE, "length exceeds int32");
    memset(out, 0, sizeof(*out));
    const int64_t off = 0;
    const int32_t lm = (int32_t)m, ln = (int32_t)n;
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    const size_t stride = (m + n + 15) / 16 + 1;
    std::vector<uint32_t> words(tb ? stride : 0);
    psa_batch_item it;
    int rc = align_batch_host(ctx, (const uint8_t*)a, &off, &lm, (const uint8_t*)b, &off, &ln, 1, m, n, mode, g, h,
                              flags, &it, tb ? words.data() : nullptr, stride, ty);
    if (rc) return rc;
    return fill_result(ctx, out, it, tb ? words.data() : nullptr, a, b);
}

extern "C" {

int psa_align_pair(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int mode, int g, int h,
                   unsigned flags, psa_result* out) {
    return align_pair_impl(ctx, a, b, m, n, mode, g, h, flags, out, psa_piece_types{});
}

int psa_align_pair_banded(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int mode, int g, int h, int band,
                          unsigned flags, psa_result* out) {
    if (!ctx) return PSA_ERR_ARG;
    if (!out || (!a && m) || (!b && n)) return psa_fail(ctx, PSA_ERR_ARG, "null pointer");
    int rc = check_banded_pair(ctx, m, n, mode, g, h, band, flags);
    if (rc) return rc;
    if (m == 0 || n == 0) return align_pair_impl(ctx, a, b, m, n, mode, g, h, flags, out, psa_piece_types{});
    memset(out, 0, sizeof(*out));
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    const size_t words = (m + n + 15) / 16 + 1;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    // an asynchronous device call of this context may still be using the shared scratch on a user stream
    if (ctx->last_valid) { PSA_CUDA_OK(ctx, cudaEventSynchronize(ctx->last_event)); ctx->last_valid = false; }
    const size_t o_a = 0, o_b = align_up(m, 256), o_it = o_b + align_up(n, 256), o_op = o_it + 256;
    rc = ensure_scratch(ctx, o_op + (tb ? words * 4 : 0));
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_scratch;
    cudaStream_t st = ctx->stream;
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_a, a, m, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_b, b, n, cudaMemcpyHostToDevice, st));
    rc = psa_launch_banded_pair(ctx, d + o_a, d + o_b, (int)m, (int)n, mode, g, h, band, tb, (psa_batch_item*)(d + o_it),
                                tb ? (uint32_t*)(d + o_op) : nullptr, st);
    if (rc) return rc;
    psa_batch_item it;
    std::vector<uint32_t> w(tb ? words : 0);
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(&it, d + o_it, sizeof(it), cudaMemcpyDeviceToHost, st));
    if (tb) PSA_CUDA_OK(ctx, cudaMemcpyAsync(w.data(), d + o_op, words * 4, cudaMemcpyDeviceToHost, st));
    PSA_CUDA_OK(ctx, cudaStreamSynchronize(st));
    return fill_result(ctx, out, it, tb ? w.data() : nullptr, a, b);
}

int psa_align_pair_guided(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, const psa_anchor* anchors,
                          size_t n_anchors, int mode, int g, int h, int band, unsigned flags, psa_result* out) {
    if (!ctx) return PSA_ERR_ARG;
    if (!out || (!a && m) || (!b && n) || (!anchors && n_anchors)) return psa_fail(ctx, PSA_ERR_ARG, "null pointer");
    int rc = check_banded_pair(ctx, m, n, mode, g, h, band, flags);
    if (rc) return rc;
    if (n_anchors > (size_t)INT32_MAX) return psa_fail(ctx, PSA_ERR_ARG, "more than 2^31 - 1 anchors");
    const int64_t off0 = 0;
    const int32_t cnt = (int32_t)n_anchors, lm = (int32_t)m, ln = (int32_t)n;
    rc = check_chains(ctx, anchors, &off0, &cnt, n_anchors, &lm, &ln, 1);
    if (rc) return rc;
    if (m == 0 || n == 0) return align_pair_impl(ctx, a, b, m, n, mode, g, h, flags, out, psa_piece_types{});
    memset(out, 0, sizeof(*out));
    const bool tb = (flags & PSA_WANT_TRACEBACK) != 0;
    const size_t words = (m + n + 15) / 16 + 1;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    // an asynchronous device call of this context may still be using the shared scratch on a user stream
    if (ctx->last_valid) { PSA_CUDA_OK(ctx, cudaEventSynchronize(ctx->last_event)); ctx->last_valid = false; }
    const size_t o_a = 0, o_b = align_up(m, 256), o_an = o_b + align_up(n, 256);
    const size_t o_it = o_an + align_up(n_anchors * sizeof(psa_anchor), 256), o_op = o_it + 256;
    rc = ensure_scratch(ctx, o_op + (tb ? words * 4 : 0));
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_scratch;
    cudaStream_t st = ctx->stream;
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_a, a, m, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_b, b, n, cudaMemcpyHostToDevice, st));
    if (n_anchors) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_an, anchors, n_anchors * sizeof(psa_anchor), cudaMemcpyHostToDevice, st));
    rc = psa_launch_guided_pair(ctx, d + o_a, d + o_b, (int)m, (int)n, mode, g, h, band, anchors, (const psa_anchor*)(d + o_an),
                                cnt, tb, (psa_batch_item*)(d + o_it), tb ? (uint32_t*)(d + o_op) : nullptr, st);
    if (rc) return rc;
    psa_batch_item it;
    std::vector<uint32_t> w(tb ? words : 0);
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(&it, d + o_it, sizeof(it), cudaMemcpyDeviceToHost, st));
    if (tb) PSA_CUDA_OK(ctx, cudaMemcpyAsync(w.data(), d + o_op, words * 4, cudaMemcpyDeviceToHost, st));
    PSA_CUDA_OK(ctx, cudaStreamSynchronize(st));
    return fill_result(ctx, out, it, tb ? w.data() : nullptr, a, b);
}

int psa_align_pair_typed(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int start_type, int end_type,
                         int g, int h, unsigned flags, psa_result* out) {
    if (!ctx) return PSA_ERR_ARG;
    if (!ok_type(start_type) || !ok_type(end_type)) return psa_fail(ctx, PSA_ERR_ARG, "start/end type must be one of -1,-2,-3,1,2,3");
    if (m == 0 || n == 0) return psa_fail(ctx, PSA_ERR_ARG, "typed subproblems need m, n >= 1");
    psa_piece_types ty;
    ty.start_type = start_type; ty.end_type = end_type;
    return align_pair_impl(ctx, a, b, m, n, PSA_GLOBAL, g, h, flags, out, ty);
}

int psa_align_partition(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, const psa_bp* bp, size_t n_bp,
                        int g, int h, psa_result* out) {
    if (!ctx) return PSA_ERR_ARG;
    if (!out || !bp || (!a && m) || (!b && n)) return psa_fail(ctx, PSA_ERR_ARG, "null pointer");
    if (n_bp < 2) return psa_fail(ctx, PSA_ERR_ARG, "a partition needs at least two points");
    const size_t np = n_bp - 1;
    std::vector<int64_t> off_a(np), off_b(np);
    std::vector<int32_t> len_a(np), len_b(np);
    std::vector<uint8_t> types(np);
    size_t max_a = 0, max_b = 0;
    for (size_t k = 0; k < n_bp; ++k) {
        if (bp[k].i < 0 || bp[k].j < 0 || (uint64_t)bp[k].i > m || (uint64_t)bp[k].j > n || !ok_type(bp[k].t))
            return psa_fail(ctx, PSA_ERR_ARG, "partition point " + std::to_string(k) + " outside the matrix or with a bad type");
        if (k + 1 < n_bp) {
            if (bp[k + 1].i < bp[k].i || bp[k + 1].j < bp[k].j)
                return psa_fail(ctx, PSA_ERR_ARG, "partition points must not decrease");
            if (bp[k + 1].i - bp[k].i > INT32_MAX || bp[k + 1].j - bp[k].j > INT32_MAX)
                return psa_fail(ctx, PSA_ERR_RANGE, "piece exceeds int32");
            off_a[k] = bp[k].i; off_b[k] = bp[k].j;
            len_a[k] = (int32_t)(bp[k + 1].i - bp[k].i); len_b[k] = (int32_t)(bp[k + 1].j - bp[k].j);
            // piece k runs from point k to point k+1 (main_alignment.cpp:240-251): its start type is the type of
            // point k, its end type the negated type of point k+1
            types[k] = (uint8_t)((bp[k].t + 3) | ((-bp[k + 1].t + 3) << 4));
            max_a = std::max(max_a, (size_t)len_a[k]); max_b = std::max(max_b, (size_t)len_b[k]);
        }
    }
    const size_t stride = (max_a + max_b + 15) / 16 + 1;
    memset(out, 0, sizeof(*out));
    std::vector<psa_batch_item> items(np);
    std::vector<uint32_t> words(np * stride);
    psa_piece_types ty;
    ty.per_pair = types.data();
    int rc = align_batch_host(ctx, (const uint8_t*)a, off_a.data(), len_a.data(), (const uint8_t*)b, off_b.data(),
                              len_b.data(), np, m, n, PSA_GLOBAL, g, h, PSA_WANT_SCORE | PSA_WANT_TRACEBACK,
                              items.data(), words.data(), stride, ty);
    if (rc) return rc;
    int64_t total = 0;
    for (size_t k = 0; k < np; ++k) total += items[k].aln_len;
    rc = alloc_alignment(ctx, out, total);
    if (rc) return rc;
    int64_t at = 0;
    bool first = true;
    for (size_t k = 0; k < np; ++k) {            // link the pieces in order (main_alignment.cpp:343-347)
        const psa_batch_item& it = items[k];
        if (it.aln_len == 0) continue;
        psa_ops_unpack(words.data() + k * stride, it.aln_len, out->ops + at);
        psa_render_rows(a + off_a[k], b + off_b[k], out->ops + at, it.aln_len, it.start_i, it.start_j, out->row_a + at,
                        out->row_b + at);
        if (first) { out->start_i = off_a[k] + it.start_i; out->start_j = off_b[k] + it.start_j; first = false; }
        at += it.aln_len;
    }
    const psa_batch_item& last = items[np - 1];
    out->t1 = last.t1; out->t2 = last.t2; out->t3 = last.t3; out->end_state = last.end_state;
    out->end_i = bp[n_bp - 1].i; out->end_j = bp[n_bp - 1].j;
    // score of the linked alignment as printed: +1 per matching column, h + g*k per run of k gap columns
    int64_t score = 0;
    int prev = 0;
    for (int64_t k = 0; k < total; ++k) {
        const int t = out->ops[k];
        if (t == 1) score += (out->row_a[k] == out->row_b[k]) ? 1 : 0;
        else score -= (t == prev ? 0 : h) + g;
        prev = t;
    }
    out->score = (int32_t)score;
    return PSA_OK;
}

// SURVEY 8 f-3: partition finder + stitched alignment -- the job sequence_alignment/partial.cpp:81-163 and
// optimal_alignment (main_alignment.cpp:202-351) were meant to do together.
int psa_align_long_partitioned(psa_ctx* ctx, const char* a, const char* b, size_t m, size_t n, int g, int h, int pieces,
                               psa_result* out, psa_bp* bp_out, size_t bp_cap, size_t* n_bp) {
    if (!ctx) return PSA_ERR_ARG;
    if (!out || !a || !b || m == 0 || n == 0 || pieces < 1) return psa_fail(ctx, PSA_ERR_ARG, "psa_align_long_partitioned: bad argument");
    if (m > (size_t)INT32_MAX || n > (size_t)INT32_MAX) return psa_fail(ctx, PSA_ERR_RANGE, "length exceeds int32");
    int rc = check_scoring(ctx, PSA_GLOBAL, g, h, (int64_t)m, (int64_t)n);
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    if (n_bp) *n_bp = 0;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    if (ctx->last_valid) { PSA_CUDA_OK(ctx, cudaEventSynchronize(ctx->last_event)); ctx->last_valid = false; }
    // ---- crossing points: forward sweep of (A, B), reverse sweep of the reversed sequences ----
    std::vector<int> pts(4 * (size_t)std::max(pieces, 1));
    int npts = 0;
    if (pieces > 1) {
        const size_t o_a = 0, o_b = align_up(m, 256), o_ar = o_b + align_up(n, 256), o_br = o_ar + align_up(m, 256);
        rc = ensure_scratch(ctx, o_br + align_up(n, 256));
        if (rc) return rc;
        uint8_t* d = (uint8_t*)ctx->d_scratch;
        std::vector<char> ar(a, a + m), br(b, b + n);
        std::reverse(ar.begin(), ar.end());
        std::reverse(br.begin(), br.end());
        cudaStream_t st = ctx->stream;
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_a, a, m, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_b, b, n, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ar, ar.data(), m, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_br, br.data(), n, cudaMemcpyHostToDevice, st));
        rc = psa_find_crossings(ctx, d + o_a, d + o_b, d + o_ar, d + o_br, (int)m, (int)n, g, h, pieces - 1, pts.data(), &npts, st);
        if (rc) return rc;
    }
    struct Pt { int64_t i, j; int t; };
    auto rescore = [&](const std::vector<uint8_t>& ops) -> int64_t {
        int64_t sc = 0, i = 0, j = 0;
        int prev = 0;
        for (uint8_t t : ops) {
            if (t == 1) { sc += (a[i] == b[j]) ? 1 : 0; ++i; ++j; }
            else { sc -= (t == prev ? 0 : h) + g; if (t == 2) ++j; else ++i; }
            prev = t;
        }
        return (i == (int64_t)m && j == (int64_t)n) ? sc : INT64_MIN;
    };
    // Solve the pieces between consecutive points as typed subproblems and stitch them.  A type-3 point sits inside a
    // vertical gap: the piece before it must END in T3 (end type 3), the piece after it CONTINUES the gap without a
    // second opening penalty (start type -3, subproblem_alignment.cpp:282-292).  Returns false if the pieces do not
    // add up to one complete alignment (possible only when tied co-optimal paths cross between two special rows).
    auto stitch = [&](const std::vector<Pt>& P, std::vector<uint8_t>& ops, psa_result* last) -> int {
        ops.clear();
        for (size_t k = 0; k + 1 < P.size(); ++k) {
            const int64_t mi = P[k + 1].i - P[k].i, nj = P[k + 1].j - P[k].j;
            if (mi < 0 || nj < 0) return 1;
            if (mi == 0 || nj == 0) { ops.insert(ops.end(), (size_t)(mi + nj), (uint8_t)(mi == 0 ? 2 : 3)); continue; }
            psa_piece_types ty;
            ty.start_type = (k > 0 && P[k].t == 3) ? -3 : -1;
            ty.end_type = (k + 2 < P.size() && P[k + 1].t == 3) ? 3 : -1;
            psa_result r;
            const int prc = align_pair_impl(ctx, a + P[k].i, b + P[k].j, (size_t)mi, (size_t)nj, PSA_GLOBAL, g, h,
                                            PSA_WANT_SCORE | PSA_WANT_TRACEBACK, &r, ty);
            if (prc) return prc;
            int64_t ri = 0, ci = 0;
            for (int64_t x = 0; x < r.aln_len; ++x) { ri += r.ops[x] != 2; ci += r.ops[x] != 3; }
            const int64_t dr = mi - ri, dc = nj - ci;      // the border run find_alignment drops (cpp:170)
            const bool ok = dr >= 0 && dc >= 0 && (dr == 0 || dc == 0);
            if (ok) {
                ops.insert(ops.end(), (size_t)(dr + dc), (uint8_t)(dr > 0 ? 3 : 2));
                ops.insert(ops.end(), r.ops, r.ops + r.aln_len);
            }
            if (last && k + 2 == P.size()) { last->t1 = r.t1; last->t2 = r.t2; last->t3 = r.t3; last->end_state = r.end_state; }
            psa_result_free(&r);
            if (!ok) return 1;
        }
        return 0;
    };
    std::vector<Pt> P;
    P.push_back({0, 0, -1});
    int64_t opt = INT64_MIN;
    for (int k = 0; k < npts; ++k) {
        opt = pts[4 * k + 3];
        if (pts[4 * k + 1] >= P.back().j) P.push_back({pts[4 * k + 0], pts[4 * k + 1], pts[4 * k + 2]});
    }
    P.push_back({(int64_t)m, (int64_t)n, -1});
    std::vector<uint8_t> ops;
    psa_result last;
    memset(&last, 0, sizeof(last));
    // tries: all crossings, then the middle one alone, then no cut at all -- each verified against the optimum
    for (int attempt = 0; attempt < 3; ++attempt) {
        std::vector<Pt> Q = P;
        if (attempt == 1 && P.size() > 3) { Q = {P.front(), P[P.size() / 2], P.back()}; }
        else if (attempt == 1) continue;
        if (attempt == 2) Q = {P.front(), P.back()};
        rc = stitch(Q, ops, &last);
        if (rc < 0) return rc;
        if (rc == 0) {
            const int64_t sc = rescore(ops);
            if (sc != INT64_MIN && (opt == INT64_MIN || sc == opt || Q.size() == 2)) {
                P = Q;
                rc = alloc_alignment(ctx, out, (int64_t)ops.size());
                if (rc) return rc;
                memcpy(out->ops, ops.data(), ops.size());
                // cell of the first column in print_seq's convention: a leading gap sits on the border row / column 0
                const int64_t si = (!ops.empty() && ops[0] == 2) ? 0 : 1, sj = (!ops.empty() && ops[0] == 3) ? 0 : 1;
                psa_render_rows(a, b, out->ops, out->aln_len, si, sj, out->row_a, out->row_b);
                out->score = (int32_t)sc;
                out->t1 = last.t1; out->t2 = last.t2; out->t3 = last.t3; out->end_state = last.end_state;
                out->end_i = (int64_t)m; out->end_j = (int64_t)n; out->start_i = si; out->start_j = sj;
                const size_t inner = P.size() - 2;
                if (n_bp) *n_bp = inner;
                for (size_t k = 0; bp_out && k < inner && k < bp_cap; ++k) bp_out[k] = psa_bp{P[k + 1].i, P[k + 1].j, P[k + 1].t, 0};
                return PSA_OK;
            }
        }
    }
    return psa_fail(ctx, PSA_ERR_CUDA, "psa_align_long_partitioned: pieces do not add up (internal error)");
}

void psa_result_free(psa_result* r) {
    if (!r) return;
    free(r->ops); free(r->row_a); free(r->row_b);
    r->ops = nullptr; r->row_a = nullptr; r->row_b = nullptr;
}

int psa_similarity_batch_device(psa_ctx* ctx, const uint8_t* d_bases_a, const int64_t* d_off_a, const int32_t* d_len_a,
                                const uint8_t* d_bases_b, const int64_t* d_off_b, const int32_t* d_len_b, size_t n_pairs,
                                int max_len, double* d_out, void* cuda_stream) {
    if (!ctx) return PSA_ERR_ARG;
    if (n_pairs == 0) return PSA_OK;
    if (!d_bases_a || !d_bases_b || !d_off_a || !d_off_b || !d_len_a || !d_len_b || !d_out)
        return psa_fail(ctx, PSA_ERR_ARG, "null device pointer");
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    psa_batch_args args{d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, (int64_t)n_pairs, 0, 0, nullptr, nullptr, 0};
    return psa_launch_similarity(ctx, args, max_len, d_out, cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream);
}

int psa_similarity_batch(psa_ctx* ctx, const uint8_t* bases_a, const int64_t* off_a, const int32_t* len_a,
                         const uint8_t* bases_b, const int64_t* off_b, const int32_t* len_b, size_t n_pairs,
                         size_t bytes_a, size_t bytes_b, double* out) {
    if (!ctx) return PSA_ERR_ARG;
    if (n_pairs == 0) return PSA_OK;
    if (!off_a || !off_b || !len_a || !len_b || !out || (!bases_a && bytes_a) || (!bases_b && bytes_b))
        return psa_fail(ctx, PSA_ERR_ARG, "null host pointer");
    int max_len = 0;
    for (size_t k = 0; k < n_pairs; ++k) {
        if (len_a[k] < 0 || len_b[k] < 0 || off_a[k] < 0 || off_b[k] < 0 || (size_t)off_a[k] + (size_t)len_a[k] > bytes_a ||
            (size_t)off_b[k] + (size_t)len_b[k] > bytes_b)
            return psa_fail(ctx, PSA_ERR_ARG, "pair " + std::to_string(k) + ": offset/length outside the base arrays");
        max_len = std::max(max_len, std::max(len_a[k], len_b[k]));
    }
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    size_t o = 0;
    const size_t o_ba = o; o = align_up(o + std::max<size_t>(bytes_a, 1), 256);
    const size_t o_bb = o; o = align_up(o + std::max<size_t>(bytes_b, 1), 256);
    const size_t o_oa = o; o = align_up(o + n_pairs * 8, 256);
    const size_t o_ob = o; o = align_up(o + n_pairs * 8, 256);
    const size_t o_la = o; o = align_up(o + n_pairs * 4, 256);
    const size_t o_lb = o; o = align_up(o + n_pairs * 4, 256);
    const size_t o_out = o; o = align_up(o + n_pairs * 8, 256);
    int rc = ensure_scratch(ctx, o);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_scratch;
    cudaStream_t st = ctx->stream;
    if (bytes_a) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ba, bases_a, bytes_a, cudaMemcpyHostToDevice, st));
    if (bytes_b) PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_bb, bases_b, bytes_b, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_oa, off_a, n_pairs * 8, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_ob, off_b, n_pairs * 8, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_la, len_a, n_pairs * 4, cudaMemcpyHostToDevice, st));
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_lb, len_b, n_pairs * 4, cudaMemcpyHostToDevice, st));
    psa_batch_args args{d + o_ba, (const int64_t*)(d + o_oa), (const int32_t*)(d + o_la), d + o_bb,
                        (const int64_t*)(d + o_ob), (const int32_t*)(d + o_lb), (int64_t)n_pairs, 0, 0, nullptr, nullptr, 0};
    rc = psa_launch_similarity(ctx, args, max_len, (double*)(d + o_out), st);
    if (rc) return rc;
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(out, d + o_out, n_pairs * 8, cudaMemcpyDeviceToHost, st));
    PSA_CUDA_OK(ctx, cudaStreamSynchronize(st));
    return PSA_OK;
}

int psa_peak_int_ops(psa_ctx* ctx, int kind, double* lane_ops_per_s, double* ms) {
    if (!ctx || !lane_ops_per_s) return PSA_ERR_ARG;
    PSA_CUDA_OK(ctx, cudaSetDevice(ctx->device));
    return psa_launch_peak(ctx, kind, lane_ops_per_s, ms);
}

}  // extern "C"
