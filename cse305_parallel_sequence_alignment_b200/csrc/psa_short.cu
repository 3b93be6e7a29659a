// psa_short.cu -- inter-pair kernel for batches of short pairs (BASELINE configs 1 and 2).
//
// One warp per pair.  Lane t owns K consecutive columns (K = ceil(n/32) <= 8, so n <= 256); the
// warp sweeps the rows as a skewed wavefront: at step s lane t works on row s - t, receiving the
// (H, E) of the column to its left from lane t-1 by warp shuffle -- the B200 replacement for the
// reference's per-row fork/join over column blocks + ParallelPrefixMax
// (subproblem_alignment.cpp:251-327, :29-103).  Sequences are staged in shared memory.
//
// Recurrence (subproblem_alignment.cpp:229-249, :396-398), with E = T2, F = T3, H = max(T1,T2,T3):
//     T1 = H[i-1][j-1] + (A[i]==B[j])          (local: max(0, H[i-1][j-1]) + ...)
//     E  = max(H[i][j-1] - g - h, E[i][j-1] - g)      == the reference's T2 because h >= 0
//     F  = max(H[i-1][j] - g - h, F[i-1][j] - g)      == the reference's T3
//
// Traceback without an O(mn) table in HBM: every cell leaves a 4-bit code in SHARED memory that
// is enough to replay find_alignment()'s first-equality order (subproblem_alignment.cpp:147-169):
//     d1 = first of T1,T2,T3 equal to H          (bits 0-1; 0 = "H == 0" in local mode: the floor)
//     z2 = d1==1 ? (E + h > H) : (E + h >= H)    (bit 2)  -> predecessor of a T2 state to the right
//     e3 = (F + h > H)                           (bit 3)  -> predecessor of a T3 state below
// Lane 0 then walks the codes and writes 2-bit ops.
#include "psa_result.cuh"

namespace {

constexpr int kMaxK = 8;

template <int K, int MODE, bool TB>
__global__ void __launch_bounds__(256) psa_short_kernel(psa_batch_args P, int sa_stride, int sb_stride,
                                                         int per_warp_bytes, const uint8_t* only_flagged) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int wpb = blockDim.x >> 5;
    uint8_t* sA = smem + (size_t)warp * per_warp_bytes;
    uint8_t* sB = sA + sa_stride;
    uint32_t* dirs = reinterpret_cast<uint32_t*>(sB + sb_stride);
    const int g = P.g, go = P.g + P.h, h = P.h;
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    if (only_flagged != nullptr && P.flagged_count != nullptr && *P.flagged_count == 0) return;   // nothing flagged in this chunk

    for (int64_t p = (int64_t)blockIdx.x * wpb + warp; p < P.n_pairs; p += (int64_t)gridDim.x * wpb) {
        if (only_flagged != nullptr && only_flagged[p] == 0) continue;
        const int m = P.len_a[p], n = P.len_b[p];
        psa_batch_item* item = P.items + p;
        const int st = P.types ? (int)(P.types[p] & 15) - 3 : P.start_type;
        const int et = P.types ? (int)(P.types[p] >> 4) - 3 : P.end_type;
        if (m <= 0 || n <= 0) {   // degenerate: borders only (subproblem_alignment.cpp:259-292)
            if (lane == 0) *item = empty_item<MODE>(m, n, g, h, st, et);
            continue;
        }
        // ---- stage both sequences (coalesced byte loads) ----
        {
            const uint8_t* ga = P.bases_a + P.off_a[p];
            const uint8_t* gb = P.bases_b + P.off_b[p];
            for (int i = lane; i < m; i += 32) sA[i] = ga[i];
            for (int j = lane; j < n; j += 32) sB[j] = gb[j];
        }
        __syncwarp();

        const int c0 = lane * K;   // columns c0+1 .. c0+K (1-based)
        int Hc[K], Fc[K], bcol[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int j = c0 + k + 1;
            bcol[k] = (j <= n) ? (int)sB[j - 1] : 256;          // 256 never equals a byte
            Hc[k] = LOCAL ? PSA_KNEG : border_row0_H<PSA_GLOBAL>(j, g, h, st);     // row 0: T2[0][j] (cpp:216-224)
            Fc[k] = PSA_KNEG;
        }
        int hd = LOCAL ? PSA_KNEG : border_row0_H<PSA_GLOBAL>(c0, g, h, st);   // H[0][c0]; the single 0 of row 0 sits at (0,0) (cpp:261-272)
        int recv_h = PSA_KNEG, recv_e = PSA_KNEG;
        int best = 0, bi = 0, bj = 0;           // local: best T1 and its first cell in this lane
        int c1 = PSA_KNEG, c2 = PSA_KNEG, c3 = PSA_KNEG;   // global: corner capture

        const int steps = m + 31;
        for (int s = 0; s < steps; ++s) {
            const int i = s - lane + 1;
            int hl, el;
            if (lane == 0) { hl = LOCAL ? PSA_KNEG : border_col0_H<PSA_GLOBAL>(i, g, h, st); el = PSA_KNEG; }   // T3[i][0] (cpp:284-292)
            else { hl = recv_h; el = recv_e; }
            if (i >= 1 && i <= m) {
                const int a = sA[i - 1];
                const int hl0 = hl;
                int diag = hd;
                uint32_t word = 0;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int t1 = (LOCAL ? imax(diag, 0) : diag) + (a == bcol[k] ? 1 : 0);
                    const int e = imax(hl - go, el - g);
                    const int f = imax(Hc[k] - go, Fc[k] - g);
                    const int H = imax(t1, imax(e, f));
                    if (TB) {
                        int d1 = (t1 == H) ? 1 : (e >= f ? 2 : 3);
                        const int z2 = (d1 == 1) ? (e + h > H) : (e + h >= H);
                        const int e3 = (f + h > H);
                        if (LOCAL && H == 0) d1 = 0;
                        word |= (uint32_t)(d1 | (z2 << 2) | (e3 << 3)) << (4 * k);
                    }
                    if (LOCAL) {
                        if (t1 > best && c0 + k < n) { best = t1; bi = i; bj = c0 + k + 1; }
                    } else {
                        if (i == m && c0 + k + 1 == n) { c1 = t1; c2 = e; c3 = f; }
                    }
                    diag = Hc[k]; Hc[k] = H; Fc[k] = f; hl = H; el = e;
                }
                hd = hl0;
                if (TB) dirs[(i - 1) * 32 + lane] = word;
            }
            recv_h = __shfl_up_sync(0xffffffffu, hl, 1);
            recv_e = __shfl_up_sync(0xffffffffu, el, 1);
        }

        // ---- gather the result ----
        psa_batch_item r;
        if (LOCAL) {
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const int ob = __shfl_xor_sync(0xffffffffu, best, off);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
                const bool take = (ob > best) || (ob == best && (oi < bi || (oi == bi && oj < bj)));
                if (take) { best = ob; bi = oi; bj = oj; }
            }
            r = local_item(best, best > 0 ? bi : 0, best > 0 ? bj : 0);
        } else {
            const int src = (n - 1) / K;
            c1 = __shfl_sync(0xffffffffu, c1, src);
            c2 = __shfl_sync(0xffffffffu, c2, src);
            c3 = __shfl_sync(0xffffffffu, c3, src);
            r = global_item(c1, c2, c3, m, n, h, et);
        }

        if (TB) {
            __syncwarp();
            if (lane == 0) {
                uint32_t* ow = P.ops + p * P.ops_stride_words;
                uint32_t acc = 0;
                int len = 0;
                int i = (int)r.end_i, j = (int)r.end_j, state = r.end_state;
                while (i > 0 && j > 0) {
                    acc |= (uint32_t)state << (2 * (len & 15));
                    if ((len & 15) == 15) { ow[len >> 4] = acc; acc = 0; }
                    ++len;
                    r.start_i = i; r.start_j = j;
                    // predecessor (source) cell of this state
                    const int si = (state == 2) ? i : i - 1;
                    const int sj = (state == 3) ? j : j - 1;
                    int code = 0;
                    const bool border = (si == 0 || sj == 0);
                    if (!border) code = (dirs[(si - 1) * 32 + (sj - 1) / K] >> (4 * ((sj - 1) % K))) & 15;
                    state = next_state<MODE>(state, code, border);
                    if (state == 0) break;     // nothing precedes this column: the 0 floor of a local alignment, or a border source
                    i = si; j = sj;
                    // on the border the predecessor node is the one find_alignment() drops (cpp:170)
                }
                if (len & 15) ow[len >> 4] = acc;
                r.aln_len = len;
            }
        }
        if (lane == 0) *item = r;
        __syncwarp();
    }
}

template <int K, int MODE, bool TB>
int launch_inst(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, cudaStream_t stream, const uint8_t* flags) {
    const int sa = (max_m + 15) & ~15, sb = (max_n + 15) & ~15;
    const int per_warp = sa + sb + (TB ? max_m * 128 : 0);
    int wpb = per_warp > 0 ? (96 * 1024) / per_warp : 8;
    if (wpb > 8) wpb = 8;
    if (wpb < 1) wpb = 1;
    const size_t smem = (size_t)per_warp * wpb;
    auto kern = psa_short_kernel<K, MODE, TB>;
    if (smem > (size_t)ctx->smem_optin) return psa_fail(ctx, PSA_ERR_RANGE, "short kernel: pair does not fit in shared memory");
    int rc = psa_kernel_optin_smem(ctx, (const void*)kern);
    if (rc) return rc;
    int per_sm = 0;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, wpb * 32, smem));
    if (per_sm < 1) return psa_fail(ctx, PSA_ERR_RANGE, "short kernel: pair does not fit in shared memory");
    int64_t want = (args.n_pairs + wpb - 1) / wpb;
    int64_t cap = (int64_t)per_sm * ctx->sm_count;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, wpb * 32, smem, stream>>>(args, sa, sb, per_warp, flags);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 1;
    return PSA_OK;
}

template <int K>
int launch_k(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool tb, cudaStream_t st,
             const uint8_t* flags) {
    if (mode == PSA_LOCAL) return tb ? launch_inst<K, PSA_LOCAL, true>(ctx, args, max_m, max_n, st, flags)
                                     : launch_inst<K, PSA_LOCAL, false>(ctx, args, max_m, max_n, st, flags);
    return tb ? launch_inst<K, PSA_GLOBAL, true>(ctx, args, max_m, max_n, st, flags)
              : launch_inst<K, PSA_GLOBAL, false>(ctx, args, max_m, max_n, st, flags);
}

}  // namespace

bool psa_short_supported(int max_m, int max_n, bool traceback) {
    if (max_n > 32 * kMaxK) return false;
    const size_t per_warp = (size_t)((max_m + 15) & ~15) + ((max_n + 15) & ~15) + (traceback ? (size_t)max_m * 128 : 0);
    return per_warp <= 200 * 1024;
}

int psa_launch_short(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                     cudaStream_t stream) {
    return psa_launch_short_flagged(ctx, args, max_m, max_n, mode, traceback, nullptr, stream);
}

int psa_launch_short_flagged(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                             const uint8_t* d_flags, cudaStream_t stream) {
    if (!psa_short_supported(max_m, max_n, traceback))
        return psa_fail(ctx, PSA_ERR_RANGE, "short kernel: n > 256 or pair too large for shared memory");
    if (max_m < 1) max_m = 1;
    if (max_n < 1) max_n = 1;
    const int K = (max_n + 31) / 32;
    switch (K) {
        case 1: return launch_k<1>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 2: return launch_k<2>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 3: return launch_k<3>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 4: return launch_k<4>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 5: return launch_k<5>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 6: return launch_k<6>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        case 7: return launch_k<7>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
        default: return launch_k<8>(ctx, args, max_m, max_n, mode, traceback, stream, d_flags);
    }
}
