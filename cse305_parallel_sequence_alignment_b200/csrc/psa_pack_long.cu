// psa_pack_long.cu -- packed (.S16x2) score-only kernel for batches of LONG DNA pairs
// (BASELINE config 5: 100k pairs of 5 kbp x 5 kbp, score + end coordinates).
//
// One warp per pair-of-pairs (two pairs share every register, as in psa_pack.cu).  The matrix is
// cut into column strips of W = 32*K columns (K = 16 from 1 kbp up: 3 999 vs 3 194 GCUPS on config 5,
// K = 8 below); the warp sweeps each strip top to bottom as a skewed
// wavefront (lane t owns K columns, (H-(g+h), E) of the column to the left arrive by shuffle) and
// parks the strip's right boundary column -- 8 bytes per row for both pairs -- in a per-warp
// scratch that stays in L2; lane 0 of the next strip reads it back through a coalesced 32-row
// block load + shuffle.  Same recurrence / borders as everywhere else (subproblem_alignment.cpp:
// 229-292); no O(mn) state, no traceback (the checkpointed single-pair path does that).
//
// Every max is the .RELU form, so padding cells (rows/columns past a member's own m, n) clamp at 0
// instead of decaying below it; real cells are >= 16 after every operation by the choice of the
// bias, so the clamp never touches them and plain 32-bit adds cannot borrow between the halves.
// Local mode finds the end cell with the packed key T1*8 + (7 - k%8) (VIMNMX3.U16x2), one running key per
// 8 columns, folded after every strip into a 64-bit (T1 desc, i asc, j asc) key.
#include "psa_result.cuh"

namespace {

constexpr int WPB = 4;          // K (columns per lane) is 8 or 16: strips of 256 or 512 columns

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ bool dna_code(int c, int& code) {
    code = (c >> 1) & 3;       // A=0 C=1 T=2 G=3
    return c == 'A' || c == 'C' || c == 'G' || c == 'T';
}

struct PLArgs {
    psa_batch_args P;
    int g, h, bias;
    uint32_t ng2, ngo2, go4;
    uint32_t mul8;             // = 8 at run time: keeps "t1*8 + c" an IMAD (FMA pipe) instead of an ALU-pipe LEA
    int max_m;
    uint2* tables;             // per resident warp: [max_m] row tables (tA, tB)
    uint2* bound;              // per resident warp: 2 x [max_m] boundary columns (hgo, e), ping-pong
    int* ticket;
    uint8_t* fallback;
};

// rowkey[half]: best key (T1*8 + 7 - k%8) of this row among the lane's columns 8*half .. 8*half+7; the key
// keeps 3 bits for the column so that scores up to ~8000 fit the 16-bit half whatever K is.
template <int K, bool LOCAL, bool CAP>
__device__ __forceinline__ void strip_step(uint32_t (&hgo)[K], uint32_t (&f)[K], const uint32_t (&sel)[K], uint32_t& hl,
                                           uint32_t& el, uint32_t diag, uint32_t tA, uint32_t tB, const PLArgs& A,
                                           uint32_t (&rowkey)[K / 8], int kcapA, int kcapB, uint32_t* cap) {
    uint32_t key_prev = 0;
    const uint32_t ng2 = A.ng2, ngo2 = A.ngo2, mul8 = A.mul8;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t s = prmt(tA, tB, sel[k]);
        const uint32_t t1 = diag + s;
        const uint32_t e = __viaddmax_s16x2_relu(el, ng2, hl);
        const uint32_t ff = __viaddmax_s16x2_relu(f[k], ng2, hgo[k]);
        const uint32_t H = __vimax3_s16x2_relu(t1, e, ff);
        if (LOCAL) {
            const uint32_t key = t1 * mul8 + (uint32_t)(7 - (k & 7)) * 0x00010001u;
            if (k & 1) rowkey[k / 8] = __vimax3_u16x2(rowkey[k / 8], key_prev, key);
            key_prev = key;
        }
        if (CAP) {
            if (k == kcapA) { cap[0] = t1; cap[1] = e; cap[2] = ff; }
            if (k == kcapB) { cap[3] = t1; cap[4] = e; cap[5] = ff; }
        }
        diag = hgo[k];
        const uint32_t hg = __viaddmax_s16x2_relu(H, ngo2, ngo2);     // max(H - (g+h), 0): third operand < 0 (no zero register)
        hgo[k] = hg; f[k] = ff; hl = hg; el = e;
    }
}

template <int MODE, int K>
__global__ void __launch_bounds__(WPB * 32) psa_pack_long_kernel(PLArgs A) {
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    constexpr int W = 32 * K;
    const int lane = threadIdx.x & 31;
    const long long gw = (long long)blockIdx.x * WPB + (threadIdx.x >> 5);
    const psa_batch_args& P = A.P;
    uint2* tab = A.tables + gw * A.max_m;
    uint2* bnd[2] = {A.bound + gw * 2 * A.max_m, A.bound + gw * 2 * A.max_m + A.max_m};
    const long long n_pp = (P.n_pairs + 1) / 2;
    const int go = A.g + A.h;

    for (;;) {
        long long pp = 0;
        if (lane == 0) pp = atomicAdd(A.ticket, 1);
        pp = __shfl_sync(0xffffffffu, pp, 0);
        if (pp >= n_pp) break;
        const long long pA = 2 * pp, pB = pA + 1;
        const bool haveB = pB < P.n_pairs;
        const int mA = P.len_a[pA], nA = P.len_b[pA];
        const int mB = haveB ? P.len_a[pB] : 0, nB = haveB ? P.len_b[pB] : 0;
        const int mpp = max(mA, mB), npp = max(nA, nB);
        const uint8_t* gaA = P.bases_a + P.off_a[pA];
        const uint8_t* gbA = P.bases_b + P.off_b[pA];
        const uint8_t* gaB = haveB ? P.bases_a + P.off_a[pB] : gaA;
        const uint8_t* gbB = haveB ? P.bases_b + P.off_b[pB] : gbA;
        bool okA = true, okB = true;
        // row tables for the whole pair-of-pairs
        for (int r = lane; r < mpp; r += 32) {
            uint32_t ta = A.go4, tb = A.go4;
            int code;
            if (r < mA) { okA &= dna_code(gaA[r], code); ta += 1u << (8 * code); }
            if (r < mB) { okB &= dna_code(gaB[r], code); tb += 1u << (8 * code); }
            tab[r] = make_uint2(ta, tb);
        }
        __syncwarp();
        // local: this lane's best of the CURRENT strip -- key (T1*8 + 7-k%8), row, half -- folded after every strip
        // into the running 64-bit (T1 desc, i asc, j asc) key: a later strip can hold an equal T1 at a smaller row
        uint32_t bestA = 0, bestB = 0;
        int biA = 0, biB = 0, bsA = 0, bsB = 0;
        unsigned long long runA = 0ull, runB = 0ull;
        auto full = [&](uint32_t best, int bi, int bs) -> unsigned long long {
            const int t1v = (int)(best >> 3) - A.bias;
            if (t1v <= 0) return 0ull;
            const int j = (bs >> 1) * W + lane * K + (bs & 1) * 8 + (7 - (int)(best & 7u)) + 1;
            return best_key(t1v, bi, j);
        };
        uint32_t cap[6] = {0, 0, 0, 0, 0, 0};
        const int S = (npp + W - 1) / W;
        const int tcA = (nA > 0) ? ((nA - 1) % W) / K : -1, kcA = (nA > 0) ? (nA - 1) % K : -1, scA = (nA > 0) ? (nA - 1) / W : -1;
        const int tcB = (nB > 0) ? ((nB - 1) % W) / K : -1, kcB = (nB > 0) ? (nB - 1) % K : -1, scB = (nB > 0) ? (nB - 1) / W : -1;

        for (int s = 0; s < S; ++s) {
            const uint2* bin = bnd[s & 1];
            uint2* bout = bnd[(s & 1) ^ 1];
            const int c0 = s * W + lane * K;          // 0-based first column of this lane
            uint32_t hgo[K], f[K], sel[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int j = c0 + k;
                int ca = 8, cb = 8, code;
                if (j < nA) { okA &= dna_code(gbA[j], code); ca = code; }
                if (j < nB) { okB &= dna_code(gbB[j], code); cb = 4 + code; }
                sel[k] = (uint32_t)ca | 0x80u | ((uint32_t)cb << 8) | 0x8000u;
                const int hb = LOCAL ? A.bias : A.bias - A.h - A.g * (j + 1);     // H[0][j+1]
                hgo[k] = (uint32_t)max(hb - go, 0) * 0x00010001u;
                f[k] = 0u;
            }
            uint32_t hd;
            {
                const int hb = (LOCAL || c0 == 0) ? A.bias : A.bias - A.h - A.g * c0;   // H[0][c0]
                hd = (uint32_t)max(hb - go, 0) * 0x00010001u;
            }
            uint32_t recv_h = 0, recv_e = 0;
            uint2 blk = make_uint2(0u, 0u);            // boundary rows of the current 32-row block (lane L: row base+L)
            const int steps = mpp + 31;
            for (int st = 0; st < steps; ++st) {
                const int r = st - lane;
                if (s > 0 && (st & 31) == 0) {         // lane 0 is at row st: load rows st..st+31 of the left boundary
                    const int rr = st + lane;
                    blk = (rr < mpp) ? __ldcg(bin + rr) : make_uint2(0u, 0u);
                }
                uint32_t hl, el;
                {
                    const uint32_t bh = __shfl_sync(0xffffffffu, blk.x, st & 31);
                    const uint32_t be = __shfl_sync(0xffffffffu, blk.y, st & 31);
                    if (lane == 0) {
                        if (s == 0) {                  // column 0: H[i][0] = T3[i][0] = -h - g*i (cpp:290-292), E = -inf
                            const int hb = LOCAL ? A.bias : A.bias - A.h - A.g * (r + 1);
                            hl = (uint32_t)max(hb - go, 0) * 0x00010001u; el = 0u;
                        } else { hl = bh; el = be; }
                    } else { hl = recv_h; el = recv_e; }
                }
                const bool active = (r >= 0 && r < mpp);
                bool capstep = false;
                if (!LOCAL) capstep = active && ((r == mA - 1 && s == scA && lane == tcA) || (r == mB - 1 && s == scB && lane == tcB));
                const bool anycap = LOCAL ? false : __any_sync(0xffffffffu, capstep);
                if (active) {
                    const uint2 tt = tab[r];
                    const uint32_t hl0 = hl;
                    uint32_t rowkey[K / 8];
#pragma unroll
                    for (int q = 0; q < K / 8; ++q) rowkey[q] = 0;
                    if (!anycap) strip_step<K, LOCAL, false>(hgo, f, sel, hl, el, hd, tt.x, tt.y, A, rowkey, -1, -1, cap);
                    else {
                        const int ka = (r == mA - 1 && s == scA && lane == tcA) ? kcA : -1;
                        const int kb = (r == mB - 1 && s == scB && lane == tcB) ? kcB : -1;
                        strip_step<K, LOCAL, true>(hgo, f, sel, hl, el, hd, tt.x, tt.y, A, rowkey, ka, kb, cap);
                    }
                    hd = hl0;
                    if (LOCAL) {
#pragma unroll
                        for (int q = 0; q < K / 8; ++q) {       // lower columns first: a tie keeps the smaller j
                            const uint32_t lo = rowkey[q] & 0xffffu, hi = rowkey[q] >> 16;
                            if (lo > (bestA | 7u)) { bestA = lo; biA = r + 1; bsA = s * 2 + q; }
                            if (hi > (bestB | 7u)) { bestB = hi; biB = r + 1; bsB = s * 2 + q; }
                        }
                    }
                    if (lane == 31 && s + 1 < S) bout[r] = make_uint2(hl, el);
                }
                recv_h = __shfl_up_sync(0xffffffffu, hl, 1);
                recv_e = __shfl_up_sync(0xffffffffu, el, 1);
            }
            if (LOCAL) {
                const unsigned long long ka = full(bestA, biA, bsA), kb = full(bestB, biB, bsB);
                runA = ka > runA ? ka : runA; runB = kb > runB ? kb : runB;
                bestA = 0; bestB = 0;
            }
            __syncwarp();
        }
        okA = __all_sync(0xffffffffu, okA);
        okB = __all_sync(0xffffffffu, okB);

        if (LOCAL) {
            // lexicographic (T1 desc, i asc, j asc) across lanes, 64-bit key
            unsigned long long fa = runA, fb = runB;
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                const unsigned long long oa = __shfl_xor_sync(0xffffffffu, fa, off), ob = __shfl_xor_sync(0xffffffffu, fb, off);
                fa = oa > fa ? oa : fa; fb = ob > fb ? ob : fb;
            }
            if (lane == 0) {
                if (mA > 0 && nA > 0) P.items[pA] = local_item_from_key(fa);
                if (haveB && mB > 0 && nB > 0) P.items[pB] = local_item_from_key(fb);
            }
        } else {
            if (mA > 0 && nA > 0 && lane == tcA) P.items[pA] = packed_corner_item(cap, 0, A.bias, mA, nA);
            if (haveB && mB > 0 && nB > 0 && lane == tcB) P.items[pB] = packed_corner_item(cap + 3, 16, A.bias, mB, nB);
        }
        if (lane == 0) {
            A.fallback[pA] = (!okA || mA == 0 || nA == 0) ? 1 : 0;
            if (haveB) A.fallback[pB] = (!okB || mB == 0 || nB == 0) ? 1 : 0;
        }
        __syncwarp();
    }
}

}  // namespace

bool psa_pack_long_supported(int max_m, int max_n, int mode, int g, int h) {
    if (max_m < 1 || max_n < 1 || g + h + 1 > 120) return false;
    if (mode == PSA_LOCAL && g + h < 1) return false;   // padding cells can only tie the best when g+h == 0
    const long long mn = std::min(max_m, max_n);
    if (mode == PSA_LOCAL) return ((long long)(g + h + 16) + mn) * 8 + 7 < 65536;
    const long long bias = (long long)g * (max_m + max_n) + 2 * h + (g + h) + 16;
    return bias + mn + g + h + 2 < 32700;
}

int psa_launch_pack_long(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st) {
    const int g = args.g, h = args.h;
    PLArgs A;
    A.P = args; A.g = g; A.h = h; A.max_m = max_m;
    A.bias = (mode == PSA_LOCAL) ? (g + h + 16) : (g * (max_m + max_n) + 2 * h + (g + h) + 16);
    A.ng2 = (uint32_t)((-g) & 0xffff) * 0x00010001u;
    A.ngo2 = (uint32_t)((-(g + h)) & 0xffff) * 0x00010001u;
    A.go4 = (uint32_t)(g + h) * 0x01010101u;
    A.mul8 = 8u;
    // 16 columns per lane halve the per-step overhead (shuffles, row table, boundary hand-over) per cell;
    // below ~1 kbp the wider strips only add padding
    int wide = max_n >= 1024 ? 1 : 0;
    if (ctx->opt.pack_long_k) wide = ctx->opt.pack_long_k == 16 ? 1 : 0;
    const void* kern = mode == PSA_LOCAL ? (wide ? (const void*)psa_pack_long_kernel<PSA_LOCAL, 16> : (const void*)psa_pack_long_kernel<PSA_LOCAL, 8>)
                                         : (wide ? (const void*)psa_pack_long_kernel<PSA_GLOBAL, 16> : (const void*)psa_pack_long_kernel<PSA_GLOBAL, 8>);
    int per_sm = 0;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WPB * 32, 0));
    if (per_sm > 4) per_sm = 4;
    const long long n_pp = (args.n_pairs + 1) / 2;
    int grid = (int)std::min<long long>((n_pp + WPB - 1) / WPB, (long long)per_sm * ctx->sm_count);
    if (grid < 1) grid = 1;
    const size_t warps = (size_t)grid * WPB;
    const size_t o_flags = 0, o_tab = ((size_t)args.n_pairs + 255) / 256 * 256;
    const size_t o_bnd = o_tab + warps * max_m * sizeof(uint2);
    const size_t o_tick = o_bnd + warps * 2 * max_m * sizeof(uint2);
    const size_t o_fb_scratch = o_tick + 256;          // scratch of the int32 fallback kernel, behind ours
    const size_t total = o_fb_scratch + psa_long_batch_scratch_bytes(ctx, args.n_pairs, max_n);
    if (total > ctx->d_work_bytes) {
        if (ctx->d_work) cudaFree(ctx->d_work);
        ctx->d_work = nullptr; ctx->d_work_bytes = 0;
        if (cudaMalloc(&ctx->d_work, total) != cudaSuccess) { cudaGetLastError(); return psa_fail(ctx, PSA_ERR_NOMEM, "packed long kernel scratch"); }
        ctx->d_work_bytes = total;
    }
    uint8_t* d = (uint8_t*)ctx->d_work;
    PSA_CUDA_OK(ctx, cudaMemsetAsync(d + o_tick, 0, 256, st));
    A.fallback = d + o_flags; A.tables = (uint2*)(d + o_tab); A.bound = (uint2*)(d + o_bnd); A.ticket = (int*)(d + o_tick);
    void* kargs[] = {&A};
    PSA_CUDA_OK(ctx, cudaLaunchKernel(kern, dim3(grid), dim3(WPB * 32), kargs, 0, st));
    ctx->launches += 1;
    // non-ACGT / empty members: the int32 long-batch kernel, flagged pairs only (own scratch after ours)
    return psa_launch_long_batch_at(ctx, args, max_m, max_n, mode, d + o_flags, d + o_fb_scratch, st);
}
