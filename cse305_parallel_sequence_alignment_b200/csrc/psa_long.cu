// psa_long.cu -- intra-pair wavefront kernels for long pairs (BASELINE configs 3, 4, 5).
//
// The DP matrix is cut into row blocks of R rows and column strips of W = 32*K columns.  One warp
// owns a row block and sweeps its tiles left to right (psa_tile::sweep); the bottom boundary of
// every tile (H and F per column) goes to a global "hbuf", the right boundary stays in the warp's
// shared memory for the next tile.  Row block rb may start strip s once row block rb-1 has
// finished strip s: a per-row-block progress counter published with release/acquire semantics.
// Row blocks are handed out by an atomic ticket in increasing order, so every dependency points at
// a warp that already holds an earlier ticket -- forward progress never depends on co-residency.
// This replaces the reference's Subproblem::compute_tables (subproblem_alignment.cpp:329-355):
// per-row fork/join + ParallelPrefixMax become a two-level wavefront (lanes inside a tile, warps
// across tiles), and the three O(mn) double tables (subproblem_alignment.h:66-73) become O(m+n)
// boundaries.
//
// Traceback (config 3) never needs the full matrix: with checkpoints enabled the fill keeps every
// row-block bottom row and every strip right column (8*m*n*(1/R + 1/W) bytes); the traceback
// kernel then recomputes only the tiles the path crosses, with 4-bit codes in shared memory -- the
// role the reference intended for its partial-balanced-partition stage (sequence_alignment/
// partial.cpp:81-163, never wired up).
#include <climits>
#include <vector>

#include "psa_tile.cuh"

using namespace psa_tile;

namespace {

constexpr int K = 8;
constexpr int W = 32 * K;      // strip width
constexpr int R = 128;         // row-block height
constexpr int WPB = 4;         // warps per CTA

struct LongJob {
    const uint8_t* a;
    const uint8_t* b;
    int m, n;
    int g, h;
    int mul8;                   // = 8 at run time (keeps the local-mode key an IMAD)
    int* hbufH;                 // bottom boundaries; row-block stride hb_stride ints (0 = one recycled row)
    int* hbufF;
    long long hb_stride;
    int* ckvH;                  // right-boundary checkpoint columns [S][m+1] (null without checkpoints)
    int* ckvE;
    int* progress;              // [NB] strips finished per row block (null in batch mode: no waiting)
    int* ticket;
    unsigned long long* best;   // local: packed (score, end_i, end_j) key, atomicMax
    int* corner;                // global: T1,T2,T3 of (m,n)
    int col0, n_total;          // always 0 / n (kept so that the tile engine can address a column window)
    int start_type, end_type;   // Subproblem border variants (global mode); -1 / -1 = the live case
    int row_off;                // ROWOFF instantiation only: height of the FIRST row block (partition sweeps); else 0
};

// Polling load: relaxed at gpu scope (served by L2, no L1 invalidate).  ld.acquire would emit a
// CCTL.IVALL per poll, and a few spinning warps then starve the shared-memory pipe of the working
// warps on the same SM (measured: 1.35e9 invalidates, 4x slower tiles).  One fence follows the
// successful poll instead.
__device__ __forceinline__ int ld_relaxed(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <int RR>
struct WarpSmem {
    int bH[2][RR];     // ping-pong boundary columns: [cur] = left boundary in, [cur^1] = right out
    int bE[2][RR];
    uint8_t sA[RR];
};

// One row block: rows rb*R+1 .. , all strips.  Warp-collective.
// RR rows per block, KK columns per lane (strip width 32*KK); checkpoints and the traceback grid need <128, 8>.
template <int MODE, int RR, int KK, bool ROWOFF = false>
__device__ void process_rowblock(const LongJob& J, int rb, WarpSmem<RR>& sm, Track& tr) {
    constexpr int WW = 32 * KK;
    const int lane = threadIdx.x & 31;
    const int m = J.m, n = J.n, g = J.g, h = J.h;
    // ROWOFF (partition sweeps only): the first row block is J.row_off rows high, the grid is shifted accordingly
    const int i0 = (!ROWOFF || rb == 0) ? rb * RR : J.row_off + (rb - 1) * RR;
    const int nrows = (ROWOFF && rb == 0) ? min(J.row_off, m) : min(RR, m - i0);
    const int S = (n + WW - 1) / WW;
    for (int r = lane; r < nrows; r += 32) sm.sA[r] = J.a[i0 + r];
    // left boundary of strip 0: column 0 of the matrix (subproblem_alignment.cpp:282-292)
    for (int r = lane; r < nrows; r += 32) { sm.bH[0][r] = border_col0_H<MODE>(i0 + 1 + r, g, h, J.start_type); sm.bE[0][r] = PSA_KNEG; }
    int corner = border_col0_H<MODE>(i0, g, h, J.start_type);           // H[i0][0]
    __syncwarp();
    int cur = 0;
    const int* topH = J.hbufH + (J.hb_stride ? (long long)(rb - 1) * J.hb_stride : 0);
    const int* topF = J.hbufF + (J.hb_stride ? (long long)(rb - 1) * J.hb_stride : 0);
    int* botH = J.hbufH + (J.hb_stride ? (long long)rb * J.hb_stride : 0);
    int* botF = J.hbufF + (J.hb_stride ? (long long)rb * J.hb_stride : 0);
    int cap1 = PSA_KNEG, cap2 = PSA_KNEG, cap3 = PSA_KNEG;
    bool captured = false;
    for (int s = 0; s < S; ++s) {
        if (rb > 0 && J.progress != nullptr) {
            // Every lane polls the same word (one broadcast request): a lane-0-only spin loop left
            // the warp split into two convergence groups for the rest of the row block -- each
            // step then ran twice and the shuffles took the slow collective path (3.3x slower).
            unsigned ns = 32;
            while (ld_relaxed(J.progress + rb - 1) <= s) { __nanosleep(ns); if (ns < 2048) ns <<= 1; }
            __threadfence();              // acquire side: order the boundary reads after the flag read
            __syncwarp();
        }
        const int c0 = s * WW + lane * KK;
        ColsS<KK> cs;
#pragma unroll
        for (int k = 0; k < KK; ++k) {
            const int j = c0 + k + 1;
            cs.b[k] = (j <= n) ? (int)J.b[j - 1] : 256;
            int H0, F0 = PSA_KNEG;
            if (rb == 0) H0 = border_row0_H<MODE>(J.col0 + j, g, h, J.start_type);
            else if (j <= n) { H0 = __ldcg(topH + j); F0 = __ldcg(topF + j); }
            else H0 = (MODE == PSA_LOCAL) ? 0 : PSA_KNEG;
            cs.set_top(k, H0, F0, g + h);
            cs.set_key_addend(k, j <= n, g + h);
        }
        // H[i0][c0] for every lane: the top value of the previous lane's last column; lane 0: the corner
        const int hlast = cs.top_H(KK - 1, g + h);
        int hd = __shfl_up_sync(0xffffffffu, hlast, 1);
        if (lane == 0) hd = corner;
        const int next_corner = __shfl_sync(0xffffffffu, hlast, 31);   // H[i0][(s+1)*WW]
        const bool has_cell = (J.col0 + n == J.n_total) && (i0 + nrows == m) && (n > s * WW) && (n <= (s + 1) * WW);
        int bestkey = 0, besti = 0;
        sweep_score<KK, MODE>(cs, hd, sm.bH[cur], sm.bE[cur], sm.bH[cur ^ 1], sm.bE[cur ^ 1], sm.sA, nrows, i0, c0, m, n, g, h,
                             J.mul8, bestkey, besti, cap1, cap2, cap3);
        if (MODE == PSA_LOCAL) {          // fold this tile's best (T1, first row, first column) into the lane's tracker
            const int t1v = bestkey / key_mult(KK);
            const int bj = c0 + (key_mult(KK) - 1 - (bestkey % key_mult(KK))) + 1;
            if (t1v > 0 && bj <= n) {
                const bool better = t1v > tr.best || (t1v == tr.best && (besti < tr.bi || (besti == tr.bi && bj < tr.bj)));
                if (better) { tr.best = t1v; tr.bi = besti; tr.bj = bj; }     // bj is strip-local; col0 is added when packed
            }
        }
        if (has_cell) captured = true;
        // publish the bottom boundary
#pragma unroll
        for (int k = 0; k < KK; ++k) {
            const int j = c0 + k + 1;
            if (j <= n) { botH[j] = cs.top_H(k, g + h); botF[j] = cs.ff[k]; }
        }
        __syncwarp();
        if (J.ckvH != nullptr) {          // checkpoint the right boundary column (col (s+1)*WW)
            int* vh = J.ckvH + (long long)s * (m + 1);
            int* ve = J.ckvE + (long long)s * (m + 1);
            for (int r = lane; r < nrows; r += 32) { vh[i0 + 1 + r] = sm.bH[cur ^ 1][r]; ve[i0 + 1 + r] = sm.bE[cur ^ 1][r]; }
        }
        if (J.progress != nullptr) {
            __threadfence();
            __syncwarp();
            if (lane == 0) st_release(J.progress + rb, s + 1);
        }
        corner = next_corner;
        cur ^= 1;
        __syncwarp();
    }
    if (MODE == PSA_GLOBAL && captured) {
        // exactly one lane of one tile holds cell (m, n)
        const int src = ((n - 1) % WW) / KK;
        if (lane == src) { J.corner[0] = cap1; J.corner[1] = cap2; J.corner[2] = cap3; }
    }
}

template <int MODE>
__device__ void flush_track(const LongJob& J, Track& tr) {
    if (MODE != PSA_LOCAL) return;
    unsigned long long key = tr.best > 0 ? best_key(tr.best, tr.bi, J.col0 + tr.bj) : 0ull;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, key, off);
        key = o > key ? o : key;
    }
    if ((threadIdx.x & 31) == 0 && key != 0ull) atomicMax(J.best, key);
}

// Single long pair: every warp of the grid pulls row blocks of the same job.
template <int MODE, int RR, int KK, bool ROWOFF = false>
__global__ void __launch_bounds__(WPB * 32) psa_long_single_kernel(LongJob J) {
    __shared__ WarpSmem<RR> smem[WPB];
    WarpSmem<RR>& sm = smem[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int NB = ROWOFF ? 1 + max(0, J.m - J.row_off + RR - 1) / RR : (J.m + RR - 1) / RR;
    Track tr{0, 0, 0};
    for (;;) {
        int rb = 0;
        if (lane == 0) rb = atomicAdd(J.ticket, 1);
        rb = __shfl_sync(0xffffffffu, rb, 0);
        if (rb >= NB) break;
        process_rowblock<MODE, RR, KK, ROWOFF>(J, rb, sm, tr);
    }
    flush_track<MODE>(J, tr);
}

// Batch of long pairs, score only: one warp per pair (pairs are independent -- no flags).
struct LongBatch {
    psa_batch_args P;
    int* hbuf;                 // per resident warp: 2*(max_n+1) ints
    long long hbuf_warp_stride;
    int* ticket;
    const uint8_t* only_flagged;   // optional: one byte per pair, process only non-zero entries
    int mul8;
};

template <int MODE, int KK>      // KK columns per lane: 16 from 1 kbp (pairs are independent, wide lanes only amortise overhead), else 8
__global__ void __launch_bounds__(WPB * 32) psa_long_batch_kernel(LongBatch Bt) {
    __shared__ WarpSmem<R> smem[WPB];
    __shared__ unsigned long long s_best[WPB];
    __shared__ int s_corner[WPB][4];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpSmem<R>& sm = smem[w];
    const long long gw = (long long)blockIdx.x * WPB + w;
    for (;;) {
        long long p = 0;
        if (lane == 0) p = atomicAdd(Bt.ticket, 1);
        p = __shfl_sync(0xffffffffu, p, 0);
        if (p >= Bt.P.n_pairs) break;
        if (Bt.only_flagged != nullptr && Bt.only_flagged[p] == 0) continue;
        LongJob J;
        J.a = Bt.P.bases_a + Bt.P.off_a[p]; J.b = Bt.P.bases_b + Bt.P.off_b[p];
        J.m = Bt.P.len_a[p]; J.n = Bt.P.len_b[p]; J.g = Bt.P.g; J.h = Bt.P.h; J.mul8 = Bt.mul8;
        J.hbufH = Bt.hbuf + gw * Bt.hbuf_warp_stride; J.hbufF = J.hbufH + Bt.hbuf_warp_stride / 2; J.hb_stride = 0;
        J.ckvH = nullptr; J.ckvE = nullptr; J.progress = nullptr; J.ticket = nullptr;
        J.best = &s_best[w]; J.corner = s_corner[w];
        J.col0 = 0; J.n_total = J.n; J.row_off = 0;
        J.start_type = -1; J.end_type = -1;
        if (lane == 0) { s_best[w] = 0ull; s_corner[w][0] = s_corner[w][1] = s_corner[w][2] = PSA_KNEG; }
        __syncwarp();
        if (J.m > 0 && J.n > 0) {
            Track tr{0, 0, 0};
            const int NB = (J.m + R - 1) / R;
            for (int rb = 0; rb < NB; ++rb) process_rowblock<MODE, R, KK>(J, rb, sm, tr);
            flush_track<MODE>(J, tr);
            __syncwarp();
        }
        if (lane == 0) {
            psa_batch_item r;
            if (J.m <= 0 || J.n <= 0) r = empty_item<MODE>(J.m, J.n, J.g, J.h, -1, -1);
            else if (MODE == PSA_LOCAL) r = local_item_from_key(s_best[w]);
            else r = global_item(s_corner[w][0], s_corner[w][1], s_corner[w][2], J.m, J.n, J.h, -1);
            Bt.P.items[p] = r;
        }
        __syncwarp();
    }
}

// ---- checkpointed traceback: one warp recomputes only the tiles the path crosses ----------
struct TbArgs {
    LongJob J;
    psa_batch_item* item;      // device result
    uint32_t* ops;             // 2-bit ops, traceback order
    uint32_t* band;            // optional: direction codes of BAND_TILES tiles per row block, recomputed in parallel
};

constexpr int BAND_TILES = 3;

// Result record the traceback starts from: end cell and end state (find_alignment, subproblem_alignment.cpp:112-145).
template <int MODE>
__device__ __forceinline__ psa_batch_item tb_end(const LongJob& J) {
    if (MODE == PSA_LOCAL) return local_item_from_key(*J.best);
    return global_item(J.corner[0], J.corner[1], J.corner[2], J.m, J.n_total, J.h, J.end_type);
}

// First strip of the band in row block rb: the tiles around the straight line the path is expected to
// follow -- the corner-to-corner diagonal for a global alignment, the slope-1 diagonal through the end
// cell for a local one.  A path that leaves the band only costs the on-demand recompute it always had.
template <int MODE>
__device__ __forceinline__ int band_first_strip(const LongJob& J, int end_i, int end_j, int rb) {
    const int S = (J.n + W - 1) / W;
    const long long mid_i = (long long)rb * R + R / 2;
    long long cj = (MODE == PSA_LOCAL) ? (long long)end_j - ((long long)end_i - mid_i)
                                       : (long long)J.n * mid_i / (J.m > 0 ? J.m : 1);
    cj = cj < 0 ? 0 : (cj > J.n - 1 ? J.n - 1 : cj);
    int first = (int)(cj / W) - 1;
    if (first > S - BAND_TILES) first = S - BAND_TILES;
    return first < 0 ? 0 : first;
}

// Direction codes of rows i0+1 .. i0+nrows of tile (rb, s), recomputed from the checkpointed boundaries
// (row-block bottom rows in hbuf, strip right columns in ckv) into `dirs` (32 words per row).
template <int MODE>
__device__ __forceinline__ void recompute_tile(const LongJob& J, int rb, int s, int nrows, uint32_t* dirs, int* lbH, int* lbE,
                                               uint8_t* sA) {
    const int lane = threadIdx.x & 31;
    const int m = J.m, n = J.n, g = J.g, h = J.h;
    const int i0 = rb * R, c0 = s * W + lane * K;
    __syncwarp();
    for (int q = lane; q < nrows; q += 32) {
        sA[q] = J.a[i0 + q];
        if (s == 0) { lbH[q] = border_col0_H<MODE>(i0 + 1 + q, g, h, J.start_type); lbE[q] = PSA_KNEG; }
        else { lbH[q] = J.ckvH[(long long)(s - 1) * (m + 1) + i0 + 1 + q]; lbE[q] = J.ckvE[(long long)(s - 1) * (m + 1) + i0 + 1 + q]; }
    }
    Cols<K> cs;
    const int* topH = J.hbufH + (long long)(rb - 1) * J.hb_stride;
    const int* topF = J.hbufF + (long long)(rb - 1) * J.hb_stride;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int jj = c0 + k + 1;
        cs.b[k] = (jj <= n) ? (int)J.b[jj - 1] : 256;
        if (rb == 0) { cs.H[k] = border_row0_H<MODE>(jj, g, h, J.start_type); cs.F[k] = PSA_KNEG; }
        else if (jj <= n) { cs.H[k] = topH[jj]; cs.F[k] = topF[jj]; }
        else { cs.H[k] = PSA_KNEG; cs.F[k] = PSA_KNEG; }
    }
    int hd = __shfl_up_sync(0xffffffffu, cs.H[K - 1], 1);
    if (lane == 0) hd = (s == 0) ? border_col0_H<MODE>(i0, g, h, J.start_type) : (rb == 0 ? border_row0_H<MODE>(s * W, g, h, J.start_type) : topH[s * W]);
    __syncwarp();
    Track tr{0, 0, 0};
    int d1 = 0, d2 = 0, d3 = 0;
    sweep<K, MODE, true>(cs, hd, lbH, lbE, nullptr, nullptr, sA, nrows, i0, c0, m, n, g, h, dirs, tr, d1, d2, d3);
    __syncwarp();
}

// Every tile is a function of its checkpointed boundaries alone, so the tiles the path will most likely
// cross are recomputed by independent warps all over the GPU before the (inherently serial) walk starts;
// the walker then only copies 16 KB per tile into its shared memory instead of sweeping it.
constexpr int BAND_WPB = 2;
template <int MODE>
__global__ void __launch_bounds__(BAND_WPB * 32) psa_long_band_kernel(TbArgs T) {
    __shared__ uint32_t dirs[BAND_WPB][R * 32];
    __shared__ int lbH[BAND_WPB][R], lbE[BAND_WPB][R];
    __shared__ uint8_t sA[BAND_WPB][R];
    const LongJob& J = T.J;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NB = (J.m + R - 1) / R, S = (J.n + W - 1) / W;
    const int u = blockIdx.x * BAND_WPB + w;
    if (u >= NB * BAND_TILES) return;
    const int rb = u / BAND_TILES, bt = u % BAND_TILES;
    const psa_batch_item r = tb_end<MODE>(J);
    if (rb * R >= r.end_i) return;                       // rows below the end cell are never visited
    const int s = band_first_strip<MODE>(J, r.end_i, r.end_j, rb) + bt;
    if (s >= S) return;
    const int nrows = min(R, J.m - rb * R);
    recompute_tile<MODE>(J, rb, s, nrows, dirs[w], lbH[w], lbE[w], sA[w]);
    uint4* out = reinterpret_cast<uint4*>(T.band + (long long)u * (R * 32));
    const uint4* in = reinterpret_cast<const uint4*>(dirs[w]);
    for (int q = lane; q < nrows * 8; q += 32) out[q] = in[q];
}

// The walk from the end cell and end state of `r`, lane 0 stepping through the codes of the tile held in `dirs` and the
// whole warp recomputing the next tile whenever the path leaves it.  Writes the 2-bit ops to `ops` and completes `r`
// (start cell, aln_len); `band` (optional) holds tiles psa_long_band_kernel recomputed ahead of time.
// Shared by the single-pair kernel and the batched walk (one warp per pair).
template <int MODE>
__device__ void tb_walk(const LongJob& J, psa_batch_item& r, uint32_t* ops, const uint32_t* band, uint32_t* dirs, int* lbH,
                        int* lbE, uint8_t* sA) {
    const int lane = threadIdx.x & 31;
    const int m = J.m;
    int i = r.end_i, j = r.end_j, state = r.end_state;
    int trb = -1, ts = -1;      // tile currently held in `dirs`
    int len = 0;
    int hits = 0, misses = 0;
    uint32_t acc = 0;
    bool done = !(i > 0 && j > 0);
    while (!done) {
        // lane 0 walks as far as the loaded tile allows
        int need_rb = -1, need_s = -1;
        if (lane == 0) {
            while (i > 0 && j > 0) {
                const int si = (state == 2) ? i : i - 1;
                const int sj = (state == 3) ? j : j - 1;
                const bool border = (si == 0 || sj == 0);
                int code = 0;
                if (!border) {
                    const int rb = (si - 1) / R, s = (sj - 1) / W;
                    if (rb != trb || s != ts) { need_rb = rb; need_s = s; break; }
                    const int cj = sj - 1 - s * W;
                    code = (dirs[(si - 1 - rb * R) * 32 + cj / K] >> (4 * (cj % K))) & 15;
                }
                acc |= (uint32_t)state << (2 * (len & 15));
                if ((len & 15) == 15) { ops[len >> 4] = acc; acc = 0; }
                ++len;
                r.start_i = i; r.start_j = j;
                const int ns = next_state<MODE>(state, code, border);
                if (ns == 0) { i = 0; break; }     // local alignment starts here
                state = ns; i = si; j = sj;
            }
        }
        need_rb = __shfl_sync(0xffffffffu, need_rb, 0);
        need_s = __shfl_sync(0xffffffffu, need_s, 0);
        if (need_rb < 0) { done = true; break; }
        const int rb = need_rb, s = need_s;
        const int need_row = __shfl_sync(0xffffffffu, (lane == 0) ? ((state == 2) ? i : i - 1) : 0, 0);   // source row of the pending step
        const int i0 = rb * R, nrows = min(min(R, m - i0), need_row - i0);      // rows below the entry row are never consulted
        const int bt = (band != nullptr) ? s - band_first_strip<MODE>(J, r.end_i, r.end_j, rb) : -1;
        if (bt >= 0 && bt < BAND_TILES) {
            // ---- the tile was recomputed ahead of time by psa_long_band_kernel: copy its codes in ----
            __syncwarp();
            const uint4* in = reinterpret_cast<const uint4*>(band + ((long long)rb * BAND_TILES + bt) * (R * 32));
            uint4* out = reinterpret_cast<uint4*>(dirs);
            const int total = nrows * 8;                       // 16-byte pieces; eight loads in flight per lane
            for (int q0 = 0; q0 < total; q0 += 256) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int q = q0 + u * 32 + lane; if (q < total) v[u] = __ldcg(in + q); }
#pragma unroll
                for (int u = 0; u < 8; ++u) { const int q = q0 + u * 32 + lane; if (q < total) out[q] = v[u]; }
            }
            __syncwarp();
            if (lane == 0) ++hits;
        } else {
            // ---- recompute tile (rb, s) from its checkpointed boundaries ----
            recompute_tile<MODE>(J, rb, s, nrows, dirs, lbH, lbE, sA);
            if (lane == 0) ++misses;
        }
        trb = rb; ts = s;
    }
#ifdef PSA_TB_DEBUG
    if (lane == 0) printf("tb_walk: %d band tiles, %d recomputed tiles, %d ops\n", hits, misses, len);
#endif
    if (lane == 0) {
        if (len & 15) ops[len >> 4] = acc;
        r.aln_len = len;
    }
}

template <int MODE>
__global__ void __launch_bounds__(32) psa_long_tb_kernel(TbArgs T) {
    __shared__ uint32_t dirs[R * 32];
    __shared__ int lbH[R], lbE[R];
    __shared__ uint8_t sA[R];
    psa_batch_item r = tb_end<MODE>(T.J);
    if (T.ops != nullptr) tb_walk<MODE>(T.J, r, T.ops, T.band, dirs, lbH, lbE, sA);
    if (threadIdx.x == 0) *T.item = r;
}

// ---- batch of long pairs with traceback: checkpointed fill (one warp per pair), then one walk warp per pair ----
// Pair p of the chunk [p0, p0 + count) owns slot p - p0 of the region: [best (8 B) | corner (3 x 4 B) | pad to 256 B |
// row-block bottom rows H, F (NB rows of up256((n+1)*4) bytes each) | strip right columns H, E ([S][m+1] ints each)],
// sized by the pair's own m, n inside slot_bytes (computed from the largest m, n of the batch).
struct LongBatchTb {
    psa_batch_args P;
    long long p0, count;
    uint8_t* region;
    long long slot_bytes;
    int* ticket;
};

__device__ __forceinline__ long long up256_d(long long x) { return (x + 255) / 256 * 256; }

// The LongJob of pair p (its checkpoints in the slot); the same for the fill and the walk.
__device__ __forceinline__ LongJob batch_tb_job(const LongBatchTb& Bt, long long p) {
    const psa_batch_args& P = Bt.P;
    LongJob J;
    J.a = P.bases_a + P.off_a[p]; J.b = P.bases_b + P.off_b[p];
    J.m = P.len_a[p]; J.n = P.len_b[p]; J.g = P.g; J.h = P.h; J.mul8 = key_mult(K);
    uint8_t* slot = Bt.region + (p - Bt.p0) * Bt.slot_bytes;
    const int NB = (J.m + R - 1) / R, S = (J.n + W - 1) / W;
    const long long row = up256_d((long long)(J.n + 1) * 4), ckv = up256_d((long long)S * (J.m + 1) * 4);
    J.best = (unsigned long long*)slot; J.corner = (int*)(slot + 8);
    J.hbufH = (int*)(slot + 256); J.hbufF = (int*)(slot + 256 + row * NB); J.hb_stride = row / 4;
    J.ckvH = (int*)(slot + 256 + 2 * row * NB); J.ckvE = (int*)(slot + 256 + 2 * row * NB + ckv);
    J.progress = nullptr; J.ticket = nullptr;
    J.col0 = 0; J.n_total = J.n; J.row_off = 0;
    J.start_type = P.types ? (int)(P.types[p] & 15) - 3 : P.start_type;
    J.end_type = P.types ? (int)(P.types[p] >> 4) - 3 : P.end_type;
    return J;
}

// Fill: the <128, 8> tile grid the walk decodes (pairs are independent: no progress flags).
template <int MODE>
__global__ void __launch_bounds__(WPB * 32) psa_long_batch_tb_fill_kernel(LongBatchTb Bt) {
    __shared__ WarpSmem<R> smem[WPB];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpSmem<R>& sm = smem[w];
    for (;;) {
        long long q = 0;
        if (lane == 0) q = atomicAdd(Bt.ticket, 1);
        q = __shfl_sync(0xffffffffu, q, 0);
        if (q >= Bt.count) break;
        const long long p = Bt.p0 + q;
        const LongJob J = batch_tb_job(Bt, p);
        if (J.m <= 0 || J.n <= 0) continue;          // borders only: the walk kernel writes the item
        if (lane == 0) { *J.best = 0ull; J.corner[0] = J.corner[1] = J.corner[2] = PSA_KNEG; }
        __syncwarp();
        Track tr{0, 0, 0};
        const int NB = (J.m + R - 1) / R;
        for (int rb = 0; rb < NB; ++rb) process_rowblock<MODE, R, K>(J, rb, sm, tr);
        flush_track<MODE>(J, tr);
        __syncwarp();
    }
}

// Walk: one warp per pair of the chunk, the single-pair walk without the band (the other pairs are the parallelism).
constexpr int WALK_WPB = 2;      // 2 x 17.3 KB of static shared memory per CTA
template <int MODE>
__global__ void __launch_bounds__(WALK_WPB * 32) psa_long_batch_tb_walk_kernel(LongBatchTb Bt) {
    __shared__ uint32_t dirs[WALK_WPB][R * 32];
    __shared__ int lbH[WALK_WPB][R], lbE[WALK_WPB][R];
    __shared__ uint8_t sA[WALK_WPB][R];
    const int w = threadIdx.x >> 5;
    const long long q = (long long)blockIdx.x * WALK_WPB + w;
    if (q >= Bt.count) return;
    const long long p = Bt.p0 + q;
    const LongJob J = batch_tb_job(Bt, p);
    psa_batch_item r;
    if (J.m <= 0 || J.n <= 0) {
        r = empty_item<MODE>(J.m, J.n, J.g, J.h, J.start_type, J.end_type);
    } else {
        r = tb_end<MODE>(J);
        tb_walk<MODE>(J, r, Bt.P.ops + p * Bt.P.ops_stride_words, nullptr, dirs[w], lbH[w], lbE[w], sA[w]);
    }
    if ((threadIdx.x & 31) == 0) Bt.P.items[p] = r;
}

// ---- banded batches (psa_align_batch_banded) -----------------------------------------------------------------------
// Cell (i, j) is in the band iff |j - c(i)| <= bw, c(i) = floor(i*n/m): the line from (0,0) to (m,n).  Outside the band
// H = T1 = 0 in local mode (the value of the local borders, DESIGN.md section 3), the sentinel in global mode; E = F =
// sentinel in both.  Row block rb sweeps only strips s_lo(rb) .. s_hi(rb), the strips its band rows touch (both
// non-decreasing in rb); everything it reads from outside that range -- the top of strips rb - 1 did not compute, the
// left column of strip s_lo > 0, border cells beyond the band -- is out of band.  Tiles that a band edge cuts take the
// masked sweeps (sweep_score / sweep with BANDED), tiles wholly inside the band the plain ones.
struct Band {
    int m, n, bw;
    __device__ __forceinline__ int c(int i) const { return (int)((long long)i * n / m); }
    __device__ __forceinline__ int lo(int i) const { return max(0, c(i) - bw); }
    __device__ __forceinline__ int hi(int i) const { return (int)min((long long)n, (long long)c(i) + bw); }
    // strips of width WW touched by rows i0+1 .. i0+nrows
    __device__ __forceinline__ int s_lo(int i0, int WW) const { return (max(1, lo(i0 + 1)) - 1) / WW; }
    __device__ __forceinline__ int s_hi(int i0, int nrows, int WW) const { return max(s_lo(i0, WW), (max(1, hi(i0 + nrows)) - 1) / WW); }
    // every cell of rows i0+1 .. i0+nrows, columns s*WW+1 .. min(n, (s+1)*WW) is in the band
    __device__ __forceinline__ bool inside(int i0, int nrows, int s, int WW) const {
        return lo(i0 + nrows) <= s * WW + 1 && hi(i0 + 1) >= min(n, (s + 1) * WW);
    }
};

// The band around a caller's anchor chain (psa_align_batch_guided, psa_align_pair_guided; include/psa.h).  The guide is
// the polyline P_0 = (0, 0), P_1 .. P_K (the anchors), P_{K+1} = (m, n).  Row i's guide columns [cmin(i), cmax(i)] are
// the j of the first and of the last chain point on row i, else the point at floor of the segment P_k -> P_{k+1} that
// crosses row i; lo(i) = max(0, cmin(i) - bw), hi(i) = min(n, cmax(i) + bw).  A valid chain (coordinates in range and
// non-decreasing) gives cmin(i + 1) >= cmax(i), so lo and hi are non-decreasing and s_lo / s_hi / inside keep Band's
// formulas.  Each row costs a binary search over the chain; nothing is evaluated per cell.  K = 0 gives Band's rows.
struct ChainBand {
    int m, n, bw;
    const psa_anchor* anc;     // the pair's K anchors, a valid chain
    int K;
    __host__ __device__ __forceinline__ int2 pt(int k) const {          // P_k, k = 0 .. K + 1
        return k == 0 ? make_int2(0, 0) : k > K ? make_int2(m, n) : make_int2(anc[k - 1].i, anc[k - 1].j);
    }
    // first k with P_k.i > i (strict) or P_k.i >= i
    __host__ __device__ __forceinline__ int bound(int i, bool strict) const {
        int a = 0, b = K + 2;
        while (a < b) {
            const int mid = (a + b) >> 1, pi = pt(mid).x;
            if (pi < i || (strict && pi == i)) a = mid + 1; else b = mid;
        }
        return a;
    }
    // column of the segment P_k -> P_{k+1} on row i, P_k.i < i < P_{k+1}.i
    __host__ __device__ __forceinline__ int seg(int k, int i) const {
        const int2 p = pt(k), q = pt(k + 1);
        return p.y + (int)((long long)(i - p.x) * (q.y - p.y) / (q.x - p.x));
    }
    __host__ __device__ __forceinline__ int cmin(int i) const {
        const int k = bound(i, false);
        return pt(k).x == i ? pt(k).y : seg(k - 1, i);
    }
    __host__ __device__ __forceinline__ int cmax(int i) const {
        const int k = bound(i, true);
        return pt(k - 1).x == i ? pt(k - 1).y : seg(k - 1, i);
    }
    __host__ __device__ __forceinline__ int lo(int i) const { const int v = cmin(i) - bw; return v < 0 ? 0 : v; }
    __host__ __device__ __forceinline__ int hi(int i) const { const long long v = (long long)cmax(i) + bw; return v > n ? n : (int)v; }
    __host__ __device__ __forceinline__ int s_lo(int i0, int WW) const { const int l = lo(i0 + 1); return ((l > 1 ? l : 1) - 1) / WW; }
    __host__ __device__ __forceinline__ int s_hi(int i0, int nrows, int WW) const {
        const int h = hi(i0 + nrows), s = ((h > 1 ? h : 1) - 1) / WW, sl = s_lo(i0, WW);
        return s > sl ? s : sl;
    }
    __host__ __device__ __forceinline__ bool inside(int i0, int nrows, int s, int WW) const {
        const int right = n < (s + 1) * WW ? n : (s + 1) * WW;
        return lo(i0 + nrows) <= s * WW + 1 && hi(i0 + 1) >= right;
    }
};

// Warp-collective: anchors[0 .. K) form a valid chain for an m x n pair (K >= 0, 0 <= i <= m, 0 <= j <= n, both
// coordinates non-decreasing).  Reads nothing when K < 0.
__device__ bool chain_ok(const psa_anchor* anc, int K, int m, int n) {
    if (K < 0) return false;
    bool bad = false;
    for (int k = threadIdx.x & 31; k < K; k += 32) {
        const psa_anchor a = anc[k];
        bad |= a.i < 0 || a.i > m || a.j < 0 || a.j > n;
        if (k > 0) { const psa_anchor p = anc[k - 1]; bad |= a.i < p.i || a.j < p.j; }
    }
    return !__any_sync(0xffffffffu, bad);
}

// Where the batch kernels take each pair's band from: the diagonal of psa_align_batch_banded, or the pair's chain.
struct DiagGuide {
    using BandT = Band;
    __device__ __forceinline__ Band band(long long, int m, int n, int bw) const { return Band{m, n, bw}; }
    __device__ __forceinline__ bool ok(long long, int, int) const { return true; }
};
struct ChainGuide {
    using BandT = ChainBand;
    const psa_anchor* anc;     // pair p: anc[off[p] .. off[p] + cnt[p])
    const int64_t* off;
    const int32_t* cnt;
    __device__ __forceinline__ ChainBand band(long long p, int m, int n, int bw) const { return ChainBand{m, n, bw, anc + off[p], cnt[p]}; }
    __device__ __forceinline__ bool ok(long long p, int m, int n) const {
        const int k = cnt[p];
        return chain_ok(k >= 0 ? anc + off[p] : nullptr, k, m, n);
    }
};

// Record of a pair whose chain the device form rejects: -inf corners and score, end state 0 (no other path produces
// it), every cell 0, aln_len 0.
__device__ __forceinline__ psa_batch_item rejected_item() {
    psa_batch_item r;
    r.t1 = r.t2 = r.t3 = r.score = PSA_NEG_INF;
    r.end_state = 0; r.end_i = r.end_j = r.start_i = r.start_j = 0; r.aln_len = 0;
    return r;
}

template <int MODE>
__device__ __forceinline__ constexpr int oob_H() { return MODE == PSA_LOCAL ? 0 : PSA_KNEG; }

// Checkpoints of a banded traceback fill, per computed tile (rb, s) of the <128, 8> grid: the tile's bottom row (H, F
// over its W columns) and its right column (H, E over its R rows).  Row block rb's tiles are records
// tile_base[rb] .. tile_base[rb] + s_hi - s_lo, in strip order.
constexpr int REC = 2 * W + 2 * R;     // ints per tile record
template <class BandT>
struct BandCkT {
    BandT B;
    int* rec;
    long long* tile_base;              // [NB]
};
using BandCk = BandCkT<Band>;

struct BandSmem {
    WarpSmem<R> w;
    int lo[R], hi[R];                  // band of each row of the row block
};

// H and F of row i0 (the top boundary of row block rb) at column j.  prev: row block rb-1's strips p_lo .. p_hi, kept in
// the recycled row J.hbufH / J.hbufF (score only) or in the records from rec_prev on (traceback).
template <int MODE, int WW, bool TB, class BandT>
__device__ __forceinline__ void band_top(const LongJob& J, const BandT& B, const int* rec_prev, int rb, int i0, int p_lo, int p_hi,
                                         int j, int& H, int& F) {
    F = PSA_KNEG;
    if (rb == 0) { H = j <= B.hi(0) ? border_row0_H<MODE>(j, J.g, J.h) : oob_H<MODE>(); return; }
    if (j == 0) { H = B.lo(i0) == 0 ? border_col0_H<MODE>(i0, J.g, J.h) : oob_H<MODE>(); return; }
    const int sj = (j - 1) / WW;
    if (sj < p_lo || sj > p_hi) { H = oob_H<MODE>(); return; }
    if (TB) {
        const int* rr = rec_prev + (long long)(sj - p_lo) * REC;
        H = __ldcg(rr + (j - 1 - sj * WW)); F = __ldcg(rr + W + (j - 1 - sj * WW));
    } else {
        H = __ldcg(J.hbufH + j); F = __ldcg(J.hbufF + j);
    }
}

// One row block of a banded pair, warp-collective.  Score only (TB = false): <128, KK> grid, TF-form sweeps, bottom row
// into the recycled row.  Traceback fill (TB = true): <128, 8> grid, sweep<> without codes, every tile's bottom row and
// right column into the records rec_cur (row block rb) -- rec_prev are row block rb-1's.
// WAIT (one pair over many warps): row block rb-1 may still be running; J.progress[rb] = 1 + the last strip finished.
template <int MODE, int KK, bool TB, bool WAIT = false, class BandT>
__device__ void process_rowblock_banded(const LongJob& J, const BandT& B, int rb, BandSmem& sm, Track& tr, int* rec_cur,
                                        const int* rec_prev) {
    constexpr int WW = 32 * KK;
    static_assert(!TB || WW == W, "traceback checkpoints use the walk's tile grid");
    const int lane = threadIdx.x & 31;
    const int m = J.m, n = J.n, g = J.g, h = J.h;
    const int i0 = rb * R, nrows = min(R, m - i0);
    const int s_lo = B.s_lo(i0, WW), s_hi = B.s_hi(i0, nrows, WW);
    const int p_lo = rb > 0 ? B.s_lo(i0 - R, WW) : 0, p_hi = rb > 0 ? B.s_hi(i0 - R, R, WW) : -1;
    for (int r = lane; r < nrows; r += 32) {
        const int i = i0 + 1 + r;
        sm.w.sA[r] = J.a[i0 + r];
        sm.lo[r] = B.lo(i); sm.hi[r] = B.hi(i);
        sm.w.bH[0][r] = (s_lo == 0 && sm.lo[r] == 0) ? border_col0_H<MODE>(i, g, h) : oob_H<MODE>();
        sm.w.bE[0][r] = PSA_KNEG;
    }
    // Row block rb-1 wrote strips p_lo .. p_hi of row i0; the top of strip s and the corner H[i0][s_lo*WW] (strip s_lo - 1)
    // are ready once it has finished strip min(s, p_hi).  Polling as process_rowblock does.
    auto wait_for = [&](int strip) {
        if constexpr (WAIT) {
            if (rb > 0) {
                unsigned ns = 32;
                while (ld_relaxed(J.progress + rb - 1) <= strip) { __nanosleep(ns); if (ns < 2048) ns <<= 1; }
                __threadfence();
                __syncwarp();
            }
        }
    };
    wait_for(min(s_lo, p_hi));
    int corner, dummy;
    band_top<MODE, WW, TB>(J, B, rec_prev, rb, i0, p_lo, p_hi, s_lo * WW, corner, dummy);
    __syncwarp();
    int cur = 0;
    int cap1 = PSA_KNEG, cap2 = PSA_KNEG, cap3 = PSA_KNEG;
    bool captured = false;
    for (int s = s_lo; s <= s_hi; ++s) {
        if (s > s_lo && s <= p_hi) wait_for(s);
        const int c0 = s * WW + lane * KK;
        const bool inside = B.inside(i0, nrows, s, WW);
        int hlast;
        if constexpr (TB) {
            Cols<KK> cs;
#pragma unroll
            for (int k = 0; k < KK; ++k) {
                const int j = c0 + k + 1;
                cs.b[k] = (j <= n) ? (int)J.b[j - 1] : 256;
                if (j <= n) band_top<MODE, WW, TB>(J, B, rec_prev, rb, i0, p_lo, p_hi, j, cs.H[k], cs.F[k]);
                else { cs.H[k] = PSA_KNEG; cs.F[k] = PSA_KNEG; }
            }
            hlast = cs.H[KK - 1];
            int hd = __shfl_up_sync(0xffffffffu, hlast, 1);
            if (lane == 0) hd = corner;
            Track tt{0, 0, 0};
            int* rc = rec_cur + (long long)(s - s_lo) * REC;
            if (inside) sweep<KK, MODE, false>(cs, hd, sm.w.bH[cur], sm.w.bE[cur], rc + 2 * W, rc + 2 * W + R, sm.w.sA, nrows, i0, c0,
                                               m, n, g, h, nullptr, tt, cap1, cap2, cap3);
            else sweep<KK, MODE, false, true>(cs, hd, sm.w.bH[cur], sm.w.bE[cur], rc + 2 * W, rc + 2 * W + R, sm.w.sA, nrows, i0, c0,
                                              m, n, g, h, nullptr, tt, cap1, cap2, cap3, sm.lo, sm.hi);
            if (MODE == PSA_LOCAL && tt.best > 0) {      // first cell of the tile's best, in row-major order, against the earlier tiles'
                const bool better = tt.best > tr.best || (tt.best == tr.best && (tt.bi < tr.bi || (tt.bi == tr.bi && tt.bj < tr.bj)));
                if (better) tr = tt;
            }
#pragma unroll
            for (int k = 0; k < KK; ++k) { rc[lane * KK + k] = cs.H[k]; rc[W + lane * KK + k] = cs.F[k]; }
            __syncwarp();
            // the right column went straight to the record; the next tile's left boundary is read from there
            for (int r = lane; r < nrows; r += 32) { sm.w.bH[cur ^ 1][r] = rc[2 * W + r]; sm.w.bE[cur ^ 1][r] = rc[2 * W + R + r]; }
        } else {
            ColsS<KK> cs;
#pragma unroll
            for (int k = 0; k < KK; ++k) {
                const int j = c0 + k + 1;
                cs.b[k] = (j <= n) ? (int)J.b[j - 1] : 256;
                int H0 = oob_H<MODE>(), F0 = PSA_KNEG;
                if (j <= n) band_top<MODE, WW, TB>(J, B, rec_prev, rb, i0, p_lo, p_hi, j, H0, F0);
                cs.set_top(k, H0, F0, g + h);
                cs.set_key_addend(k, j <= n, g + h);
            }
            hlast = cs.top_H(KK - 1, g + h);
            int hd = __shfl_up_sync(0xffffffffu, hlast, 1);
            if (lane == 0) hd = corner;
            int bestkey = 0, besti = 0;
            if (inside) sweep_score<KK, MODE>(cs, hd, sm.w.bH[cur], sm.w.bE[cur], sm.w.bH[cur ^ 1], sm.w.bE[cur ^ 1], sm.w.sA, nrows, i0,
                                              c0, m, n, g, h, J.mul8, bestkey, besti, cap1, cap2, cap3);
            else sweep_score<KK, MODE, true>(cs, hd, sm.w.bH[cur], sm.w.bE[cur], sm.w.bH[cur ^ 1], sm.w.bE[cur ^ 1], sm.w.sA, nrows, i0,
                                             c0, m, n, g, h, J.mul8, bestkey, besti, cap1, cap2, cap3, sm.lo, sm.hi);
            if (MODE == PSA_LOCAL) {          // as process_rowblock
                const int t1v = bestkey / key_mult(KK);
                const int bj = c0 + (key_mult(KK) - 1 - (bestkey % key_mult(KK))) + 1;
                if (t1v > 0 && bj <= n) {
                    const bool better = t1v > tr.best || (t1v == tr.best && (besti < tr.bi || (besti == tr.bi && bj < tr.bj)));
                    if (better) { tr.best = t1v; tr.bi = besti; tr.bj = bj; }
                }
            }
#pragma unroll
            for (int k = 0; k < KK; ++k) {
                const int j = c0 + k + 1;
                if (j <= n) { J.hbufH[j] = cs.top_H(k, g + h); J.hbufF[j] = cs.ff[k]; }
            }
        }
        if ((i0 + nrows == m) && (n > s * WW) && (n <= (s + 1) * WW)) captured = true;
        corner = __shfl_sync(0xffffffffu, hlast, 31);   // H[i0][(s+1)*WW]
        cur ^= 1;
        __syncwarp();
        if constexpr (WAIT) {
            __threadfence();
            __syncwarp();
            if (lane == 0) st_release(J.progress + rb, s + 1);
        }
    }
    if (MODE == PSA_GLOBAL && captured) {
        const int src = ((n - 1) % WW) / KK;
        if (lane == src) { J.corner[0] = cap1; J.corner[1] = cap2; J.corner[2] = cap3; }
    }
}

// Banded result record: a global call whose band admits no path reports -inf corners with end state 1 (the state
// find_alignment picks among equal corners) and no columns.
__device__ __forceinline__ psa_batch_item banded_item(psa_batch_item r) {
    if (r.score == PSA_NEG_INF) r.end_state = 1;
    return r;
}

struct BandedBatch {
    psa_batch_args P;
    int* hbuf;                 // per resident warp: 2*(max_n+1) ints
    long long hbuf_warp_stride;
    int* ticket;
    int bw;
};

// Score only: one warp per pair, one recycled boundary row, <128, 16> tiles.  G: each pair's band (DiagGuide /
// ChainGuide); a pair whose chain G rejects gets rejected_item() and touches nothing else.
template <int MODE, class Guide>
__device__ __forceinline__ void banded_batch(const BandedBatch& Bt, const Guide& G) {
    constexpr int KB = 16;
    __shared__ BandSmem smem[WPB];
    __shared__ unsigned long long s_best[WPB];
    __shared__ int s_corner[WPB][4];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    BandSmem& sm = smem[w];
    const long long gw = (long long)blockIdx.x * WPB + w;
    for (;;) {
        long long p = 0;
        if (lane == 0) p = atomicAdd(Bt.ticket, 1);
        p = __shfl_sync(0xffffffffu, p, 0);
        if (p >= Bt.P.n_pairs) break;
        LongJob J;
        J.a = Bt.P.bases_a + Bt.P.off_a[p]; J.b = Bt.P.bases_b + Bt.P.off_b[p];
        J.m = Bt.P.len_a[p]; J.n = Bt.P.len_b[p]; J.g = Bt.P.g; J.h = Bt.P.h; J.mul8 = key_mult(KB);
        J.hbufH = Bt.hbuf + gw * Bt.hbuf_warp_stride; J.hbufF = J.hbufH + Bt.hbuf_warp_stride / 2; J.hb_stride = 0;
        J.ckvH = nullptr; J.ckvE = nullptr; J.progress = nullptr; J.ticket = nullptr;
        J.best = &s_best[w]; J.corner = s_corner[w];
        J.col0 = 0; J.n_total = J.n; J.row_off = 0;
        J.start_type = -1; J.end_type = -1;
        if (lane == 0) { s_best[w] = 0ull; s_corner[w][0] = s_corner[w][1] = s_corner[w][2] = PSA_KNEG; }
        __syncwarp();
        const bool ok = G.ok(p, J.m, J.n);
        if (ok && J.m > 0 && J.n > 0) {
            const auto B = G.band(p, J.m, J.n, Bt.bw);
            Track tr{0, 0, 0};
            const int NB = (J.m + R - 1) / R;
            for (int rb = 0; rb < NB; ++rb) process_rowblock_banded<MODE, KB, false>(J, B, rb, sm, tr, nullptr, nullptr);
            flush_track<MODE>(J, tr);
            __syncwarp();
        }
        if (lane == 0) {
            psa_batch_item r;
            if (J.m <= 0 || J.n <= 0) r = empty_item<MODE>(J.m, J.n, J.g, J.h, -1, -1);
            else if (MODE == PSA_LOCAL) r = local_item_from_key(s_best[w]);
            else r = global_item(s_corner[w][0], s_corner[w][1], s_corner[w][2], J.m, J.n, J.h, -1);
            Bt.P.items[p] = ok ? banded_item(r) : rejected_item();
        }
        __syncwarp();
    }
}

template <int MODE>
__global__ void __launch_bounds__(WPB * 32) psa_banded_batch_kernel(BandedBatch Bt) { banded_batch<MODE>(Bt, DiagGuide{}); }
template <int MODE>
__global__ void __launch_bounds__(WPB * 32) psa_guided_batch_kernel(BandedBatch Bt, ChainGuide G) { banded_batch<MODE>(Bt, G); }

// Traceback: pair p of the chunk [p0, p0 + count) owns slot p - p0: [best (8 B) | corner (3 x 4 B) | pad to 256 B |
// tile_base (NB x 8 B, padded to 256 B) | tile records (REC ints each)], inside slot_bytes (planned from max m, max n, bw).
struct BandedTb {
    psa_batch_args P;
    long long p0, count;
    uint8_t* region;
    long long slot_bytes;
    int* ticket;
    int bw;
};

template <class Guide>
__device__ __forceinline__ LongJob banded_tb_job(const BandedTb& Bt, const Guide& G, long long p, BandCkT<typename Guide::BandT>& bk) {
    const psa_batch_args& P = Bt.P;
    LongJob J;
    J.a = P.bases_a + P.off_a[p]; J.b = P.bases_b + P.off_b[p];
    J.m = P.len_a[p]; J.n = P.len_b[p]; J.g = P.g; J.h = P.h; J.mul8 = key_mult(K);
    uint8_t* slot = Bt.region + (p - Bt.p0) * Bt.slot_bytes;
    const int NB = (J.m + R - 1) / R;
    J.best = (unsigned long long*)slot; J.corner = (int*)(slot + 8);
    J.hbufH = nullptr; J.hbufF = nullptr; J.hb_stride = 0;
    J.ckvH = nullptr; J.ckvE = nullptr; J.progress = nullptr; J.ticket = nullptr;
    J.col0 = 0; J.n_total = J.n; J.row_off = 0; J.start_type = -1; J.end_type = -1;
    bk.B = G.band(p, J.m, J.n, Bt.bw);
    bk.tile_base = (long long*)(slot + 256);
    bk.rec = (int*)(slot + 256 + up256_d((long long)NB * 8));
    return J;
}

template <int MODE, class Guide>
__device__ __forceinline__ void banded_tb_fill(const BandedTb& Bt, const Guide& G) {
    __shared__ BandSmem smem[WPB];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    BandSmem& sm = smem[w];
    for (;;) {
        long long q = 0;
        if (lane == 0) q = atomicAdd(Bt.ticket, 1);
        q = __shfl_sync(0xffffffffu, q, 0);
        if (q >= Bt.count) break;
        BandCkT<typename Guide::BandT> bk;
        const LongJob J = banded_tb_job(Bt, G, Bt.p0 + q, bk);
        if (J.m <= 0 || J.n <= 0) continue;          // borders only: the walk kernel writes the item
        if (!G.ok(Bt.p0 + q, J.m, J.n)) continue;    // rejected chain: its slot stays untouched, the walk writes the item
        if (lane == 0) { *J.best = 0ull; J.corner[0] = J.corner[1] = J.corner[2] = PSA_KNEG; }
        __syncwarp();
        Track tr{0, 0, 0};
        const int NB = (J.m + R - 1) / R;
        long long base = 0, prev = 0;
        for (int rb = 0; rb < NB; ++rb) {
            if (lane == 0) bk.tile_base[rb] = base;
            process_rowblock_banded<MODE, K, true>(J, bk.B, rb, sm, tr, bk.rec + base * REC, bk.rec + prev * REC);
            prev = base;
            base += bk.B.s_hi(rb * R, min(R, J.m - rb * R), W) - bk.B.s_lo(rb * R, W) + 1;
        }
        flush_track<MODE>(J, tr);
        __syncwarp();
    }
}

template <int MODE>
__global__ void __launch_bounds__(WPB * 32) psa_banded_tb_fill_kernel(BandedTb Bt) { banded_tb_fill<MODE>(Bt, DiagGuide{}); }
template <int MODE>
__global__ void __launch_bounds__(WPB * 32) psa_guided_tb_fill_kernel(BandedTb Bt, ChainGuide G) { banded_tb_fill<MODE>(Bt, G); }

// recompute_tile for the banded layout: boundaries from the records, out-of-band values outside them, masked sweep.
template <int MODE, class BandT>
__device__ void recompute_tile_banded(const LongJob& J, const BandCkT<BandT>& bk, int rb, int s, int nrows, uint32_t* dirs, int* lbH,
                                      int* lbE, uint8_t* sA, int* bLo, int* bHi) {
    const int lane = threadIdx.x & 31;
    const int m = J.m, n = J.n, g = J.g, h = J.h;
    const BandT& B = bk.B;
    const int i0 = rb * R, c0 = s * W + lane * K;
    const int s_lo = B.s_lo(i0, W);
    const int p_lo = rb > 0 ? B.s_lo(i0 - R, W) : 0, p_hi = rb > 0 ? B.s_hi(i0 - R, R, W) : -1;
    const int* rec_prev = rb > 0 ? bk.rec + __ldcg(bk.tile_base + rb - 1) * REC : nullptr;
    const int* rec_left = s > s_lo ? bk.rec + (__ldcg(bk.tile_base + rb) + (s - 1 - s_lo)) * REC : nullptr;
    __syncwarp();
    for (int q = lane; q < nrows; q += 32) {
        const int i = i0 + 1 + q;
        sA[q] = J.a[i0 + q];
        bLo[q] = B.lo(i); bHi[q] = B.hi(i);
        if (s > s_lo) { lbH[q] = __ldcg(rec_left + 2 * W + q); lbE[q] = __ldcg(rec_left + 2 * W + R + q); }
        else { lbH[q] = (s == 0 && bLo[q] == 0) ? border_col0_H<MODE>(i, g, h) : oob_H<MODE>(); lbE[q] = PSA_KNEG; }
    }
    Cols<K> cs;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int jj = c0 + k + 1;
        cs.b[k] = (jj <= n) ? (int)J.b[jj - 1] : 256;
        if (jj <= n) band_top<MODE, W, true>(J, B, rec_prev, rb, i0, p_lo, p_hi, jj, cs.H[k], cs.F[k]);
        else { cs.H[k] = PSA_KNEG; cs.F[k] = PSA_KNEG; }
    }
    int hd = __shfl_up_sync(0xffffffffu, cs.H[K - 1], 1);
    int corner, dummy;
    band_top<MODE, W, true>(J, B, rec_prev, rb, i0, p_lo, p_hi, s * W, corner, dummy);
    if (lane == 0) hd = corner;
    __syncwarp();
    Track tr{0, 0, 0};
    int d1 = 0, d2 = 0, d3 = 0;
    sweep<K, MODE, true, true>(cs, hd, lbH, lbE, nullptr, nullptr, sA, nrows, i0, c0, m, n, g, h, dirs, tr, d1, d2, d3, bLo, bHi);
    __syncwarp();
}

// Lane 0's steps of a banded walk through tile (trb, ts), whose codes `dirs` holds: ops from (i, j, state) on until the
// path ends (need_rb stays -1) or its next source cell lies in tile (need_rb, need_s).  The loop of tb_walk_banded,
// which keeps its own copy so that the batch walk compiles unchanged.
template <int MODE>
__device__ __forceinline__ void walk_steps(const uint32_t* dirs, int trb, int ts, int& i, int& j, int& state, int& len,
                                           uint32_t& acc, uint32_t* ops, psa_batch_item& r, int& need_rb, int& need_s) {
    while (i > 0 && j > 0) {
        const int si = (state == 2) ? i : i - 1;
        const int sj = (state == 3) ? j : j - 1;
        const bool border = (si == 0 || sj == 0);
        int code = 0;
        if (!border) {
            const int rb = (si - 1) / R, s = (sj - 1) / W;
            if (rb != trb || s != ts) { need_rb = rb; need_s = s; break; }
            const int cj = sj - 1 - s * W;
            code = (dirs[(si - 1 - rb * R) * 32 + cj / K] >> (4 * (cj % K))) & 15;
        }
        acc |= (uint32_t)state << (2 * (len & 15));
        if ((len & 15) == 15) { ops[len >> 4] = acc; acc = 0; }
        ++len;
        r.start_i = i; r.start_j = j;
        const int ns = next_state<MODE>(state, code, border);
        if (ns == 0) { i = 0; break; }
        state = ns; i = si; j = sj;
    }
}

// tb_walk over the banded layout: the same steps, every tile the path enters recomputed by recompute_tile_banded.  (A
// separate function so that the unbanded walks keep their code.)
template <int MODE, class BandT>
__device__ void tb_walk_banded(const LongJob& J, const BandCkT<BandT>& bk, psa_batch_item& r, uint32_t* ops, uint32_t* dirs, int* lbH,
                               int* lbE, uint8_t* sA, int* bLo, int* bHi) {
    const int lane = threadIdx.x & 31;
    const int m = J.m;
    int i = r.end_i, j = r.end_j, state = r.end_state;
    int trb = -1, ts = -1;      // tile currently held in `dirs`
    int len = 0;
    uint32_t acc = 0;
    bool done = !(i > 0 && j > 0);
    while (!done) {
        int need_rb = -1, need_s = -1;
        if (lane == 0) {
            while (i > 0 && j > 0) {
                const int si = (state == 2) ? i : i - 1;
                const int sj = (state == 3) ? j : j - 1;
                const bool border = (si == 0 || sj == 0);
                int code = 0;
                if (!border) {
                    const int rb = (si - 1) / R, s = (sj - 1) / W;
                    if (rb != trb || s != ts) { need_rb = rb; need_s = s; break; }
                    const int cj = sj - 1 - s * W;
                    code = (dirs[(si - 1 - rb * R) * 32 + cj / K] >> (4 * (cj % K))) & 15;
                }
                acc |= (uint32_t)state << (2 * (len & 15));
                if ((len & 15) == 15) { ops[len >> 4] = acc; acc = 0; }
                ++len;
                r.start_i = i; r.start_j = j;
                const int ns = next_state<MODE>(state, code, border);
                if (ns == 0) { i = 0; break; }
                state = ns; i = si; j = sj;
            }
        }
        need_rb = __shfl_sync(0xffffffffu, need_rb, 0);
        need_s = __shfl_sync(0xffffffffu, need_s, 0);
        if (need_rb < 0) break;
        const int need_row = __shfl_sync(0xffffffffu, (lane == 0) ? ((state == 2) ? i : i - 1) : 0, 0);
        const int i0 = need_rb * R, nrows = min(min(R, m - i0), need_row - i0);
        recompute_tile_banded<MODE>(J, bk, need_rb, need_s, nrows, dirs, lbH, lbE, sA, bLo, bHi);
        trb = need_rb; ts = need_s;
    }
    if (lane == 0) {
        if (len & 15) ops[len >> 4] = acc;
        r.aln_len = len;
    }
}

// tid, bid: threadIdx.x, blockIdx.x, read by the kernel itself (which knows their range from its launch bounds)
template <int MODE, class Guide>
__device__ __forceinline__ void banded_tb_walk(const BandedTb& Bt, const Guide& G, unsigned tid, unsigned bid) {
    __shared__ uint32_t dirs[WALK_WPB][R * 32];
    __shared__ int lbH[WALK_WPB][R], lbE[WALK_WPB][R], bLo[WALK_WPB][R], bHi[WALK_WPB][R];
    __shared__ uint8_t sA[WALK_WPB][R];
    const int w = tid >> 5;
    const long long q = (long long)bid * WALK_WPB + w;
    if (q >= Bt.count) return;
    const long long p = Bt.p0 + q;
    BandCkT<typename Guide::BandT> bk;
    const LongJob J = banded_tb_job(Bt, G, p, bk);
    psa_batch_item r;
    if (!G.ok(p, J.m, J.n)) {
        r = rejected_item();
    } else if (J.m <= 0 || J.n <= 0) {
        r = empty_item<MODE>(J.m, J.n, J.g, J.h, -1, -1);
    } else {
        r = banded_item(tb_end<MODE>(J));
        if (r.score != PSA_NEG_INF)
            tb_walk_banded<MODE>(J, bk, r, Bt.P.ops + p * Bt.P.ops_stride_words, dirs[w], lbH[w], lbE[w], sA[w], bLo[w], bHi[w]);
    }
    if ((tid & 31) == 0) Bt.P.items[p] = r;
}

template <int MODE>
__global__ void __launch_bounds__(WALK_WPB * 32) psa_banded_tb_walk_kernel(BandedTb Bt) {
    banded_tb_walk<MODE>(Bt, DiagGuide{}, threadIdx.x, blockIdx.x);
}
template <int MODE>
__global__ void __launch_bounds__(WALK_WPB * 32) psa_guided_tb_walk_kernel(BandedTb Bt, ChainGuide G) {
    banded_tb_walk<MODE>(Bt, G, threadIdx.x, blockIdx.x);
}

// ---- one banded pair over the whole GPU (psa_align_pair_banded, psa_align_long_banded_device) --------------------------
// Fill: the row blocks of the batch kernels above, handed out by ticket in increasing order to every warp of the grid, with
// the progress handshake of process_rowblock_banded<..., WAIT>.  Score only: one recycled H/F row of n + 1 ints (row block
// rb reads strip s of it before it overwrites it, rb + 1 reads it only afterwards).  Traceback: the per-tile records of
// BandCk at tile_base[rb], computed beforehand by psa_banded_tile_base_kernel.
template <class BandT>
struct PairFillT {
    LongJob J;                 // progress, ticket, best, corner; hbufH / hbufF: the recycled row (score only)
    BandCkT<BandT> bk;         // traceback only
};
struct BandedPair : PairFillT<Band> {};
struct GuidedPair : PairFillT<ChainBand> {};   // psa_align_pair_guided: the chain, validated on the host

template <int MODE, int KK, bool TB, class BandT>
__device__ __forceinline__ void banded_pair_fill(const PairFillT<BandT>& P) {
    __shared__ BandSmem smem[WPB];
    BandSmem& sm = smem[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const LongJob& J = P.J;
    const int NB = (J.m + R - 1) / R;
    Track tr{0, 0, 0};
    for (;;) {
        int rb = 0;
        if (lane == 0) rb = atomicAdd(J.ticket, 1);
        rb = __shfl_sync(0xffffffffu, rb, 0);
        if (rb >= NB) break;
        int* cur = TB ? P.bk.rec + P.bk.tile_base[rb] * REC : nullptr;
        const int* prev = (TB && rb > 0) ? P.bk.rec + P.bk.tile_base[rb - 1] * REC : nullptr;
        process_rowblock_banded<MODE, KK, TB, true>(J, P.bk.B, rb, sm, tr, cur, prev);
    }
    flush_track<MODE>(J, tr);
}

template <int MODE, int KK, bool TB>
__global__ void __launch_bounds__(WPB * 32) psa_banded_pair_fill_kernel(BandedPair P) { banded_pair_fill<MODE, KK, TB>(P); }
template <int MODE, int KK, bool TB>
__global__ void __launch_bounds__(WPB * 32) psa_guided_pair_fill_kernel(GuidedPair P) { banded_pair_fill<MODE, KK, TB>(P); }

// tile_base[rb] = tiles of row blocks 0 .. rb-1 (NB <= 16384: at most 16 row blocks per thread).
template <class BandT>
__device__ __forceinline__ void banded_tile_base(const BandT& B, long long* tile_base) {
    __shared__ long long part[1024];
    const int NB = (B.m + R - 1) / R, t = threadIdx.x;
    const int per = (NB + 1023) / 1024, r0 = min(NB, t * per), r1 = min(NB, r0 + per);
    auto tiles = [&](int rb) { return (long long)(B.s_hi(rb * R, min(R, B.m - rb * R), W) - B.s_lo(rb * R, W) + 1); };
    long long sum = 0;
    for (int rb = r0; rb < r1; ++rb) sum += tiles(rb);
    part[t] = sum;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {          // inclusive scan
        const long long v = t >= off ? part[t - off] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    long long base = part[t] - sum;
    for (int rb = r0; rb < r1; ++rb) { tile_base[rb] = base; base += tiles(rb); }
}

__global__ void __launch_bounds__(1024) psa_banded_tile_base_kernel(Band B, long long* tile_base) { banded_tile_base(B, tile_base); }
__global__ void __launch_bounds__(1024) psa_guided_tile_base_kernel(ChainBand B, long long* tile_base) { banded_tile_base(B, tile_base); }

// Walk: bottom-up in windows of row blocks rb_lo .. rb_hi-1.  For each window psa_banded_pair_codes_kernel first recomputes
// the codes of every band tile of the window the path can still reach -- rows above the walk's current row, strips not
// right of its current column -- all tiles in parallel; then the one-warp walk copies those codes in tile by tile (a tile
// missing from the buffer is recomputed on demand) and leaves its state in BandedWalk for the next window.
struct BandedWalk {
    psa_batch_item r;          // the record being completed
    int i, j, state, len;
    uint32_t acc;              // partial op word
    int done;
};

struct BandedPairTb {
    LongJob J;
    BandCk bk;
    uint32_t* codes;           // [rb - rb_lo][tpr] tiles of R*32 code words
    int tpr;                   // tile slots per row block (>= s_hi - s_lo + 1 of every row block)
    int rb_lo, rb_hi;          // this window; rb_hi == NB: the first window
    BandedWalk* walk;
    psa_batch_item* item;
    uint32_t* ops;             // null: score only (one window, which writes the record)
};
struct GuidedPairTb {
    LongJob J;
    BandCkT<ChainBand> bk;
    uint32_t* codes;           // [rb - rb_lo][tpr] tiles of R*32 code words
    int tpr;                   // tile slots per row block (>= s_hi - s_lo + 1 of every row block)
    int rb_lo, rb_hi;          // this window; rb_hi == NB: the first window
    BandedWalk* walk;
    psa_batch_item* item;
    uint32_t* ops;             // null: score only (one window, which writes the record)
};

// Start of the walk: the end cell and end state of the banded record in the first window, else the saved state.
template <int MODE, class TbT>
__device__ __forceinline__ BandedWalk walk_start(const TbT& T) {
    if (T.rb_hi * R < T.J.m) return *T.walk;
    BandedWalk w;
    w.r = banded_item(tb_end<MODE>(T.J));
    w.i = w.r.end_i; w.j = w.r.end_j; w.state = w.r.end_state; w.len = 0; w.acc = 0;
    w.done = T.ops == nullptr || w.r.score == PSA_NEG_INF;
    return w;
}

constexpr int CODES_WPB = 2;
template <int MODE, class TbT>
__device__ __forceinline__ void banded_pair_codes(const TbT& T, unsigned tid, unsigned bid) {   // as banded_tb_walk
    __shared__ uint32_t dirs[CODES_WPB][R * 32];
    __shared__ int lbH[CODES_WPB][R], lbE[CODES_WPB][R], bLo[CODES_WPB][R], bHi[CODES_WPB][R];
    __shared__ uint8_t sA[CODES_WPB][R];
    const int w = tid >> 5, lane = tid & 31;
    const long long u = (long long)bid * CODES_WPB + w;
    if (u >= (long long)(T.rb_hi - T.rb_lo) * T.tpr) return;
    const int rb = T.rb_lo + (int)(u / T.tpr), t = (int)(u % T.tpr);
    const BandedWalk st = walk_start<MODE>(T);
    const auto& B = T.bk.B;
    const int i0 = rb * R, nrows = min(R, T.J.m - i0), s = B.s_lo(i0, W) + t;
    if (st.done || i0 >= st.i || s > B.s_hi(i0, nrows, W) || s * W >= st.j) return;
    recompute_tile_banded<MODE>(T.J, T.bk, rb, s, nrows, dirs[w], lbH[w], lbE[w], sA[w], bLo[w], bHi[w]);
    uint4* out = reinterpret_cast<uint4*>(T.codes + u * (R * 32));
    const uint4* in = reinterpret_cast<const uint4*>(dirs[w]);
    for (int q = lane; q < nrows * 8; q += 32) out[q] = in[q];
}

template <int MODE>
__global__ void __launch_bounds__(CODES_WPB * 32) psa_banded_pair_codes_kernel(BandedPairTb T) { banded_pair_codes<MODE>(T, threadIdx.x, blockIdx.x); }
template <int MODE>
__global__ void __launch_bounds__(CODES_WPB * 32) psa_guided_pair_codes_kernel(GuidedPairTb T) { banded_pair_codes<MODE>(T, threadIdx.x, blockIdx.x); }

template <int MODE>
__global__ void __launch_bounds__(32) psa_banded_pair_walk_kernel(BandedPairTb T) {
    __shared__ uint32_t dirs[R * 32];
    __shared__ int lbH[R], lbE[R], bLo[R], bHi[R];
    __shared__ uint8_t sA[R];
    const int lane = threadIdx.x;
    const LongJob& J = T.J;
    const Band& B = T.bk.B;
    BandedWalk st = walk_start<MODE>(T);
    const bool first = T.rb_hi * R >= J.m;
    if (st.done && !first) return;                        // finished in an earlier window
    int i = st.i, j = st.j, state = st.state, len = st.len;
    uint32_t acc = st.acc;
    bool done = st.done || !(i > 0 && j > 0);
    int trb = -1, ts = -1;
    while (!done) {
        int need_rb = -1, need_s = -1;
        if (lane == 0) walk_steps<MODE>(dirs, trb, ts, i, j, state, len, acc, T.ops, st.r, need_rb, need_s);
        need_rb = __shfl_sync(0xffffffffu, need_rb, 0);
        need_s = __shfl_sync(0xffffffffu, need_s, 0);
        if (need_rb < 0) { done = true; break; }
        if (need_rb < T.rb_lo) break;                     // the next window's rows
        const int need_row = __shfl_sync(0xffffffffu, (lane == 0) ? ((state == 2) ? i : i - 1) : 0, 0);
        const int i0 = need_rb * R, full = min(R, J.m - i0), nrows = min(full, need_row - i0);
        const int t = need_s - B.s_lo(i0, W);
        if (t >= 0 && t < T.tpr && need_s <= B.s_hi(i0, full, W)) {
            const uint4* in = reinterpret_cast<const uint4*>(T.codes + ((long long)(need_rb - T.rb_lo) * T.tpr + t) * (R * 32));
            uint4* out = reinterpret_cast<uint4*>(dirs);
            const int total = nrows * 8;
            __syncwarp();
            for (int q0 = 0; q0 < total; q0 += 256) {       // as tb_walk: eight 16-byte loads in flight per lane
                uint4 v[8];
#pragma unroll
                for (int x = 0; x < 8; ++x) { const int q = q0 + x * 32 + lane; if (q < total) v[x] = __ldcg(in + q); }
#pragma unroll
                for (int x = 0; x < 8; ++x) { const int q = q0 + x * 32 + lane; if (q < total) out[q] = v[x]; }
            }
            __syncwarp();
        } else {
            recompute_tile_banded<MODE>(J, T.bk, need_rb, need_s, nrows, dirs, lbH, lbE, sA, bLo, bHi);
        }
        trb = need_rb; ts = need_s;
    }
    if (lane == 0) {
        if (done) {
            if (T.ops != nullptr && st.r.score != PSA_NEG_INF) {     // as tb_walk_banded
                if (len & 15) T.ops[len >> 4] = acc;
                st.r.aln_len = len;
            }
            *T.item = st.r;
        }
        st.i = i; st.j = j; st.state = state; st.len = len; st.acc = acc; st.done = done;
        *T.walk = st;
    }
}


// The guided pair's walk: psa_banded_pair_walk_kernel's body over ChainBand.  A copy, not a shared template: inlined into
// a helper the diagonal kernel compiles to different SASS.
template <int MODE>
__global__ void __launch_bounds__(32) psa_guided_pair_walk_kernel(GuidedPairTb T) {
    __shared__ uint32_t dirs[R * 32];
    __shared__ int lbH[R], lbE[R], bLo[R], bHi[R];
    __shared__ uint8_t sA[R];
    const int lane = threadIdx.x;
    const LongJob& J = T.J;
    const auto& B = T.bk.B;
    BandedWalk st = walk_start<MODE>(T);
    const bool first = T.rb_hi * R >= J.m;
    if (st.done && !first) return;                        // finished in an earlier window
    int i = st.i, j = st.j, state = st.state, len = st.len;
    uint32_t acc = st.acc;
    bool done = st.done || !(i > 0 && j > 0);
    int trb = -1, ts = -1;
    while (!done) {
        int need_rb = -1, need_s = -1;
        if (lane == 0) walk_steps<MODE>(dirs, trb, ts, i, j, state, len, acc, T.ops, st.r, need_rb, need_s);
        need_rb = __shfl_sync(0xffffffffu, need_rb, 0);
        need_s = __shfl_sync(0xffffffffu, need_s, 0);
        if (need_rb < 0) { done = true; break; }
        if (need_rb < T.rb_lo) break;                     // the next window's rows
        const int need_row = __shfl_sync(0xffffffffu, (lane == 0) ? ((state == 2) ? i : i - 1) : 0, 0);
        const int i0 = need_rb * R, full = min(R, J.m - i0), nrows = min(full, need_row - i0);
        const int t = need_s - B.s_lo(i0, W);
        if (t >= 0 && t < T.tpr && need_s <= B.s_hi(i0, full, W)) {
            const uint4* in = reinterpret_cast<const uint4*>(T.codes + ((long long)(need_rb - T.rb_lo) * T.tpr + t) * (R * 32));
            uint4* out = reinterpret_cast<uint4*>(dirs);
            const int total = nrows * 8;
            __syncwarp();
            for (int q0 = 0; q0 < total; q0 += 256) {       // as tb_walk: eight 16-byte loads in flight per lane
                uint4 v[8];
#pragma unroll
                for (int x = 0; x < 8; ++x) { const int q = q0 + x * 32 + lane; if (q < total) v[x] = __ldcg(in + q); }
#pragma unroll
                for (int x = 0; x < 8; ++x) { const int q = q0 + x * 32 + lane; if (q < total) out[q] = v[x]; }
            }
            __syncwarp();
        } else {
            recompute_tile_banded<MODE>(J, T.bk, need_rb, need_s, nrows, dirs, lbH, lbE, sA, bLo, bHi);
        }
        trb = need_rb; ts = need_s;
    }
    if (lane == 0) {
        if (done) {
            if (T.ops != nullptr && st.r.score != PSA_NEG_INF) {     // as tb_walk_banded
                if (len & 15) T.ops[len >> 4] = acc;
                st.r.aln_len = len;
            }
            *T.item = st.r;
        }
        st.i = i; st.j = j; st.state = state; st.len = len; st.acc = acc; st.done = done;
        *T.walk = st;
    }
}

}  // namespace

// ---- host side ---------------------------------------------------------------------------
namespace {
int ensure_work(psa_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->d_work_bytes) return PSA_OK;
    if (ctx->d_work) cudaFree(ctx->d_work);
    ctx->d_work = nullptr; ctx->d_work_bytes = 0;
    bytes = ((bytes + bytes / 8) + (1 << 20) - 1) / (1 << 20) * (size_t)(1 << 20);
    if (cudaMalloc(&ctx->d_work, bytes) != cudaSuccess) {
        cudaGetLastError();
        return psa_fail(ctx, PSA_ERR_NOMEM, "cudaMalloc of long-pair work buffers failed (" + std::to_string(bytes >> 20) + " MiB)");
    }
    ctx->d_work_bytes = bytes;
    return PSA_OK;
}
size_t up256(size_t x) { return (x + 255) / 256 * 256; }
}  // namespace

// One long pair, sequences already on the device.  Writes *d_item (and d_ops when traceback).
int psa_launch_long_single(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h,
                           bool traceback, psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st,
                           int start_type, int end_type) {
    if (m <= 0 || n <= 0) return psa_fail(ctx, PSA_ERR_ARG, "long path needs m, n >= 1");
    if (m >= 0x1FFFFF || n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    // One pair that is wide enough to fill the GPU with strips, score only: the column-stationary systolic kernel
    // (psa_systolic.cu) -- no per-tile drains, every resident warp busy for all m rows.
    {
        const bool plain = (start_type == -1 && end_type == -1 && !traceback);
        // on ONE GPU the row-block tiles below are faster (wider lanes, 12 instead of ~25 instructions per cell); the
        // systolic kernel is what several GPUs share one pair with (psa_align_long_cyclic_device) and an option here
        const bool want = ctx->opt.long_systolic == 1;
        if (plain && want) return psa_launch_systolic(ctx, d_a, d_b, m, n, mode, g, h, 0, 1, 0, nullptr, nullptr, 0, d_item, st);
    }
    const int NB = (m + R - 1) / R, S = (n + W - 1) / W;
    const size_t row = up256((size_t)(n + 1) * 4);
    const size_t hb = traceback ? row * NB : row;
    const size_t ckv = traceback ? up256((size_t)S * (m + 1) * 4) : 0;
    size_t o = 0;
    const size_t o_hH = o; o += hb;
    const size_t o_hF = o; o += hb;
    const size_t o_vH = o; o += ckv;
    const size_t o_vE = o; o += ckv;
    const size_t o_pr = o; o += up256((size_t)NB * 4);
    const size_t o_misc = o; o += 256;      // ticket(4) | pad | best(8 @ +8) | corner(3*4 @ +16)
    // direction codes of the band tiles (16 KB each), recomputed in parallel before the walk
    const size_t band_bytes = (size_t)NB * BAND_TILES * R * 32 * 4;
    const bool use_band = traceback && band_bytes <= ((size_t)1 << 30) && ctx->opt.long_band;
    const size_t o_band = o; o += use_band ? band_bytes : 0;
    int rc = ensure_work(ctx, o);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_work;
    PSA_CUDA_OK(ctx, cudaMemsetAsync(d + o_pr, 0, (o_misc + 256) - o_pr, st));
    LongJob J;
    J.a = d_a; J.b = d_b; J.m = m; J.n = n; J.g = g; J.h = h; J.mul8 = 8;
    J.hbufH = (int*)(d + o_hH); J.hbufF = (int*)(d + o_hF);
    J.hb_stride = traceback ? (long long)(row / 4) : 0;
    J.ckvH = traceback ? (int*)(d + o_vH) : nullptr; J.ckvE = traceback ? (int*)(d + o_vE) : nullptr;
    J.progress = (int*)(d + o_pr);
    J.ticket = (int*)(d + o_misc);
    J.best = (unsigned long long*)(d + o_misc + 8);
    J.corner = (int*)(d + o_misc + 16);
    J.col0 = 0; J.n_total = n; J.row_off = 0;
    J.start_type = start_type; J.end_type = end_type;
    const bool typed = (J.start_type != -1 || J.end_type != -1);
    if (typed && mode != PSA_GLOBAL) return psa_fail(ctx, PSA_ERR_ARG, "start/end types apply to global alignment only");
    // geometry: checkpoints (traceback) fix the 128 x 256 tile grid; score-only runs may use taller row
    // blocks (less skew drain) and wider lanes (less per-step overhead)
    // At most one tile per strip column is in flight, so the wavefront is n/(32*K) tiles wide: pick the
    // widest lanes that still keep most of the resident warps busy (measured, same box: 1 Mbp <128,8> 865 ms,
    // <128,12> 815, <128,16> 725, <128,20> 639, <128,24> 635, <128,28> 638, <128,32> 698; 300 kbp <128,24> 156 ms,
    // <128,8> 159, <128,4> 136; 100 kbp <128,8> 42 ms vs <128,4> 36 ms).  Wide lanes amortise the per-step
    // overhead and leave sleeping warps' issue slots to the busy ones; narrow lanes widen the wavefront.
    int geo = 0;
    if (!traceback) {
        const long long resident = (long long)ctx->sm_count * 4 * WPB;
        if ((long long)n / 256 * 5 >= resident * 4)                    // from ~485 kbp (600 kbp: 332 ms vs 357 with <128,8>):
            geo = ((long long)m / 256 >= resident) ? 7 : 6;            // <256,24> when there are row blocks to spare (1 Mbp: 616 vs 632 ms), else <128,24>
        else geo = 4;                                                  // <128,4>
    }
    if (ctx->opt.long_geometry >= 0 && !traceback) geo = ctx->opt.long_geometry;
    auto launch = [&](auto kern, int RRv, int KKv) -> int {
        int per_sm = 0;
        PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WPB * 32, 0));
        if (ctx->opt.long_ctas_per_sm > 0) per_sm = std::max(1, std::min(per_sm, ctx->opt.long_ctas_per_sm));
        else if (per_sm > 4) per_sm = 4;
        const int NBv = (m + RRv - 1) / RRv;
        int grid = std::min((NBv + WPB - 1) / WPB, per_sm * ctx->sm_count);
        if (grid < 1) grid = 1;
        J.mul8 = key_mult(KKv);
        kern<<<grid, WPB * 32, 0, st>>>(J);
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
        return PSA_OK;
    };
    int lrc;
    if (mode == PSA_LOCAL) {
        if (geo == 1) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 256, 8>, 256, 8);
        else if (geo == 2) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 128, 16>, 128, 16);
        else if (geo == 3) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 256, 16>, 256, 16);
        else if (geo == 4) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 128, 4>, 128, 4);
        else if (geo == 6) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 128, 24>, 128, 24);
        else if (geo == 7) lrc = launch(psa_long_single_kernel<PSA_LOCAL, 256, 24>, 256, 24);
        else lrc = launch(psa_long_single_kernel<PSA_LOCAL, 128, 8>, 128, 8);
    } else {
        if (geo == 1) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 256, 8>, 256, 8);
        else if (geo == 2) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 128, 16>, 128, 16);
        else if (geo == 3) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 256, 16>, 256, 16);
        else if (geo == 4) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 128, 4>, 128, 4);
        else if (geo == 6) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 128, 24>, 128, 24);
        else if (geo == 7) lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 256, 24>, 256, 24);
        else lrc = launch(psa_long_single_kernel<PSA_GLOBAL, 128, 8>, 128, 8);
    }
    if (lrc) return lrc;
    TbArgs T{J, d_item, traceback ? d_ops : nullptr, use_band ? (uint32_t*)(d + o_band) : nullptr};
    if (use_band) {
        const int units = NB * BAND_TILES;
        if (mode == PSA_LOCAL) psa_long_band_kernel<PSA_LOCAL><<<(units + BAND_WPB - 1) / BAND_WPB, BAND_WPB * 32, 0, st>>>(T);
        else psa_long_band_kernel<PSA_GLOBAL><<<(units + BAND_WPB - 1) / BAND_WPB, BAND_WPB * 32, 0, st>>>(T);
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
    }
    if (mode == PSA_LOCAL) psa_long_tb_kernel<PSA_LOCAL><<<1, 32, 0, st>>>(T);
    else psa_long_tb_kernel<PSA_GLOBAL><<<1, 32, 0, st>>>(T);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 1;
    return PSA_OK;
}

// Batch of long pairs, score (+ end cell) only.  Scratch layout: [per-warp hbuf rows | ticket].
static const void* long_batch_kernel_for(int mode, int max_n, int* lane_cols) {
    *lane_cols = max_n >= 1024 ? 16 : 8;
    if (mode == PSA_LOCAL) return *lane_cols == 16 ? (const void*)psa_long_batch_kernel<PSA_LOCAL, 16> : (const void*)psa_long_batch_kernel<PSA_LOCAL, 8>;
    return *lane_cols == 16 ? (const void*)psa_long_batch_kernel<PSA_GLOBAL, 16> : (const void*)psa_long_batch_kernel<PSA_GLOBAL, 8>;
}

static int long_batch_grid(psa_ctx* ctx, long long n_pairs, const void* kern, int* grid) {
    int per_sm = 0;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WPB * 32, 0));
    if (per_sm > 4) per_sm = 4;
    const long long want = (n_pairs + WPB - 1) / WPB;
    *grid = (int)std::min<long long>(want, (long long)per_sm * ctx->sm_count);
    if (*grid < 1) *grid = 1;
    return PSA_OK;
}

size_t psa_long_batch_scratch_bytes(psa_ctx* ctx, long long n_pairs, int max_n) {
    const size_t warp_stride = up256((size_t)(max_n + 1) * 4) / 4 * 2;
    const size_t max_grid = (size_t)4 * ctx->sm_count;
    return max_grid * WPB * warp_stride * 4 + 256;
}

int psa_launch_long_batch_at(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode,
                             const uint8_t* d_flags, uint8_t* scratch, cudaStream_t st) {
    if (max_m >= 0x1FFFFF || max_n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    int grid = 1, lane_cols = 8;
    const void* kern = long_batch_kernel_for(mode, max_n, &lane_cols);
    int rc = long_batch_grid(ctx, args.n_pairs, kern, &grid);
    if (rc) return rc;
    const size_t warp_stride = up256((size_t)(max_n + 1) * 4) / 4 * 2;       // ints: H row + F row
    const size_t hb = (size_t)4 * ctx->sm_count * WPB * warp_stride * 4;
    PSA_CUDA_OK(ctx, cudaMemsetAsync(scratch + hb, 0, 256, st));
    LongBatch Bt{args, (int*)scratch, (long long)warp_stride, (int*)(scratch + hb), d_flags, key_mult(lane_cols)};
    void* kargs[] = {&Bt};
    PSA_CUDA_OK(ctx, cudaLaunchKernel(kern, dim3(grid), dim3(WPB * 32), kargs, 0, st));
    ctx->launches += 1;
    return PSA_OK;
}

int psa_launch_long_batch(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st) {
    int rc = ensure_work(ctx, psa_long_batch_scratch_bytes(ctx, args.n_pairs, max_n));
    if (rc) return rc;
    return psa_launch_long_batch_at(ctx, args, max_m, max_n, mode, nullptr, (uint8_t*)ctx->d_work, st);
}


// ---- batch of long pairs with traceback ----------------------------------------------------------------------------
// The plan depends on n_pairs, max_m and max_n alone (nothing is read back from the device): every pair of a chunk owns a
// checkpoint slot sized for the largest pair, a chunk holds at most one pair per resident fill warp and at most as many
// slots as half of the device memory that is free at call time (plus the context's own work buffer, which it may
// replace).  Chunks run fill -> walk on the caller's stream, one after the other.
namespace {
size_t long_tb_slot_bytes(int max_m, int max_n) {
    const size_t NB = ((size_t)max_m + R - 1) / R, S = ((size_t)max_n + W - 1) / W;
    return 256 + 2 * NB * up256((size_t)(max_n + 1) * 4) + 2 * up256(S * ((size_t)max_m + 1) * 4);
}
int long_tb_fill_ctas(psa_ctx* ctx, int mode, int* ctas) {
    int per_sm = 0;
    const void* kern = mode == PSA_LOCAL ? (const void*)psa_long_batch_tb_fill_kernel<PSA_LOCAL>
                                         : (const void*)psa_long_batch_tb_fill_kernel<PSA_GLOBAL>;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WPB * 32, 0));
    if (per_sm > 4) per_sm = 4;
    *ctas = std::max(1, per_sm * ctx->sm_count);
    return PSA_OK;
}
}  // namespace

int psa_long_batch_tb_chunk(psa_ctx* ctx, long long n_pairs, int max_m, int max_n, int mode, long long* chunk) {
    *chunk = 0;
    int ctas = 1;
    int rc = long_tb_fill_ctas(ctx, mode, &ctas);
    if (rc) return rc;
    size_t free_b = 0, total_b = 0;
    PSA_CUDA_OK(ctx, cudaMemGetInfo(&free_b, &total_b));
    const size_t budget = (free_b + ctx->d_work_bytes) / 2;
    const size_t slot = long_tb_slot_bytes(max_m, max_n);
    long long c = std::min<long long>(n_pairs, (long long)ctas * WPB);
    c = std::min<long long>(c, (long long)((budget > 256 ? budget - 256 : 0) / slot));
    if (ctx->opt.long_tb_chunk > 0) c = std::min<long long>(c, ctx->opt.long_tb_chunk);
    *chunk = std::max(0LL, c);
    return PSA_OK;
}

int psa_launch_long_batch_tb(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, cudaStream_t st) {
    if (max_m >= 0x1FFFFF || max_n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    long long chunk = 0;
    int rc = psa_long_batch_tb_chunk(ctx, args.n_pairs, max_m, max_n, mode, &chunk);
    if (rc) return rc;
    if (chunk < 1) chunk = 1;          // one slot over the budget: try it anyway (the per-pair path needs the same checkpoints)
    int ctas = 1;
    rc = long_tb_fill_ctas(ctx, mode, &ctas);
    if (rc) return rc;
    const size_t slot = long_tb_slot_bytes(max_m, max_n);
    rc = ensure_work(ctx, 256 + (size_t)chunk * slot);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_work;
    for (long long p0 = 0; p0 < args.n_pairs; p0 += chunk) {
        const long long cnt = std::min(chunk, args.n_pairs - p0);
        LongBatchTb Bt{args, p0, cnt, d + 256, (long long)slot, (int*)d};
        PSA_CUDA_OK(ctx, cudaMemsetAsync(d, 0, 256, st));
        const int fill_grid = (int)std::min<long long>((cnt + WPB - 1) / WPB, ctas);
        const int walk_grid = (int)((cnt + WALK_WPB - 1) / WALK_WPB);
        if (mode == PSA_LOCAL) {
            psa_long_batch_tb_fill_kernel<PSA_LOCAL><<<fill_grid, WPB * 32, 0, st>>>(Bt);
            psa_long_batch_tb_walk_kernel<PSA_LOCAL><<<walk_grid, WALK_WPB * 32, 0, st>>>(Bt);
        } else {
            psa_long_batch_tb_fill_kernel<PSA_GLOBAL><<<fill_grid, WPB * 32, 0, st>>>(Bt);
            psa_long_batch_tb_walk_kernel<PSA_GLOBAL><<<walk_grid, WALK_WPB * 32, 0, st>>>(Bt);
        }
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 2;
    }
    return PSA_OK;
}

// ---- banded batches ------------------------------------------------------------------------------------------------
// Every pair runs on the banded tile kernels, one warp per pair, whatever its length.  Score only: one launch, a
// recycled boundary row per resident warp.  Traceback: chunks of fill -> walk as psa_launch_long_batch_tb, with slots
// sized by the band: row block rb computes s_hi - s_lo + 1 <= (its band's column span) / W + 2 tiles, and the spans
// summed over the NB row blocks are at most n + 2*bw*NB (c(i) rises by n over the matrix), so a pair of at most
// max_m x max_n holds at most min(NB*S, (max_n + 2*bw*NB)/W + 2*NB) tiles -- a bound that needs no lengths.
namespace {
size_t banded_slot_bytes(int max_m, int max_n, int bw) {
    const long long NB = ((long long)max_m + R - 1) / R, S = ((long long)max_n + W - 1) / W;
    const long long tiles = std::min(NB * S, ((long long)max_n + 2LL * bw * NB) / W + 2 * NB);
    return 256 + up256((size_t)NB * 8) + (size_t)tiles * REC * 4;
}
}  // namespace

// guide (device arrays) selects the guided kernels: each pair's band follows its anchor chain.  The slot bound holds for
// every valid chain too: a chain's rows are monotone (cmin(i + 1) >= cmax(i)), so the row blocks' spans still sum to at
// most n + 2*bw*NB.
int psa_launch_banded(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, int band, bool traceback,
                      cudaStream_t st, const psa_guide* guide) {
    if (max_m >= 0x1FFFFF || max_n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    const int bw = (int)std::min<long long>(band, (long long)max_m + max_n);     // wider bands admit the same cells
    const bool local = mode == PSA_LOCAL;
    ChainGuide G{guide ? guide->anchors : nullptr, guide ? guide->off : nullptr, guide ? guide->n : nullptr};
    if (!traceback) {
        const void* kern = guide ? (local ? (const void*)psa_guided_batch_kernel<PSA_LOCAL> : (const void*)psa_guided_batch_kernel<PSA_GLOBAL>)
                                 : (local ? (const void*)psa_banded_batch_kernel<PSA_LOCAL> : (const void*)psa_banded_batch_kernel<PSA_GLOBAL>);
        int grid = 1;
        int rc = long_batch_grid(ctx, args.n_pairs, kern, &grid);
        if (rc) return rc;
        const size_t warp_stride = up256((size_t)(max_n + 1) * 4) / 4 * 2;       // ints: H row + F row
        const size_t hb = (size_t)grid * WPB * warp_stride * 4;
        rc = ensure_work(ctx, hb + 256);
        if (rc) return rc;
        uint8_t* d = (uint8_t*)ctx->d_work;
        PSA_CUDA_OK(ctx, cudaMemsetAsync(d + hb, 0, 256, st));
        BandedBatch Bt{args, (int*)d, (long long)warp_stride, (int*)(d + hb), bw};
        void* kargs[] = {&Bt, &G};
        PSA_CUDA_OK(ctx, cudaLaunchKernel(kern, dim3(grid), dim3(WPB * 32), kargs, 0, st));
        ctx->launches += 1;
        return PSA_OK;
    }
    int per_sm = 0;
    const void* fill = guide ? (local ? (const void*)psa_guided_tb_fill_kernel<PSA_LOCAL> : (const void*)psa_guided_tb_fill_kernel<PSA_GLOBAL>)
                             : (local ? (const void*)psa_banded_tb_fill_kernel<PSA_LOCAL> : (const void*)psa_banded_tb_fill_kernel<PSA_GLOBAL>);
    const void* walk = guide ? (local ? (const void*)psa_guided_tb_walk_kernel<PSA_LOCAL> : (const void*)psa_guided_tb_walk_kernel<PSA_GLOBAL>)
                             : (local ? (const void*)psa_banded_tb_walk_kernel<PSA_LOCAL> : (const void*)psa_banded_tb_walk_kernel<PSA_GLOBAL>);
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fill, WPB * 32, 0));
    const long long ctas = std::max(1, std::min(per_sm, 4) * ctx->sm_count);
    size_t free_b = 0, total_b = 0;
    PSA_CUDA_OK(ctx, cudaMemGetInfo(&free_b, &total_b));
    const size_t budget = (free_b + ctx->d_work_bytes) / 2;
    const size_t slot = banded_slot_bytes(max_m, max_n, bw);
    long long chunk = std::min<long long>(args.n_pairs, ctas * WPB);
    chunk = std::min<long long>(chunk, (long long)((budget > 256 ? budget - 256 : 0) / slot));
    if (ctx->opt.long_tb_chunk > 0) chunk = std::min<long long>(chunk, ctx->opt.long_tb_chunk);
    chunk = std::max(1LL, chunk);          // one slot over the budget: try it anyway
    int rc = ensure_work(ctx, 256 + (size_t)chunk * slot);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_work;
    for (long long p0 = 0; p0 < args.n_pairs; p0 += chunk) {
        const long long cnt = std::min(chunk, args.n_pairs - p0);
        BandedTb Bt{args, p0, cnt, d + 256, (long long)slot, (int*)d, bw};
        PSA_CUDA_OK(ctx, cudaMemsetAsync(d, 0, 256, st));
        const int fill_grid = (int)std::min<long long>((cnt + WPB - 1) / WPB, ctas);
        const int walk_grid = (int)((cnt + WALK_WPB - 1) / WALK_WPB);
        void* kargs[] = {&Bt, &G};
        PSA_CUDA_OK(ctx, cudaLaunchKernel(fill, dim3(fill_grid), dim3(WPB * 32), kargs, 0, st));
        PSA_CUDA_OK(ctx, cudaLaunchKernel(walk, dim3(walk_grid), dim3(WALK_WPB * 32), kargs, 0, st));
        ctx->launches += 2;
    }
    return PSA_OK;
}

// ---- one banded pair over the whole GPU ----------------------------------------------------------------------------
// Planned from (m, n, band, mode, traceback) alone -- and, for a guided pair, its chain, which the host holds.  Launches
// (include/psa.h): score only 2 (fill, record); traceback 2 + 2 * windows (tile_base scan, fill, then per window of row
// blocks the code recompute and the walk).
namespace {
constexpr size_t kBandedCodeBytes = (size_t)256 << 20;      // window code buffer (16 KiB per tile)

// Tiles of width WW one row block of a banded pair can hold: its band rows span at most 2*bw + (R-1)*n/m + 1 columns.
long long banded_pair_tpr(int m, int n, int bw, int WW) {
    const long long S = ((long long)n + WW - 1) / WW;
    return std::min(S, (2LL * bw + (long long)R * n / m + 2) / WW + 2);
}

long long rows_per_window(long long NB, long long tpr) {
    return std::min(NB, std::max(1LL, (long long)(kBandedCodeBytes / ((size_t)tpr * R * 32 * 4))));
}

// The plan's band-dependent numbers: tiles per row block at the walk's width W and at the score-only width 32*KK, and
// the column span that picks KK.
struct PairPlan { long long span, tpr_w, tpr16, tpr4; };

PairPlan pair_plan(const Band& B) {
    return {2LL * B.bw + (long long)R * B.n / B.m, banded_pair_tpr(B.m, B.n, B.bw, W), banded_pair_tpr(B.m, B.n, B.bw, 512),
            banded_pair_tpr(B.m, B.n, B.bw, 128)};
}

// A chain's plan is exact: the largest tile count and column span over its row blocks.  The empty chain plans as the
// diagonal band, so that both take the same launches.
PairPlan pair_plan(const ChainBand& B) {
    if (B.K == 0) return pair_plan(Band{B.m, B.n, B.bw});
    PairPlan p{0, 0, 0, 0};
    for (int i0 = 0; i0 < B.m; i0 += R) {
        const int nrows = std::min(R, B.m - i0);
        p.span = std::max(p.span, (long long)B.hi(i0 + nrows) - B.lo(i0 + 1));
        p.tpr_w = std::max(p.tpr_w, (long long)B.s_hi(i0, nrows, W) - B.s_lo(i0, W) + 1);
        p.tpr16 = std::max(p.tpr16, (long long)B.s_hi(i0, nrows, 512) - B.s_lo(i0, 512) + 1);
        p.tpr4 = std::max(p.tpr4, (long long)B.s_hi(i0, nrows, 128) - B.s_lo(i0, 128) + 1);
    }
    return p;
}

// The kernels of one band type: the diagonal band's, or the chain's.
template <class BandT> struct PairKernels;
template <> struct PairKernels<Band> {
    using Fill = BandedPair;
    using Tb = BandedPairTb;
    template <int MODE, int KK, bool TB> static const void* fill() { return (const void*)psa_banded_pair_fill_kernel<MODE, KK, TB>; }
    template <int MODE> static const void* codes() { return (const void*)psa_banded_pair_codes_kernel<MODE>; }
    template <int MODE> static const void* walk() { return (const void*)psa_banded_pair_walk_kernel<MODE>; }
    static const void* tile_base() { return (const void*)psa_banded_tile_base_kernel; }
};
template <> struct PairKernels<ChainBand> {
    using Fill = GuidedPair;
    using Tb = GuidedPairTb;
    template <int MODE, int KK, bool TB> static const void* fill() { return (const void*)psa_guided_pair_fill_kernel<MODE, KK, TB>; }
    template <int MODE> static const void* codes() { return (const void*)psa_guided_pair_codes_kernel<MODE>; }
    template <int MODE> static const void* walk() { return (const void*)psa_guided_pair_walk_kernel<MODE>; }
    static const void* tile_base() { return (const void*)psa_guided_tile_base_kernel; }
};

template <class BandT>
int launch_banded_pair(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h, const BandT& band,
                       const PairPlan& plan, bool traceback, psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st) {
    using Ker = PairKernels<BandT>;
    const int bw = band.bw;
    const bool local = mode == PSA_LOCAL;
    const long long NB = ((long long)m + R - 1) / R;
    const long long resident = (long long)ctx->sm_count * 4 * WPB;
    // Score-only lane width: about (band span)/W row blocks run at once, so narrow <128, 4> tiles (W = 128) keep 4x as many
    // warps busy as <128, 16> ones; the wider lanes (less overhead per cell) only pay once the span gives even them
    // half of the resident warps, i.e. from a span of 256 columns per resident warp.
    const int KK = traceback ? K : (plan.span / 512 >= resident / 2 ? 16 : 4);
    const long long tpr = traceback ? plan.tpr_w : (KK == 16 ? plan.tpr16 : plan.tpr4);
    // memory: [misc 256: ticket | best @8 | corner @16 | walk state @64] [progress NB ints] then
    //   score only: the recycled H and F rows;  traceback: [tile_base NB x 8 B] [records, banded_slot_bytes' bound] [codes]
    const size_t row = up256((size_t)(n + 1) * 4);
    const size_t o_pr = 256, o_body = o_pr + up256((size_t)NB * 4);
    size_t ck = 0, codes = 0, total = o_body + 2 * row;
    long long rpw = 0;
    if (traceback) {
        ck = banded_slot_bytes(m, n, bw) - 256;              // tile_base + records
        rpw = rows_per_window(NB, tpr);
        codes = (size_t)rpw * tpr * R * 32 * 4;
        total = o_body + ck + codes;
        size_t free_b = 0, total_b = 0;
        PSA_CUDA_OK(ctx, cudaMemGetInfo(&free_b, &total_b));
        const size_t budget = (free_b + ctx->d_work_bytes) / 2;
        if (total > budget)
            return psa_fail(ctx, PSA_ERR_NOMEM, "banded traceback needs " + std::to_string(total >> 20) + " MiB of checkpoints and codes, more than half of the free device memory (" + std::to_string(budget >> 20) + " MiB)");
    }
    int rc = ensure_work(ctx, total);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_work;
    PSA_CUDA_OK(ctx, cudaMemsetAsync(d, 0, o_body, st));
    typename Ker::Fill P;
    LongJob& J = P.J;
    J.a = d_a; J.b = d_b; J.m = m; J.n = n; J.g = g; J.h = h; J.mul8 = key_mult(KK);
    J.hbufH = traceback ? nullptr : (int*)(d + o_body); J.hbufF = traceback ? nullptr : (int*)(d + o_body + row); J.hb_stride = 0;
    J.ckvH = nullptr; J.ckvE = nullptr;
    J.progress = (int*)(d + o_pr); J.ticket = (int*)d;
    J.best = (unsigned long long*)(d + 8); J.corner = (int*)(d + 16);
    J.col0 = 0; J.n_total = n; J.row_off = 0; J.start_type = -1; J.end_type = -1;
    P.bk.B = band;
    P.bk.tile_base = traceback ? (long long*)(d + o_body) : nullptr;
    P.bk.rec = traceback ? (int*)(d + o_body + up256((size_t)NB * 8)) : nullptr;
    if (traceback) {
        void* targs[] = {&P.bk.B, &P.bk.tile_base};
        PSA_CUDA_OK(ctx, cudaLaunchKernel(Ker::tile_base(), dim3(1), dim3(1024), targs, 0, st));
        ctx->launches += 1;
    }
    const void* fill;
    if (traceback) fill = local ? Ker::template fill<PSA_LOCAL, K, true>() : Ker::template fill<PSA_GLOBAL, K, true>();
    else if (KK == 16) fill = local ? Ker::template fill<PSA_LOCAL, 16, false>() : Ker::template fill<PSA_GLOBAL, 16, false>();
    else fill = local ? Ker::template fill<PSA_LOCAL, 4, false>() : Ker::template fill<PSA_GLOBAL, 4, false>();
    int per_sm = 0;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fill, WPB * 32, 0));
    if (ctx->opt.long_ctas_per_sm > 0) per_sm = std::max(1, std::min(per_sm, ctx->opt.long_ctas_per_sm));
    else if (per_sm > 4) per_sm = 4;
    // about tpr row blocks are in flight at once; twice as many warps keep the next ones waiting at their first strip
    const long long warps = std::min(NB, 2 * tpr + 4);
    const int grid = (int)std::max(1LL, std::min((warps + WPB - 1) / WPB, (long long)per_sm * ctx->sm_count));
    void* fargs[] = {&P};
    PSA_CUDA_OK(ctx, cudaLaunchKernel(fill, dim3(grid), dim3(WPB * 32), fargs, 0, st));
    ctx->launches += 1;
    typename Ker::Tb T{J, P.bk, traceback ? (uint32_t*)(d + o_body + ck) : nullptr, (int)tpr, 0, (int)NB,
                        (BandedWalk*)(d + 64), d_item, traceback ? d_ops : nullptr};
    void* wargs[] = {&T};
    const void* codes_k = local ? Ker::template codes<PSA_LOCAL>() : Ker::template codes<PSA_GLOBAL>();
    const void* walk_k = local ? Ker::template walk<PSA_LOCAL>() : Ker::template walk<PSA_GLOBAL>();
    if (!traceback) {
        PSA_CUDA_OK(ctx, cudaLaunchKernel(walk_k, dim3(1), dim3(32), wargs, 0, st));
        ctx->launches += 1;
        return PSA_OK;
    }
    for (long long hi = NB; hi > 0; hi -= rpw) {
        T.rb_hi = (int)hi; T.rb_lo = (int)std::max(0LL, hi - rpw);
        const long long units = (long long)(T.rb_hi - T.rb_lo) * tpr;
        const unsigned blocks = (unsigned)((units + CODES_WPB - 1) / CODES_WPB);
        PSA_CUDA_OK(ctx, cudaLaunchKernel(codes_k, dim3(blocks), dim3(CODES_WPB * 32), wargs, 0, st));
        PSA_CUDA_OK(ctx, cudaLaunchKernel(walk_k, dim3(1), dim3(32), wargs, 0, st));
        ctx->launches += 2;
    }
    return PSA_OK;
}
}  // namespace

int psa_launch_banded_pair(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h, int band,
                           bool traceback, psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st) {
    if (m <= 0 || n <= 0) return psa_fail(ctx, PSA_ERR_ARG, "banded pair path needs m, n >= 1");
    if (m >= 0x1FFFFF || n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    const Band B{m, n, (int)std::min<long long>(band, (long long)m + n)};
    return launch_banded_pair(ctx, d_a, d_b, m, n, mode, g, h, B, pair_plan(B), traceback, d_item, d_ops, st);
}

int psa_launch_guided_pair(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int mode, int g, int h, int band,
                           const psa_anchor* h_anchors, const psa_anchor* d_anchors, int n_anchors, bool traceback,
                           psa_batch_item* d_item, uint32_t* d_ops, cudaStream_t st) {
    if (m <= 0 || n <= 0) return psa_fail(ctx, PSA_ERR_ARG, "guided pair path needs m, n >= 1");
    if (m >= 0x1FFFFF || n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    const int bw = (int)std::min<long long>(band, (long long)m + n);
    const PairPlan plan = pair_plan(ChainBand{m, n, bw, h_anchors, n_anchors});
    return launch_banded_pair(ctx, d_a, d_b, m, n, mode, g, h, ChainBand{m, n, bw, d_anchors, n_anchors}, plan, traceback, d_item,
                              d_ops, st);
}

// ---- partition finder (SURVEY 8 f-3; the role of sequence_alignment/partial.cpp:81-163) ---------------------------
// Forward sweep of (A, B) and reverse sweep of (reverse A, reverse B), both score-only fills that keep the bottom row
// (H = max(T1,T2,T3) and F = T3 per column) of every 128-row block; the reverse sweep's first block is m mod 128 rows
// high, so that its block boundaries fall on the same matrix rows as the forward sweep's.  For a special row i the
// best crossing is  max_j max( Hf[i][j] + Hr[i][j],  Ff[i][j] + Fr[i][j] + h )  -- the path passes the node (i, j)
// between two operations, or a vertical gap spans the row (its opening penalty is charged by both sweeps, hence + h;
// partial.cpp:101-105).  Smallest j wins, node before gap (partial.cpp:108 uses the same >= priority).
namespace {

struct SweepRows { int* H; int* F; long long stride; int nb; };

// One checkpointed score-only fill into the region of ctx->d_work starting at byte `base`; returns the rows.
int sweep_rows(psa_ctx* ctx, uint8_t* region, size_t region_bytes, const uint8_t* d_a, const uint8_t* d_b, int m, int n, int g, int h,
               int row_off, int* d_corner, cudaStream_t st, SweepRows* out) {
    const int NB = row_off ? 1 + std::max(0, m - row_off + R - 1) / R : (m + R - 1) / R;
    const size_t row = up256((size_t)(n + 1) * 4);
    size_t o = 0;
    const size_t o_hH = o; o += row * NB;
    const size_t o_hF = o; o += row * NB;
    const size_t o_pr = o; o += up256((size_t)NB * 4);
    const size_t o_misc = o; o += 256;
    if (o > region_bytes) return psa_fail(ctx, PSA_ERR_NOMEM, "partition sweep region too small");
    PSA_CUDA_OK(ctx, cudaMemsetAsync(region + o_pr, 0, (o_misc + 256) - o_pr, st));
    LongJob J;
    J.a = d_a; J.b = d_b; J.m = m; J.n = n; J.g = g; J.h = h; J.mul8 = key_mult(K);
    J.hbufH = (int*)(region + o_hH); J.hbufF = (int*)(region + o_hF); J.hb_stride = (long long)(row / 4);
    J.ckvH = nullptr; J.ckvE = nullptr;
    J.progress = (int*)(region + o_pr); J.ticket = (int*)(region + o_misc);
    J.best = (unsigned long long*)(region + o_misc + 8); J.corner = d_corner;
    J.col0 = 0; J.n_total = n; J.row_off = row_off; J.start_type = -1; J.end_type = -1;
    int per_sm = 0;
    PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, psa_long_single_kernel<PSA_GLOBAL, R, K, true>, WPB * 32, 0));
    if (per_sm > 4) per_sm = 4;
    int grid = std::min((NB + WPB - 1) / WPB, per_sm * ctx->sm_count);
    if (grid < 1) grid = 1;
    if (row_off) psa_long_single_kernel<PSA_GLOBAL, R, K, true><<<grid, WPB * 32, 0, st>>>(J);
    else psa_long_single_kernel<PSA_GLOBAL, R, K, false><<<grid, WPB * 32, 0, st>>>(J);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 1;
    out->H = J.hbufH; out->F = J.hbufF; out->stride = J.hb_stride; out->nb = NB;
    return PSA_OK;
}

// one CTA per special row: (i, j, type) of the best crossing
__global__ void __launch_bounds__(256) psa_crossing_kernel(SweepRows fwd, SweepRows rev, int m, int n, int g, int h, int row_off_rev,
                                                           const int* rows, int n_rows, int* out /* [n_rows][4]: i, j, type, value */) {
    __shared__ long long s_best[256];
    const int q = blockIdx.x;
    if (q >= n_rows) return;
    const int i = rows[q];                              // 0 < i < m, a multiple of R
    const int* Hf = fwd.H + (long long)(i / R - 1) * fwd.stride;
    const int* Ff = fwd.F + (long long)(i / R - 1) * fwd.stride;
    const int ir = m - i;                               // the same matrix row as the reverse sweep numbers it
    const int rbr = row_off_rev ? (ir - row_off_rev) / R : ir / R - 1;
    const int* Hr = rev.H + (long long)rbr * rev.stride;
    const int* Fr = rev.F + (long long)rbr * rev.stride;
    long long best = LLONG_MIN;
    for (int j = threadIdx.x; j <= n; j += blockDim.x) {
        const int jr = n - j;
        // column 0 of either sweep: only the vertical border gap reaches it (T3[i][0] = -h - g*i, cpp:290-292)
        const int hf = j > 0 ? Hf[j] : -h - g * i, ff = j > 0 ? Ff[j] : -h - g * i;
        const int hr = jr > 0 ? Hr[jr] : -h - g * ir, fr = jr > 0 ? Fr[jr] : -h - g * ir;
        const long long v1 = (long long)hf + hr, v3 = (long long)ff + fr + h;
        const long long v = v1 >= v3 ? v1 : v3;
        const int type = v1 >= v3 ? 1 : 3;
        // order: value desc, then j asc, then node (1) before gap (3)
        const long long key = (v << 24) | ((long long)(0x3FFFFF - j) << 2) | (type == 1 ? 1 : 0);
        best = key > best ? key : best;
    }
    s_best[threadIdx.x] = best;
    __syncthreads();
    for (int off = 128; off >= 1; off >>= 1) {
        if ((int)threadIdx.x < off) s_best[threadIdx.x] = s_best[threadIdx.x] > s_best[threadIdx.x + off] ? s_best[threadIdx.x] : s_best[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const long long key = s_best[0];
        out[4 * q + 0] = i;
        out[4 * q + 1] = 0x3FFFFF - (int)((key >> 2) & 0x3FFFFF);
        out[4 * q + 2] = (key & 1) ? 1 : 3;
        out[4 * q + 3] = (int)(key >> 24);
    }
}

}  // namespace

// Crossing points of an optimal global alignment on up to max_rows special rows (multiples of 128, evenly spread).
// d_a / d_b and their reversals resident on the device.  h_points[k] = {i, j, type, optimal score}.
int psa_find_crossings(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, const uint8_t* d_ar, const uint8_t* d_br, int m, int n,
                       int g, int h, int max_rows, int* h_points, int* n_points, cudaStream_t st) {
    *n_points = 0;
    const int avail = (m - 1) / R;                      // rows R, 2R, ... < m
    const int want = std::min(max_rows, avail);
    if (want <= 0) return PSA_OK;
    if (m >= 0x1FFFFF || n >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    const int row_off_rev = m % R;                      // 0: the regular grid already lines up
    const int NBf = (m + R - 1) / R, NBr = row_off_rev ? 1 + (m - row_off_rev + R - 1) / R : NBf;
    const size_t row = up256((size_t)(n + 1) * 4);
    const size_t reg_f = 2 * row * NBf + up256((size_t)NBf * 4) + 512, reg_r = 2 * row * NBr + up256((size_t)NBr * 4) + 512;
    const size_t o_f = 0, o_r = up256(reg_f), o_rows = o_r + up256(reg_r), o_out = o_rows + up256((size_t)want * 4);
    const size_t total = o_out + up256((size_t)want * 16) + 256;
    int rc = ensure_work(ctx, total);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_work;
    SweepRows F, Rv;
    int* d_corner = (int*)(d + o_out + up256((size_t)want * 16));
    rc = sweep_rows(ctx, d + o_f, reg_f, d_a, d_b, m, n, g, h, 0, d_corner, st, &F);
    if (rc) return rc;
    rc = sweep_rows(ctx, d + o_r, reg_r, d_ar, d_br, m, n, g, h, row_off_rev, d_corner + 4, st, &Rv);
    if (rc) return rc;
    std::vector<int> rows(want);
    for (int k = 0; k < want; ++k) {
        int idx = (int)((long long)(k + 1) * (avail + 1) / (want + 1));     // 1 .. avail, evenly spread
        idx = std::max(1, std::min(avail, idx));
        rows[k] = idx * R;
    }
    rows.erase(std::unique(rows.begin(), rows.end()), rows.end());
    const int nr = (int)rows.size();
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(d + o_rows, rows.data(), (size_t)nr * 4, cudaMemcpyHostToDevice, st));
    psa_crossing_kernel<<<nr, 256, 0, st>>>(F, Rv, m, n, g, h, row_off_rev, (const int*)(d + o_rows), nr, (int*)(d + o_out));
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 1;
    PSA_CUDA_OK(ctx, cudaMemcpyAsync(h_points, d + o_out, (size_t)nr * 16, cudaMemcpyDeviceToHost, st));
    PSA_CUDA_OK(ctx, cudaStreamSynchronize(st));
    *n_points = nr;
    return PSA_OK;
}
