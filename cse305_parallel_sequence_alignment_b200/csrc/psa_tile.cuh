// psa_tile.cuh -- the int32 tile engine shared by the long-pair kernels.
//
// A tile is R rows x 32*K columns of one DP matrix, swept by ONE warp as a skewed wavefront:
// lane t owns K consecutive columns and at step s works on tile row s - t; the (H, E) of the
// column to its left arrive from lane t-1 by shuffle.  Around the tile:
//     top boundary   : H and F (= T3) of the row above, one value per column, held in the lane's
//                      column registers when the sweep starts (and the bottom boundary when it ends)
//     left boundary  : H and E (= T2) of the column to the left, one value per tile row, read by
//                      lane 0 from a shared-memory array (filled from the border formula, from
//                      the previous tile of the same row block, or from a checkpoint column)
//     right boundary : written by lane 31 to a shared-memory array, for the next tile / checkpoint
// Recurrence and 4-bit direction codes exactly as in psa_short.cu (reference:
// subproblem_alignment.cpp:229-249 for the fill, :147-169 for the predecessor order).
#pragma once
#include "psa_result.cuh"

namespace psa_tile {

template <int K>
struct Cols {
    int H[K];
    int F[K];
    int b[K];     // column characters (256 = padding, never matches)
};

struct Track {    // local mode: best T1 seen by this lane and its first cell (row-major order)
    int best, bi, bj;
};

// Sweeps `nrows` rows (global rows i0+1 .. i0+nrows) of the tile whose first column is global
// column c0+1 for this lane (c0 = tile_col0 + lane*K).  n = total columns of the pair.
//   hd        in: H[i0][c0] (value diagonal to the lane's first cell); meaningful for every lane
//   lbH/lbE   left boundary of the tile (index r = 0..nrows-1 -> row i0+1+r); read by lane 0
//   rbH/rbE   right boundary out (lane 31), may be null
//   sA        row characters of the tile rows (index r)
//   dirs      shared memory, 32 words per tile row, or null
//   cap_*     global mode: receives T1/T2/T3 of cell (m, n) when the tile contains it
//   BANDED    a band edge cuts the tile: cell (i, j) of tile row r exists only for bLo[r] <= j <= bHi[r]; every other
//             cell is forced to the out-of-band value (H = T1 = 0 in local mode, else the sentinel; E = F = sentinel)
template <int K, int MODE, bool DIRS, bool BANDED = false>
__device__ __forceinline__ void sweep(Cols<K>& cs, int hd, const int* lbH, const int* lbE, int* rbH, int* rbE,
                                      const uint8_t* sA, int nrows, int i0, int c0, int m, int n, int g, int h,
                                      uint32_t* dirs, Track& tr, int& cap1, int& cap2, int& cap3,
                                      const int* bLo = nullptr, const int* bHi = nullptr) {
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    const int lane = threadIdx.x & 31;
    const int go = g + h;
    int recv_h = PSA_KNEG, recv_e = PSA_KNEG;
    const int steps = nrows + 31;
    for (int s = 0; s < steps; ++s) {
        const int r = s - lane;
        int hl, el;
        if (lane == 0) {
            const int rr = r < nrows ? (r < 0 ? 0 : r) : nrows - 1;
            hl = lbH[rr]; el = lbE[rr];
        } else { hl = recv_h; el = recv_e; }
        if (r >= 0 && r < nrows) {
            const int i = i0 + 1 + r;
            const int a = sA[r];
            const int hl0 = hl;
            int diag = hd;
            uint32_t word = 0;
            const int klo = BANDED ? bLo[r] - c0 - 1 : 0, khi = BANDED ? bHi[r] - c0 - 1 : 0;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                int t1 = (LOCAL ? imax(diag, 0) : diag) + (a == cs.b[k] ? 1 : 0);
                int e = imax(hl - go, el - g);
                int f = imax(cs.H[k] - go, cs.F[k] - g);
                int H = imax(t1, imax(e, f));
                if (BANDED && (k < klo || k > khi)) { t1 = H = LOCAL ? 0 : PSA_KNEG; e = f = PSA_KNEG; }
                if (DIRS) {
                    int d1 = (t1 == H) ? 1 : (e >= f ? 2 : 3);
                    const int z2 = (d1 == 1) ? (e + h > H) : (e + h >= H);
                    const int e3 = (f + h > H);
                    if (LOCAL && H == 0) d1 = 0;
                    word |= (uint32_t)(d1 | (z2 << 2) | (e3 << 3)) << (4 * k);
                }
                if (LOCAL) {
                    if (t1 > tr.best && c0 + k < n) { tr.best = t1; tr.bi = i; tr.bj = c0 + k + 1; }
                } else {
                    if (i == m && c0 + k + 1 == n) { cap1 = t1; cap2 = e; cap3 = f; }
                }
                diag = cs.H[k]; cs.H[k] = H; cs.F[k] = f; hl = H; el = e;
            }
            hd = hl0;
            if (DIRS) dirs[r * 32 + lane] = word;
            if (rbH != nullptr && lane == 31) { rbH[r] = hl; rbE[r] = el; }
        }
        recv_h = __shfl_up_sync(0xffffffffu, hl, 1);
        recv_e = __shfl_up_sync(0xffffffffu, el, 1);
    }
}

// ---- lean score-only sweep (fill kernels) ----------------------------------------------------
// Same tile, same boundaries as sweep<>, written with the DPX intrinsics, in one of two forms (tf_form(K)):
//
// TF form (the form the systolic kernel uses): every recurrence is ONE VIADDMNMX.  With hg = H - (g+h) of the row
// above, F of the row above unshifted, and TF = max(T1, F) - (g+h),
//     F  = max(F' - g, H' - go)        = viaddmax(ff, -g, hg)
//     TF = max(F - go, T1 - go)        = viaddmax(F, -go, t1g)          t1g = hg_diag + match
//     E  = max(E_left - g, TF_left)    = viaddmax(e, -g, tf)            (h >= 0: H_left - go = max(E_left - go, TF_left))
//     hg = max(E - go, TF)             = viaddmax(e, -go, tf)
// i.e. per cell ISETP + IADD (match) and 4 x VIADDMNMX, ONE instruction per cell on the row's dependency chain, two
// registers of column state.  Lanes hand over (TF, E) of their last column; a tile boundary holds (H, E), and H - go
// can stand in for TF there because it only adds the term E_left - go <= E_left - g to the maximum.
//
// H form: per cell ISETP + IADD, 2 x VIADDMNMX (E, F), VIMNMX3 (H), one subtract (H - (g+h)); three registers of
// column state (H, H - go, F), three instructions per cell on the row chain.  Same ALU instruction count.
//
// Which form a lane width gets was measured, each pair of numbers on one box (the other form loaded as a second
// library, PSA_LIBRARY): 4 columns per lane -- 10 kbp x 10 kbp score-only fill 3.69 ms (H) / 3.07 ms (TF); 8 columns --
// the checkpointed 10 kbp fill + traceback 4.98 (H) / 5.17 (TF); 16 columns -- 4 736 x 5 000^2 batch 66.9 (H) / 59.6
// (TF); 24 columns -- 1 Mbp x 1 Mbp 695 (H) / 785 (TF: its temporaries no longer fit beside the column state in the
// 168 registers that keep three CTAs per SM).
//
// Local mode adds an IMAD key (T1*KM + KM-1-k) and half a VIMNMX3 to find the end cell; the global corner is captured
// in a separate instantiation taken only on the step that owns cell (m, n).  KM = the power of two >= K.
__host__ __device__ constexpr int key_mult(int K) { return K <= 4 ? 4 : (K <= 8 ? 8 : (K <= 16 ? 16 : 32)); }
__host__ __device__ constexpr bool tf_form(int K) { return K <= 4 || K == 16; }

template <int K>
struct ColsS {
    int hg[K];    // H[i-1][j] - (g+h)
    int ff[K];    // F[i-1][j]
    int H[K];     // H form only: H[i-1][j]
    int b[K];
    int ka[K];    // local mode: key addend KM-1-k, or -2^30 for padding columns (j > n); TF form: + (g+h)*KM, its key is
                  // built from T1 - (g+h).  A padding key is then T1*KM - 2^30 < 0.  Without the + (g+h)*KM there,
                  // (T1 - (g+h))*KM - 2^30 wrapped to a large positive key once (g+h)*KM > 2^30 (local mode admits g+h up
                  // to about 2^27): it outranked the real columns of the lane holding column n, and the lane's best was
                  // then dropped as lying past n.
    __device__ __forceinline__ void set_top(int k, int H0, int F0, int go) { hg[k] = H0 - go; ff[k] = F0; if (!tf_form(K)) H[k] = H0; }
    __device__ __forceinline__ int top_H(int k, int go) const { return tf_form(K) ? hg[k] + go : H[k]; }
    __device__ __forceinline__ void set_key_addend(int k, bool real, int go) {
        ka[k] = (real ? key_mult(K) - 1 - k : -(1 << 30)) + (tf_form(K) ? go * key_mult(K) : 0);
    }
};

// BANDED: columns k < klo and k > khi of the lane are outside the band; they leave (H, T1, E, F) = the out-of-band value
// (TF form: hg = TF = H - go, E = F = sentinel).
template <int K, bool LOCAL, bool CAP, bool BANDED = false>
__device__ __forceinline__ void score_step_tf(ColsS<K>& cs, int& tf_io, int& e_io, int diag_hg, int a, int ng, int ngo, int go,
                                              int mul8, int& rowkey, int kcap, int& cap1, int& cap2, int& cap3,
                                              int klo = 0, int khi = 0) {
    int t1g[K], tfn[K];
    // everything that depends only on the row above first (off the E chain)
#pragma unroll
    for (int k = 0; k < K; ++k) {
        t1g[k] = (k == 0 ? diag_hg : cs.hg[k - 1]) + (a == cs.b[k] ? 1 : 0);
        cs.ff[k] = __viaddmax_s32(cs.ff[k], ng, cs.hg[k]);
        tfn[k] = __viaddmax_s32(cs.ff[k], ngo, t1g[k]);
        if (BANDED && (k < klo || k > khi)) { cs.ff[k] = PSA_KNEG; t1g[k] = tfn[k] = (LOCAL ? 0 : PSA_KNEG) - go; }
    }
    int key_prev = 0;
    int e = e_io, tf = tf_io;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        e = __viaddmax_s32(e, ng, tf);
        if (BANDED && (k < klo || k > khi)) e = PSA_KNEG;
        tf = tfn[k];
        const int hgk = __viaddmax_s32(e, ngo, tf);
        if (LOCAL) {
            const int key = t1g[k] * mul8 + cs.ka[k];
            if (k & 1) rowkey = __vimax3_s32(rowkey, key_prev, key);
            key_prev = key;
        }
        if (CAP) { if (k == kcap) { cap1 = t1g[k] + go; cap2 = e; cap3 = cs.ff[k]; } }
        cs.hg[k] = hgk;
    }
    tf_io = tf; e_io = e;
}

template <int K, bool LOCAL, bool CAP>
__device__ __forceinline__ void score_step_h(ColsS<K>& cs, int& hlgo, int& el, int diag, int a, int ng, int go, int mul8,
                                             int& rowkey, int kcap, int& cap1, int& cap2, int& cap3) {
    int key_prev = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int t1 = diag + (a == cs.b[k] ? 1 : 0);
        const int e = __viaddmax_s32(el, ng, hlgo);
        const int f = __viaddmax_s32(cs.ff[k], ng, cs.hg[k]);
        const int H = __vimax3_s32(t1, e, f);
        if (LOCAL) {
            const int key = t1 * mul8 + cs.ka[k];
            if (k & 1) rowkey = __vimax3_s32(rowkey, key_prev, key);
            key_prev = key;
        }
        if (CAP) { if (k == kcap) { cap1 = t1; cap2 = e; cap3 = f; } }
        diag = cs.H[k];
        const int hg = H - go;
        cs.H[k] = H; cs.hg[k] = hg; cs.ff[k] = f; hlgo = hg; el = e;
    }
}

// lbH/lbE, rbH/rbE hold H and E (external format); hd = H[i0][c0].  bestkey/besti: local-mode
// tracker of this lane for this tile (key = T1*KM + KM-1-k, row), folded by the caller.
// BANDED (TF form only): the band of tile row r is columns bLo[r] .. bHi[r], as in sweep<>.
template <int K, int MODE, bool BANDED = false>
__device__ __forceinline__ void sweep_score(ColsS<K>& cs, int hd, const int* lbH, const int* lbE, int* rbH, int* rbE,
                                            const uint8_t* sA, int nrows, int i0, int c0, int m, int n, int g, int h,
                                            int mul8, int& bestkey, int& besti, int& cap1, int& cap2, int& cap3,
                                            const int* bLo = nullptr, const int* bHi = nullptr) {
    static_assert(K % 2 == 0, "the row key folds two cells per VIMNMX3");
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    constexpr bool TF = tf_form(K);
    static_assert(TF || !BANDED, "the band mask is written for the TF form");
    constexpr int KM = key_mult(K);
    const int lane = threadIdx.x & 31;
    const int go = g + h, ng = -g, ngo = -go;
    // handed from lane to lane: (TF, E) in the TF form, (H - go, E) in the H form; both start from (H - go, E) of the tile boundary
    int recv_x = PSA_KNEG, recv_e = PSA_KNEG;
    int diag = TF ? hd - go : hd;             // diagonal of the lane's first cell: H[i-1][c0] (TF form: minus go)
    // which k of this lane owns column n, and is row m in this tile?
    const int kcap = (!LOCAL && i0 + nrows == m && n > c0 && n <= c0 + K) ? (n - 1 - c0) : -1;
    const int steps = nrows + 31;
    for (int s = 0; s < steps; ++s) {
        const int r = s - lane;
        int x, el;
        if (lane == 0) {
            const int rr = r < nrows ? (r < 0 ? 0 : r) : nrows - 1;
            x = lbH[rr] - go; el = lbE[rr];
        } else { x = recv_x; el = recv_e; }
        const bool active = (r >= 0 && r < nrows);
        const bool capstep = !LOCAL && active && kcap >= 0 && r == nrows - 1;
        const bool anycap = LOCAL ? false : __any_sync(0xffffffffu, capstep);
        if (active) {
            const int a = sA[r];
            int rowkey = 0;
            if (TF) {
                const int hg_left = __viaddmax_s32(el, ngo, x);       // H[i][c0] - go: the next row's diagonal
                const int klo = BANDED ? bLo[r] - c0 - 1 : 0, khi = BANDED ? bHi[r] - c0 - 1 : 0;
                if (!anycap) score_step_tf<K, LOCAL, false, BANDED>(cs, x, el, diag, a, ng, ngo, go, mul8, rowkey, -1, cap1, cap2, cap3, klo, khi);
                else score_step_tf<K, LOCAL, true, BANDED>(cs, x, el, diag, a, ng, ngo, go, mul8, rowkey, capstep ? kcap : -1, cap1, cap2, cap3, klo, khi);
                diag = hg_left;
            } else {
                const int hin = x;
                if (!anycap) score_step_h<K, LOCAL, false>(cs, x, el, diag, a, ng, go, mul8, rowkey, -1, cap1, cap2, cap3);
                else score_step_h<K, LOCAL, true>(cs, x, el, diag, a, ng, go, mul8, rowkey, capstep ? kcap : -1, cap1, cap2, cap3);
                diag = hin + go;
            }
            if (LOCAL) { if (rowkey > (bestkey | (KM - 1))) { bestkey = rowkey; besti = i0 + 1 + r; } }
            if (rbH != nullptr && lane == 31) { rbH[r] = cs.hg[K - 1] + go; rbE[r] = el; }
        }
        recv_x = __shfl_up_sync(0xffffffffu, x, 1);
        recv_e = __shfl_up_sync(0xffffffffu, el, 1);
    }
}

}  // namespace psa_tile
