// psa_result.cuh -- the rules every kernel family follows when it turns a fill into a psa_batch_item, and the border
// and traceback rules they share (subproblem_alignment.cpp:112-170, :212-227, :259-292).  Each rule is written once
// here; the parity tests pin them to the reference.
#pragma once
#include "psa_common.cuh"

__device__ __forceinline__ int imax(int a, int b) { return a > b ? a : b; }

// The in-kernel sentinel (and anything that drifted from it) is the ABI's -infinity.  The threshold is -3 * 2^27.
// check_scoring admits span = g(m+n+2) + 2h + m + n < 2^28.  In the full matrix a finite value needs at most three gap
// openings (a start type forces the first gap, an orthogonal gap follows, and the end state needs one more) and at most
// m + n gap columns, so it is >= -(3h + g(m+n)) > -1.5 * span > -3 * 2^27.  A band can force an opening on every row:
// banded global calls are held to check_banded_scoring's g(m+n+2) + h(min(m, n) + 3) + m + n < 2^28 (psa_capi.cu),
// which keeps them >= -2^28.  A value that descends from the sentinel gains at most +1 per diagonal step, so it is
// <= PSA_KNEG + min(m, n) < -2^29 + 2^27 = -3 * 2^27.  The old threshold PSA_KNEG / 2 = -2^28 cut off finite typed
// corners such as -3h + 113 at g = 0, h = 134 217 577.
__device__ __forceinline__ int out_value(int v) { return v < PSA_KNEG / 4 * 3 ? PSA_NEG_INF : v; }

// End state of a global alignment (find_alignment, cpp:112-146): forced by a positive end type, else the first of
// T1, T2 + h', T3 + h' that is >= the others, h' = h only for the matching end type -2 / -3.
__device__ __forceinline__ int end_state(int c1, int c2, int c3, int h, int et) {
    if (et > 0) return et;
    const int e2 = c2 + (et == -2 ? h : 0), e3 = c3 + (et == -3 ? h : 0);
    return (c1 >= e2 && c1 >= e3) ? 1 : ((e2 >= c1 && e2 >= e3) ? 2 : 3);
}

// Local end cell as one 64-bit key for atomicMax / max-reductions: the largest key is the best T1 at the smallest i,
// then the smallest j.  i, j < 2^21 - 1; score > 0 (a key of 0 means "nothing positive").
__device__ __forceinline__ unsigned long long best_key(int score, int i, int j) {
    return ((unsigned long long)(unsigned)score << 42) | ((unsigned long long)(0x1FFFFF - i) << 21) |
           (unsigned long long)(0x1FFFFF - j);
}

__device__ __forceinline__ psa_batch_item local_item(int score, int i, int j) {
    psa_batch_item r;
    r.t1 = score; r.t2 = PSA_NEG_INF; r.t3 = PSA_NEG_INF; r.score = score; r.end_state = 1;
    r.end_i = i; r.end_j = j;
    r.start_i = 0; r.start_j = 0; r.aln_len = 0;
    return r;
}

__device__ __forceinline__ psa_batch_item local_item_from_key(unsigned long long key) {
    const int sc = (int)(key >> 42);
    return local_item(sc, sc > 0 ? 0x1FFFFF - (int)((key >> 21) & 0x1FFFFF) : 0, sc > 0 ? 0x1FFFFF - (int)(key & 0x1FFFFF) : 0);
}

// Global result from T1/T2/T3 of cell (m, n) as the fill left them (sentinel included); the end state is picked
// from those values.
__device__ __forceinline__ psa_batch_item global_item(int c1, int c2, int c3, int m, int n, int h, int et) {
    psa_batch_item r;
    r.t1 = out_value(c1); r.t2 = out_value(c2); r.t3 = out_value(c3); r.score = out_value(imax(c1, imax(c2, c3)));
    r.end_state = end_state(c1, c2, c3, h, et);
    r.end_i = m; r.end_j = n;
    r.start_i = 0; r.start_j = 0; r.aln_len = 0;
    return r;
}

// Global result from a corner captured in .S16x2 registers: half `sh` (0 or 16) of the words T1, T2, T3, each
// biased by `bias` (untyped: the packed kernels serve start / end type -1 only).
__device__ __forceinline__ psa_batch_item packed_corner_item(const uint32_t* c3, int sh, int bias, int m, int n) {
    return global_item((int)((c3[0] >> sh) & 0xffffu) - bias, (int)((c3[1] >> sh) & 0xffffu) - bias,
                       (int)((c3[2] >> sh) & 0xffffu) - bias, m, n, 0, -1);
}

// The 16-byte record of psa_align_batch_packed: score, cells, length and end state of the 40-byte record, the
// coordinates and length narrowed to 16 bits (its reads are at most 512 x 256).
__device__ __forceinline__ psa_packed_item packed_item(const psa_batch_item& it) {
    psa_packed_item o;
    o.score = it.score;
    o.end_i = (uint16_t)it.end_i; o.end_j = (uint16_t)it.end_j;
    o.start_i = (uint16_t)it.start_i; o.start_j = (uint16_t)it.start_j;
    o.aln_len = (uint16_t)it.aln_len; o.end_state = (uint16_t)it.end_state;
    return o;
}

// Border values by start type st (cpp:212-227, :259-292): H = max(T1,T2,T3) of the border cell; on row 0 only T2
// can be finite, on column 0 only T3, besides the (0,0) cell.  -1 is the live case; -2 / -3 continue an open gap
// along row 0 / column 0 (no h on that border); 1, 2, 3 force the first state, which leaves only T1[0][0] (1),
// row 0 (2) or column 0 (3) finite.
// Local mode uses H = 0 on the borders (E, F stay -inf): with T1 = f + max(0, .) every interior T1 is >= 0, so
// H = max(0, H_spec) everywhere and score, end cell and path flags are those of the -inf-border spec (DESIGN.md
// section 3) -- and no explicit 0-floor is needed in the fill.
template <int MODE>
__device__ __forceinline__ int border_row0_H(int j, int g, int h, int st = -1) {   // H[0][j] = T2[0][j]; (0,0): the table st selects
    if (MODE == PSA_LOCAL) return 0;
    if (j == 0) return (st == 2 || st == 3) ? PSA_KNEG : 0;
    if (st == -2) return -g * j;
    if (st == 1 || st == 3) return PSA_KNEG;
    return -h - g * j;
}
template <int MODE>
__device__ __forceinline__ int border_col0_H(int i, int g, int h, int st = -1) {   // H[i][0] = T3[i][0]
    if (MODE == PSA_LOCAL) return 0;
    if (i == 0) return (st == 2 || st == 3) ? PSA_KNEG : 0;
    if (st == -3) return -g * i;
    if (st == 1 || st == 2) return PSA_KNEG;
    return -h - g * i;
}

// Result of a member with m == 0 or n == 0: borders only.
template <int MODE>
__device__ __forceinline__ psa_batch_item empty_item(int m, int n, int g, int h, int st, int et) {
    if (MODE == PSA_LOCAL) return local_item(0, 0, 0);
    int t1 = PSA_NEG_INF, t2 = PSA_NEG_INF, t3 = PSA_NEG_INF;
    if (m == 0 && n == 0) {
        if (st == -1 || st == 1) t1 = 0; else if (st == -2) t2 = 0; else if (st == -3) t3 = 0;
    } else if (m == 0) t2 = out_value(border_row0_H<PSA_GLOBAL>(n, g, h, st));
    else if (n == 0) t3 = out_value(border_col0_H<PSA_GLOBAL>(m, g, h, st));
    return global_item(t1, t2, t3, m, n, h, et);
}

// Traceback decode (cpp:147-169) of the 4-bit code d1 | z2 << 2 | e3 << 3 of the SOURCE cell (0 when the source is
// on the border).  Returns the next state, or 0 when a local alignment stops at this column.
template <int MODE>
__device__ __forceinline__ int next_state(int state, int code, bool border) {
    const int d1 = code & 3, z2 = (code >> 2) & 1, e3 = (code >> 3) & 1;
    if (state == 1) {
        if (MODE == PSA_LOCAL && (border || d1 == 0)) return 0;
        return d1;
    }
    if (state == 2) return (d1 == 1) ? (z2 ? 2 : 1) : (z2 ? 2 : 3);
    return e3 ? 3 : d1;
}
