// psa_pack.cu -- the packed (.S16x2) inter-pair kernel for batches of short DNA pairs
// (BASELINE config 2; also config 1 when many pairs are batched).
//
// Two pairs share every 32-bit register (low half = pair 2q, high half = pair 2q+1), so each DPX
// instruction (VIADDMNMX.S16x2, VIMNMX3.S16x2, VIMNMX.U16x2) updates two cells.  A group of G
// lanes (8 or 16) owns one pair-of-pairs; lane t of the group owns K consecutive columns and the
// group sweeps the rows as a skewed wavefront (shuffles of width G), so a warp carries 32/G
// groups = up to 8 pairs.  Fill recurrence, borders and traceback order are those of
// subproblem_alignment.cpp:229-292 / :147-169 (see psa_short.cu for the derivation); what is
// specific here:
//   * values are stored with a bias B (all halves positive, B chosen per launch from g,h,m,n), so
//     "+ match", "- (g+h)" and the direction-flag differences are plain 32-bit adds that cannot
//     carry between the halves -- ptxas is free to issue them on the FMA pipe (IMAD) while the
//     DPX ops occupy the ALU pipe;
//   * the substitution score is one PRMT: the row character selects a byte table
//     (g+h or g+h+1 per symbol), the column's selector picks its symbol for both pairs;
//   * column state keeps H-(g+h) ("hgo") so that F needs no extra subtract;
//   * local mode uses zero borders for H (equivalent to the -inf borders + 0 floor of the spec
//     for every reported quantity: T1 >= 0 everywhere, see DESIGN.md) and finds the end cell with a
//     packed key T1*32 + (31-k) reduced with VIMNMX3.U16x2;
//   * each cell leaves a 5-bit code: bit0 = (H > T1), bits1-2 = min(H-E,3), bits3-4 = min(H-F,3)
//     (enough to replay find_alignment's first-equality order for h <= 2), computed as one linear
//     form of H and three clamped values (3 VIADDMNMX + 4 IMAD per cell, see pack_step); three
//     codes per 16-bit half, staged through shared memory into whole 128-byte lines of a bounded
//     global scratch ring (layout: see "Direction-code layout" below) and consumed by the traceback kernel (one
//     THREAD per pair, table-driven), which also recovers the local start cell by tracking the
//     running score.  The scratch is O(chunk), not O(batch): it is recycled every chunk.
// Pairs that are not plain upper-case ACGT are flagged and recomputed by the generic int32 kernel
// (psa_short.cu) -- results stay bit-exact for any alphabet.
#include "psa_result.cuh"
#include <chrono>
#include <functional>
#include <type_traits>
#include <vector>

namespace {

__device__ __forceinline__ uint32_t vaddmax(uint32_t a, uint32_t b, uint32_t c) { return __viaddmax_s16x2(a, b, c); }
__device__ __forceinline__ uint32_t vmax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_s16x2(a, b, c); }
__device__ __forceinline__ uint32_t umax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u16x2(a, b, c); }
// prmt with the full 4-bit selector semantics: nibble bit 3 = replicate the sign of the selected byte
// (__byte_perm masks the selector with 0x7777 and so cannot produce the 0x00 filler bytes we need).
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

struct PackConsts {
    uint32_t ng2;     // (-g, -g)
    uint32_t go2;     // (g+h, g+h)
    uint32_t go4;     // g+h in all four bytes (PRMT table base)
    int bias;         // B
    int g, h;
    uint32_t mul32;               // = 32 at run time: keeps the key's scaled add an IMAD (FMA pipe) instead of an ALU-pipe LEA/SHF
    // direction words as ONE linear form: code = 11*H - max(t1,H-1) - 2*max(e,H-3) - 8*max(f,H-3), scaled by
    // 32^x for its slot in the word; index x = 0,1,2.  Run-time values so the products stay IMADs.
    uint32_t m1, m3;              // (-1,-1), (-3,-3)
    uint32_t cH[3], cT[3], cE[3], cF[3];
};

template <int K>
struct PackCols {
    uint32_t hgo[K];   // H[i-1][j] - (g+h), biased, both pairs
    uint32_t f[K];     // F[i-1][j]
    uint32_t sel[K];   // PRMT selector of column j for both pairs
};

__host__ __device__ constexpr int words_for(int K) { return (K + 2) / 3; }
__host__ __device__ constexpr int pad_words(int w) { return w <= 1 ? 1 : (w <= 2 ? 2 : (w <= 4 ? 4 : 8)); }

// Direction-code layout in the ring (per pair-of-pairs slot).  A lane's codes for one row are NWP words.
//   NWP < 4  : row-major, word ((r*G + t)*NWP + q).
//   NWP >= 4 : "staged": indexed by wavefront step s = r + t (the step at which lane t sweeps row r), RB
//              consecutive steps of ONE lane share a 128-byte line:
//                  line = (s / RB)*G + t,   16-byte piece (s % RB)*NP + q/4 inside it,   NP = NWP/4, RB = 8/NP.
//              The fill kernel transposes RB steps through shared memory so that every STG.128 of a warp
//              covers whole, contiguous lines; the traceback, which climbs ~one row per step inside one
//              lane's columns, then finds RB consecutive rows in one line instead of one line per row.
__host__ __device__ constexpr bool dirs_staged(int nwp) { return nwp >= 4; }
__host__ __device__ constexpr int dirs_rb(int nwp) { return 8 / (nwp / 4); }
constexpr int STAGE_ROW_BYTES = 32 * 16 + 16;           // one piece-row of a warp, padded against bank conflicts
constexpr int STAGE_BYTES = 8 * STAGE_ROW_BYTES;        // per warp
__host__ __device__ inline long long dirs_slot_words_for(int max_m, int G, int nwp) {
    if (!dirs_staged(nwp)) return (long long)max_m * G * nwp;
    const int rb = dirs_rb(nwp);
    return (long long)((max_m + G - 1 + rb - 1) / rb) * G * 32;
}
// One lane-step: the K cells of row r owned by this lane, for both pairs.
template <int K, bool LOCAL, bool DIRS, bool CAP>
__device__ __forceinline__ void pack_step(PackCols<K>& L, uint32_t& hl, uint32_t& el, uint32_t diag, uint32_t tA,
                                          uint32_t tB, const PackConsts& C, uint32_t* words, uint32_t& rowkey,
                                          int kcapA, int kcapB, uint32_t* cap) {
    uint32_t acc = 0;
    uint32_t key_prev = 0;
    // all diagonal terms come from the PREVIOUS row: form every T1 first, so that the column state can be
    // updated in place below (otherwise the loop-carried "old hgo[k]" costs a register move per cell)
    uint32_t t1v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t s = prmt(tA, tB, L.sel[k]);       // (go + match) per half
        t1v[k] = (k == 0 ? diag : L.hgo[k - 1]) + s;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t t1 = t1v[k];
        const uint32_t e = vaddmax(el, C.ng2, hl);
        const uint32_t f = vaddmax(L.f[k], C.ng2, L.hgo[k]);
        const uint32_t H = vmax3(t1, e, f);
        if (DIRS) {
            // code = min(H-t1,1) + 2*min(H-e,3) + 8*min(H-f,3), with H - min(H-x,c) = max(x, H-c): three
            // VIADDMNMX and four IMADs per cell, the 32^x slot scaling folded into the multipliers.  The 16-bit
            // halves never interfere: the form is linear, its coefficients sum to zero (the bias cancels) and
            // each half's result is a 15-bit non-negative number, so the 32-bit sum is exact modulo 2^32.
            const uint32_t tc = vaddmax(H, C.m1, t1);
            const uint32_t ec = vaddmax(H, C.m3, e);
            const uint32_t fc = vaddmax(H, C.m3, f);
            constexpr int NWl = (K + 2) / 3;
            const int in_word = (k / 3 == NWl - 1) ? (K - 3 * (NWl - 1)) : 3;
            const int x = in_word - 1 - (k % 3);
            acc = (k % 3 == 0 ? 0u : acc) + H * C.cH[x] + tc * C.cT[x] + ec * C.cE[x] + fc * C.cF[x];
            if (k % 3 == 2 || k == K - 1) words[k / 3] = acc;
        }
        if (LOCAL) {
            const uint32_t key = t1 * C.mul32 + (uint32_t)(31 - k) * 0x00010001u;
            if (k & 1) rowkey = umax3(rowkey, key_prev, key);
            else if (k == K - 1) rowkey = __vmaxu2(rowkey, key);
            key_prev = key;
        }
        if (CAP) {
            if (k == kcapA) { cap[0] = t1; cap[1] = e; cap[2] = f; }
            if (k == kcapB) { cap[3] = t1; cap[4] = e; cap[5] = f; }
        }
        const uint32_t hgo = H - C.go2;
        L.hgo[k] = hgo; L.f[k] = f; hl = hgo; el = e;
    }
}

// Sequence bytes for the traceback, fetched one aligned 32-bit word at a time and reused while the path
// stays inside it (the walk moves one base per step): a quarter of the load requests of byte reads.
struct SeqBytes {
    const uint8_t* s;
    int len;
    int w0 = -(1 << 30);       // index (relative to s) of the first byte of the cached word
    uint32_t w = 0;
    const uint32_t* p2 = nullptr;      // 2-bit packed input instead of bytes: get() returns the 2-bit code
    __device__ __forceinline__ int get(int idx) {
        if (p2 != nullptr) {
            if ((unsigned)(idx - w0) >= 16u) { w0 = idx & ~15; w = __ldg(p2 + (idx >> 4)); }
            return (int)((w >> (2 * (idx - w0))) & 3u);
        }
        if ((unsigned)(idx - w0) >= 4u) {
            const int mis = (int)((uintptr_t)(s + idx) & 3);
            const int b0 = idx - mis;                                  // aligned word [b0, b0+4)
            if (b0 >= 0 && b0 + 4 <= len) { w0 = b0; w = *reinterpret_cast<const uint32_t*>(s + b0); }
            else return s[idx];                                        // word would leave this sequence
        }
        return (int)((w >> (8 * (idx - w0))) & 0xffu);
    }
};

// Per-column constants of the walk, one 32-bit entry per column c = j-1 (built once per CTA in shared
// memory): bits 0-4 lane t = c / K, bits 5-14 the column's word offset inside its line group
// (t*32 + q for the staged layout, t*NWP + q otherwise; q = (c % K) / 3), bits 15-19 the right shift
// that brings the cell's 5-bit code to bit 0 of its 16-bit half.
template <int G, int K, int NWP>
__device__ __forceinline__ uint32_t walk_column_entry(int c) {
    constexpr int NW = (K + 2) / 3;
    const int t = c / K, k = c % K, q = k / 3;
    const int cells = (q == NW - 1) ? (K - 3 * (NW - 1)) : 3;
    const int shift = 5 * (cells - 1 - k % 3);
    const int off = dirs_staged(NWP) ? t * 32 + q : t * NWP + q;
    return (uint32_t)t | ((uint32_t)off << 5) | ((uint32_t)shift << 15);
}

// Walks one pair's path through the 5-bit codes of its slot (subproblem_alignment.cpp:147-169: first
// equality in the order T1, T2, T3; the node on the border is dropped, :170).  `it` carries score / end
// cell / end state in and start cell / length out; ops go to `ow` as 2-bit states in traceback order.
// ctab = walk_column_entry table, lut = pack_tb_lut rows (both in shared memory).
template <int G, int K, int NWP>
__device__ __forceinline__ void pack_walk(const uint32_t* __restrict__ dbase, int half, const uint8_t* sa, const uint8_t* sb,
                                          int m, int n, bool local, int g, int h, const uint32_t* ctab,
                                          const unsigned long long* lut, psa_batch_item& it, uint32_t* ow,
                                          const uint32_t* a2 = nullptr, const uint32_t* b2 = nullptr) {
    constexpr int RB = dirs_staged(NWP) ? dirs_rb(NWP) : 1;
    asm volatile("" : "+l"(dbase));        // keep the slot pointer in a register pair (ptxas re-derives it per step otherwise)
    SeqBytes ca{sa, m}, cb{sb, n};
    ca.p2 = a2; cb.p2 = b2;
    int i = it.end_i, j = it.end_j, state = it.end_state;
    int v = it.score;                      // local: running value of the current state
    int len = 0, first_i = 0, first_j = 0;
    uint32_t acc = 0;
    const int hshift = 16 * half;
    while (i > 0 && j > 0) {
        acc |= (uint32_t)state << (2 * (len & 15));
        if ((len & 15) == 15) { ow[len >> 4] = acc; acc = 0; }
        ++len;
        first_i = i; first_j = j;
        const int si = (state == 2) ? i : i - 1;
        const int sj = (state == 3) ? j : j - 1;
        const bool border = (si == 0 || sj == 0);
        // the code word of the source cell is requested first: its latency (L2 / DRAM) then overlaps the
        // sequence reads and the floor test below instead of following them
        uint32_t ce = 0, w = 0;
        if (!border) {
            ce = ctab[sj - 1];
            int idx;
            if (dirs_staged(NWP)) {
                const int sstep = si - 1 + (int)(ce & 31u);          // wavefront step of the source cell
                idx = (sstep / RB) * (G * 32) + (sstep % RB) * NWP + (int)((ce >> 5) & 1023u);
            } else {
                idx = (si - 1) * (G * NWP) + (int)((ce >> 5) & 1023u);
            }
            w = __ldg(dbase + idx);
        }
        if (local && state == 1) {
            const int f = (ca.get(i - 1) == cb.get(j - 1)) ? 1 : 0;
            if (v == f) break;             // T1[i][j] == f: the 0 floor, first column of the alignment
            v -= f;
        }
        if (border) { i = si; j = sj; break; }                   // predecessor on the border: dropped node
        const uint32_t code = (w >> (hshift + (ce >> 15))) & 31u;
        // next state by table (pack_tb_lut): branch-free, so lanes in different states stay converged
        const int ns = (int)(lut[state - 1] >> (2 * code)) & 3;
        if (state != 1) v += (ns == state) ? g : g + h;
        state = ns; i = si; j = sj;
    }
    if (len & 15) ow[len >> 4] = acc;
    it.aln_len = len;
    it.start_i = first_i; it.start_j = first_j;
}

// Traceback flavours of the fill kernel.
//   TB_CODES : every cell leaves a 5-bit direction code in a global ring (20 KB per 150 x 150 pair), walked by
//              psa_pack_tb_kernel -- the default (option pack_traceback = 0), faster than TB_CKPT (DESIGN.md section 4).
//   TB_CKPT  : (option pack_traceback = 1) the fill keeps only tile-boundary checkpoints (11 KB per pair): the (H-(g+h), E) every lane receives
//              from its left neighbour at every step (= the boundary column between two lanes' strips) and, every
//              PACK_RS wavefront steps, every lane's column state (H-(g+h), F).  psa_pack_rwalk_kernel then
//              recomputes only the <= PACK_RS x K tiles the path crosses, codes in shared memory -- no O(mn)
//              matrix in HBM, no per-cell code extraction in the fill (BASELINE.json north_star).
enum { TB_NONE = 0, TB_CODES = 1, TB_CKPT = 2 };
constexpr int PACK_RS = 16;    // wavefront steps between two row checkpoints

// Checkpoint slot of one pair-of-pairs (uint2 = two packed words, low half pair 2q, high half pair 2q+1), laid out
// for the READER: everything one tile needs is contiguous.
//   col[t*SC + s]              (hl, el) received by lane t at wavefront step s (row s - t); SC = steps_cap
//   row[(c*G + t)*KP + k]      (hgo, f) of lane t's column k after step c*PACK_RS + PACK_RS-1; KP = K rounded up to even
__host__ __device__ constexpr int ck_kp(int K) { return (K + 1) & ~1; }
__host__ __device__ inline int ck_steps_cap(int m_cap, int G) { return (m_cap + G - 1 + 3) & ~3; }
__host__ __device__ inline long long ck_col_u2(int m_cap, int G) { return (long long)ck_steps_cap(m_cap, G) * G; }
__host__ __device__ inline long long ck_slot_u2(int m_cap, int G, int K) {
    const int steps_cap = ck_steps_cap(m_cap, G);
    return ck_col_u2(m_cap, G) + (long long)((steps_cap + PACK_RS - 1) / PACK_RS) * G * ck_kp(K);
}

// Shared-memory staging of the checkpoint stores (per warp): the lanes hold their data per lane, the reader wants it
// contiguous per lane, and L2 wants every store instruction to cover whole 32-byte sectors -- so the data takes a turn
// through shared memory: 4 steps of (hl, el) -> two STG.128 whose lane pairs fill one sector each; a row checkpoint
// (KP uint2 per lane) -> KP/2 STG.128 in which the 8/16 lanes of a group write 128/256 contiguous bytes.
constexpr int CK_COL_STAGE_BYTES = 4 * 32 * 8;
__host__ __device__ constexpr int ck_row_lane_stride(int K) { return ck_kp(K) * 8 + 16; }       // +16: conflict-free STS.128
__host__ __device__ constexpr int ck_stage_bytes(int K) { return CK_COL_STAGE_BYTES + 32 * ck_row_lane_stride(K); }

struct PackArgs {
    psa_batch_args P;
    PackConsts C;
    int m_cap;                 // rows of the per-group table area (>= max m)
    uint32_t* dirs;            // scratch ring for this chunk: per pair-of-pairs slot (codes, or checkpoints as uint2)
    long long dirs_slot_words; // words per pair-of-pairs
    long long pair0;           // first pair of this chunk
    long long pairs;           // pairs in this chunk
    uint8_t* fallback;         // [n_pairs] 1 = not plain ACGT -> generic kernel
    int* flag_count;           // number of pairs of this chunk flagged for the generic kernel (may be null)
};

__device__ __forceinline__ bool dna_code(int c, int& code) {
    code = (c >> 1) & 3;       // A=0 C=1 T=2 G=3
    return c == 'A' || c == 'C' || c == 'G' || c == 'T';
}

template <int G, int K, int MODE, int TB>
__global__ void __launch_bounds__(128) psa_pack_fill_kernel(PackArgs A) {
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    constexpr bool DIRS = (TB == TB_CODES), CKPT = (TB == TB_CKPT);
    constexpr int GPW = 32 / G;                 // groups per warp
    constexpr int NW = words_for(K), NWP = pad_words(NW);
    extern __shared__ __align__(16) uint2 s_tab[];     // [groups per CTA][m_cap] row tables (tA, tB)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = lane % G, grp = lane / G;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (grp * G));
    uint2* tab = s_tab + (size_t)(warp * GPW + grp) * A.m_cap;
    constexpr bool STAGED = DIRS && dirs_staged(NWP);
    constexpr int NP = NWP >= 4 ? NWP / 4 : 1, RB = 8 / NP;
    // staging area of this warp (after every warp's row tables): 8 piece-rows of 32 x 16 bytes
    uint8_t* stage = reinterpret_cast<uint8_t*>(s_tab + (size_t)(blockDim.x >> 5) * GPW * A.m_cap) +
                     (size_t)warp * (CKPT ? ck_stage_bytes(K) : STAGE_BYTES);
    const PackConsts C = A.C;
    const psa_batch_args& P = A.P;
    const long long n_pp = (A.pairs + 1) / 2;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);

    for (long long w0 = (long long)blockIdx.x * (blockDim.x >> 5) + warp; w0 * GPW < n_pp; w0 += warps_total) {
        const long long pp = w0 * GPW + grp;                 // this group's pair-of-pairs (chunk-relative)
        const bool have = pp < n_pp;
        const long long pA = A.pair0 + 2 * pp, pB = pA + 1;
        const bool haveB = have && (2 * pp + 1 < A.pairs);
        const bool pk2 = (P.a2 != nullptr);          // 2-bit packed fixed-stride input
        const int mA = have ? (pk2 ? P.fixed_m : P.len_a[pA]) : 0, nA = have ? (pk2 ? P.fixed_n : P.len_b[pA]) : 0;
        const int mB = haveB ? (pk2 ? P.fixed_m : P.len_a[pB]) : 0, nB = haveB ? (pk2 ? P.fixed_n : P.len_b[pB]) : 0;
        const int mpp = max(mA, mB);
        // ---- row tables: tA/tB[r] = (g+h) in every byte, +1 in the byte of the row's symbol ----
        bool okA = true, okB = true;
        {
            if (pk2) {
                const uint32_t* wA = P.a2 + pA * P.wa;
                const uint32_t* wB = P.a2 + pB * P.wa;
                for (int r = t; r < mpp; r += G) {
                    uint32_t ta = C.go4, tb = C.go4;
                    if (r < mA) ta += 1u << (8 * ((__ldg(wA + (r >> 4)) >> (2 * (r & 15))) & 3u));
                    if (r < mB) tb += 1u << (8 * ((__ldg(wB + (r >> 4)) >> (2 * (r & 15))) & 3u));
                    tab[r] = make_uint2(ta, tb);
                }
            } else {
            const uint8_t* gaA = have ? P.bases_a + P.off_a[pA] : nullptr;
            const uint8_t* gaB = haveB ? P.bases_a + P.off_a[pB] : nullptr;
            for (int r = t; r < mpp; r += G) {
                uint32_t ta = C.go4, tb = C.go4;
                int code;
                if (r < mA) { okA &= dna_code(gaA[r], code); ta += 1u << (8 * code); }
                if (r < mB) { okB &= dna_code(gaB[r], code); tb += 1u << (8 * code); }
                tab[r] = make_uint2(ta, tb);
            }
            }
        }
        // ---- column state ----
        PackCols<K> L;
        {
            const uint8_t* gbA = (have && !pk2) ? P.bases_b + P.off_b[pA] : nullptr;
            const uint8_t* gbB = (haveB && !pk2) ? P.bases_b + P.off_b[pB] : nullptr;
            const uint32_t* vA = pk2 ? P.b2 + pA * P.wb : nullptr;
            const uint32_t* vB = pk2 ? P.b2 + pB * P.wb : nullptr;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int j = t * K + k;     // 0-based column
                int ca = 8, cb = 8, code;
                if (pk2) {
                    if (j < nA) ca = (int)((__ldg(vA + (j >> 4)) >> (2 * (j & 15))) & 3u);
                    if (j < nB) cb = 4 + (int)((__ldg(vB + (j >> 4)) >> (2 * (j & 15))) & 3u);
                } else {
                if (j < nA) { okA &= dna_code(gbA[j], code); ca = code; }
                if (j < nB) { okB &= dna_code(gbB[j], code); cb = 4 + code; }
                }
                L.sel[k] = (uint32_t)ca | 0x80u | ((uint32_t)cb << 8) | 0x8000u;
                const int hb = LOCAL ? C.bias : C.bias - C.h - C.g * (j + 1);        // H[0][j+1] (cpp:222-224)
                L.hgo[k] = (uint32_t)(hb - (C.g + C.h)) * 0x00010001u;
                L.f[k] = 0u;                                                          // -inf
            }
        }
        okA = __all_sync(gmask, okA);
        okB = __all_sync(gmask, okB);
        __syncwarp();
        // H[0][c0] - go for the lane's first diagonal; lane 0: H[0][0] = 0 (T1[0][0], cpp:264-265)
        uint32_t hd;
        {
            const int c0 = t * K;
            const int hb = (LOCAL || c0 == 0) ? C.bias : C.bias - C.h - C.g * c0;
            hd = (uint32_t)(hb - (C.g + C.h)) * 0x00010001u;
        }
        // lane 0's left border H[i][0] - go, advanced by -g per row (T3[i][0] = -h - g*i, cpp:290-292)
        uint32_t bord = (uint32_t)((LOCAL ? C.bias : C.bias - C.h - C.g) - (C.g + C.h)) * 0x00010001u;
        uint32_t recv_h = 0, recv_e = 0;
        uint32_t bestA = 0, bestB = 0;       // local: best key per half (T1*32 + 31-k), and its row
        int biA = 0, biB = 0;
        uint32_t cap[6] = {0, 0, 0, 0, 0, 0};
        // global: which lane/k holds column n of each pair
        const int tcapA = (nA > 0) ? (nA - 1) / K : -1, kcA = (nA > 0) ? (nA - 1) % K : -1;
        const int tcapB = (nB > 0) ? (nB - 1) / K : -1, kcB = (nB > 0) ? (nB - 1) % K : -1;
        uint32_t* dbase = DIRS ? A.dirs + pp * A.dirs_slot_words : nullptr;
        // checkpoints: running pointers into this pair-of-pairs' slot (column part advances G per step, row part
        // K*G per checkpoint)
        // checkpoints: slot of the warp's first group; group x's slot follows at x * slot
        uint2* ck_warp = CKPT ? reinterpret_cast<uint2*>(A.dirs) + (w0 * GPW) * (A.dirs_slot_words / 2) : nullptr;
        const int ck_sc = ck_steps_cap(A.m_cap, G);
        int ck_c = 0;                              // row checkpoints taken so far

        int mw = mpp;                          // warp-uniform step count
#pragma unroll
        for (int off = 16; off >= G; off >>= 1) mw = max(mw, __shfl_xor_sync(0xffffffffu, mw, off));
        const int steps = mw + G - 1;
        for (int s = 0; s < steps; ++s) {
            const int r = s - t;
            uint32_t hl, el;
            if (t == 0) { hl = bord; el = 0u; } else { hl = recv_h; el = recv_e; }
            if (CKPT) *reinterpret_cast<uint2*>(stage + ((s & 3) * 32 + lane) * 8) = make_uint2(hl, el);
            const bool active = (r >= 0 && r < mpp);
            bool capstep = false;
            if (!LOCAL) capstep = active && ((r == mA - 1 && t == tcapA) || (r == mB - 1 && t == tcapB));
            const bool anycap = LOCAL ? false : __any_sync(0xffffffffu, capstep);
            if (active) {
                const uint2 tt = tab[r];
                const uint32_t hl0 = hl;
                uint32_t words[NWP];
                uint32_t rowkey = 0;
                if (!anycap) {
                    pack_step<K, LOCAL, DIRS, false>(L, hl, el, hd, tt.x, tt.y, C, words, rowkey, -1, -1, cap);
                } else {
                    const int ka = (r == mA - 1 && t == tcapA) ? kcA : -1;
                    const int kb = (r == mB - 1 && t == tcapB) ? kcB : -1;
                    pack_step<K, LOCAL, DIRS, true>(L, hl, el, hd, tt.x, tt.y, C, words, rowkey, ka, kb, cap);
                }
                hd = hl0;
                if (!LOCAL && t == 0) bord -= (uint32_t)C.g * 0x00010001u;
                if (DIRS) {
#pragma unroll
                    for (int q = NW; q < NWP; ++q) words[q] = 0;
                    if (STAGED) {
#pragma unroll
                        for (int hq = 0; hq < NP; ++hq)
                            *reinterpret_cast<uint4*>(stage + ((s % RB) * NP + hq) * STAGE_ROW_BYTES + lane * 16) =
                                make_uint4(words[4 * hq], words[4 * hq + 1], words[4 * hq + 2], words[4 * hq + 3]);
                    } else {
                        uint32_t* dst = dbase + ((long long)r * G + t) * NWP;
                        if (NWP == 2) reinterpret_cast<uint2*>(dst)[0] = make_uint2(words[0], words[1]);
                        else dst[0] = words[0];
                    }
                }
                if (LOCAL) {
                    const uint32_t lo = rowkey & 0xffffu, hi = rowkey >> 16;
                    if (lo > (bestA | 31u)) { bestA = lo; biA = r + 1; }
                    if (hi > (bestB | 31u)) { bestB = hi; biB = r + 1; }
                }
            }
            recv_h = __shfl_up_sync(0xffffffffu, hl, 1, G);
            recv_e = __shfl_up_sync(0xffffffffu, el, 1, G);
            if (CKPT) {
                if ((s & 3) == 3 || s == steps - 1) {
                    // the last 4 steps of every lane's boundary stream: lane pair (2x, 2x+1) writes the sector of stream x
                    __syncwarp();
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        const int x = jj * 16 + (lane >> 1), hh = lane & 1;            // stream = warp lane x; which half of its sector
                        const uint2 u0 = *reinterpret_cast<const uint2*>(stage + ((2 * hh) * 32 + x) * 8);
                        const uint2 u1 = *reinterpret_cast<const uint2*>(stage + ((2 * hh + 1) * 32 + x) * 8);
                        const int xg = x / G, xt = x % G;
                        if (w0 * GPW + xg < n_pp)
                            *reinterpret_cast<uint4*>(ck_warp + (long long)xg * (A.dirs_slot_words / 2) + (long long)xt * ck_sc + (s & ~3) + 2 * hh) =
                                make_uint4(u0.x, u0.y, u1.x, u1.y);
                    }
                    __syncwarp();
                }
                if ((s % PACK_RS) == PACK_RS - 1) {      // every lane, whatever row it is on: skewed checkpoint line
                    constexpr int KP = ck_kp(K), LS = ck_row_lane_stride(K);
                    uint8_t* rst = stage + CK_COL_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < KP; k += 2)
                        *reinterpret_cast<uint4*>(rst + lane * LS + k * 8) =
                            make_uint4(L.hgo[k], L.f[k], k + 1 < K ? L.hgo[k + 1 < K ? k + 1 : k] : 0u, k + 1 < K ? L.f[k + 1 < K ? k + 1 : k] : 0u);
                    __syncwarp();
                    if (have) {
                        // the group's G * KP uint2 are contiguous: 16-byte chunk u = t + G*y comes from lane u / (KP/2) of the group
                        uint4* dst = reinterpret_cast<uint4*>(ck_warp + (long long)grp * (A.dirs_slot_words / 2) + ck_col_u2(A.m_cap, G) +
                                                              (long long)ck_c * G * KP);
#pragma unroll
                        for (int y = 0; y < KP / 2; ++y) {
                            const int u = t + G * y;
                            dst[u] = *reinterpret_cast<const uint4*>(rst + (grp * G + u / (KP / 2)) * LS + (u % (KP / 2)) * 16);
                        }
                    }
                    ++ck_c;
                    __syncwarp();
                }
            }
            if (STAGED) {
                if ((s % RB) == RB - 1 || s == steps - 1) {
                    // RB steps staged: write the group's G lines of this block, 16 bytes per lane per store,
                    // consecutive lanes to consecutive addresses
                    __syncwarp();
                    if (have) {
                        uint4* out = reinterpret_cast<uint4*>(dbase + (long long)(s / RB) * G * 32);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int pc = i * G + t;                     // piece of the group's G x 128 bytes
                            out[pc] = *reinterpret_cast<const uint4*>(stage + (pc & 7) * STAGE_ROW_BYTES + (grp * G + (pc >> 3)) * 16);
                        }
                    }
                    __syncwarp();
                }
            }
        }

        // ---- results ----
        if (LOCAL) {
            // (T1, smallest i, smallest j) across the group's lanes
            auto full = [&](uint32_t best, int bi) -> uint32_t {
                const int t1v = (int)(best >> 5) - C.bias;
                if (t1v <= 0) return 0u;
                const int j = t * K + (31 - (int)(best & 31u)) + 1;
                return ((uint32_t)t1v << 20) | ((uint32_t)(1023 - bi) << 10) | (uint32_t)(1023 - j);
            };
            uint32_t fa = full(bestA, biA), fb = full(bestB, biB);
#pragma unroll
            for (int off = G / 2; off >= 1; off >>= 1) {
                fa = max(fa, __shfl_xor_sync(0xffffffffu, fa, off));
                fb = max(fb, __shfl_xor_sync(0xffffffffu, fb, off));
            }
            if (t == 0 && have) {
                auto item = [](uint32_t f) {
                    return local_item((int)(f >> 20), f ? 1023 - (int)((f >> 10) & 1023u) : 0, f ? 1023 - (int)(f & 1023u) : 0);
                };
                if (mA > 0 && nA > 0) P.items[pA] = item(fa);
                if (haveB && mB > 0 && nB > 0) P.items[pB] = item(fb);
            }
        } else {
            // the capturing lane of each pair writes its corner (exactly one lane per pair)
            if (have && mA > 0 && nA > 0 && t == tcapA) P.items[pA] = packed_corner_item(cap, 0, C.bias, mA, nA);
            if (haveB && mB > 0 && nB > 0 && t == tcapB) P.items[pB] = packed_corner_item(cap + 3, 16, C.bias, mB, nB);
        }
        if (t == 0 && have) {
            // degenerate members (a zero length) and non-ACGT members go to the generic kernel
            const int fa_ = (!okA || mA == 0 || nA == 0) ? 1 : 0, fb_ = (haveB && (!okB || mB == 0 || nB == 0)) ? 1 : 0;
            A.fallback[pA] = (uint8_t)fa_;
            if (haveB) A.fallback[pB] = (uint8_t)fb_;
            if ((fa_ | fb_) && A.flag_count != nullptr) atomicAdd(A.flag_count, fa_ + fb_);
        }
        __syncwarp();
    }
}

// ---- traceback: one thread per pair walks the 5-bit codes ------------------------------------
struct PackTbArgs {
    psa_batch_args P;
    PackConsts C;
    const uint32_t* dirs;
    long long dirs_slot_words;
    long long pair0, pairs;
    const uint8_t* fallback;
    int local;
    unsigned long long lut[3];   // next state for current state 1,2,3: 2 bits per 5-bit code (pack_tb_lut)
};

// The predecessor rule of find_alignment (subproblem_alignment.cpp:147-169) over the 5-bit code of the
// source cell (ma = min(H-T1,1), mb = min(H-T2,3), mc = min(H-T3,3)), for gap-open penalty h <= 2.
static void pack_tb_lut(int h, unsigned long long lut[3]) {
    lut[0] = lut[1] = lut[2] = 0;
    for (int code = 0; code < 32; ++code) {
        const int ma = code & 1, mb = (code >> 1) & 3, mc = (code >> 3) & 3;
        const int d1 = (ma == 0) ? 1 : (mb == 0 ? 2 : 3);
        const int z2 = (d1 == 1) ? (mb < h) : (mb <= h);
        const int n2 = (d1 == 1) ? (z2 ? 2 : 1) : (z2 ? 2 : 3);
        const int n3 = (mc < h) ? 3 : d1;
        lut[0] |= (unsigned long long)d1 << (2 * code);
        lut[1] |= (unsigned long long)n2 << (2 * code);
        lut[2] |= (unsigned long long)n3 << (2 * code);
    }
}

template <int G, int K>
__global__ void __launch_bounds__(128) psa_pack_tb_kernel(PackTbArgs A) {
    constexpr int NWP = pad_words(words_for(K));
    __shared__ uint32_t ctab[G * K];
    __shared__ unsigned long long lut[3];
    for (int c = threadIdx.x; c < G * K; c += blockDim.x) ctab[c] = walk_column_entry<G, K, NWP>(c);
    if (threadIdx.x < 3) lut[threadIdx.x] = A.lut[threadIdx.x];
    __syncthreads();
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= A.pairs) return;
    const long long p = A.pair0 + q;
    if (A.fallback[p]) return;
    const psa_batch_args& P = A.P;
    psa_batch_item it = P.items[p];
    if (P.a2 != nullptr)
        pack_walk<G, K, NWP>(A.dirs + (q >> 1) * A.dirs_slot_words, (int)(q & 1), nullptr, nullptr, P.fixed_m, P.fixed_n,
                             A.local != 0, A.C.g, A.C.h, ctab, lut, it, P.ops + p * P.ops_stride_words, P.a2 + p * P.wa, P.b2 + p * P.wb);
    else
        pack_walk<G, K, NWP>(A.dirs + (q >> 1) * A.dirs_slot_words, (int)(q & 1), P.bases_a + P.off_a[p], P.bases_b + P.off_b[p],
                             P.len_a[p], P.len_b[p], A.local != 0, A.C.g, A.C.h, ctab, lut, it, P.ops + p * P.ops_stride_words);
    P.items[p] = it;
}

// ---- traceback by tile recompute (TB_CKPT) ---------------------------------------------------
// One THREAD per pair.  The path is followed tile by tile: a tile is strip t (the K columns lane t of the fill
// owned) between two consecutive row checkpoints of that strip (<= PACK_RS rows).  The thread reloads the
// tile's top boundary (a row checkpoint, or the row-0 border) and left boundary (the (hl, el) stream lane t
// received), recomputes the tile with the SAME packed arithmetic as the fill -- the two 16-bit halves of every
// register now carry the left and the right half of the tile's columns, the right half running one row behind
// and fed by the left half's last column -- leaves the 5-bit codes in shared memory and walks them
// (find_alignment's first-equality order, subproblem_alignment.cpp:147-169) until the path leaves the tile.
// Only rows up to the entry row are recomputed.  Pairs are visited in descending order of their expected path
// length (perm, built by psa_pack_perm_kernel) so that the threads of a warp cross similar numbers of tiles.
struct PackWalkArgs {
    psa_batch_args P;
    PackConsts C;
    const uint2* ck;
    long long ck_slot;         // uint2 per pair-of-pairs
    long long ck_col;          // uint2 of the column part
    long long pair0, pairs;
    const uint8_t* fallback;
    const int* perm;           // [pairs] chunk-relative pair indices, longest expected paths first (may be null)
    int local;
    int m_cap;
    unsigned long long lut[3];
};

// dynamic shared memory of psa_pack_rwalk_kernel for `nthr` threads: codes | 2-bit sequences
__host__ __device__ inline size_t rwalk_smem_words(int K, int m_cap, int n_cap) {
    const int KH = (K + 1) / 2, NWH = words_for(KH);
    return (size_t)(PACK_RS + 1) * NWH + (size_t)((m_cap + 15) / 16) + (size_t)((n_cap + 15) / 16);
}

template <int G, int K>
__global__ void __launch_bounds__(128) psa_pack_rwalk_kernel(PackWalkArgs A) {
    constexpr int KH = (K + 1) / 2, NWH = words_for(KH), RS = PACK_RS, KP = ck_kp(K);
    extern __shared__ uint32_t s_dyn[];              // per thread, word w at [w * blockDim.x + tid]: codes, then A and B as 2-bit codes
    __shared__ uint8_t lutb[3 * 32];                 // next state for (state - 1, 5-bit code)
    __shared__ uint32_t wtab[K];                     // per tile column: word offset | shift << 8
    for (int e = threadIdx.x; e < 96; e += blockDim.x) lutb[e] = (uint8_t)((A.lut[e >> 5] >> (2 * (e & 31))) & 3u);
    for (int cc = threadIdx.x; cc < K; cc += blockDim.x) {
        const int hi = cc >= KH ? 1 : 0, k = cc - hi * KH;
        const int in_word = (k / 3 == NWH - 1) ? (KH - 3 * (NWH - 1)) : 3;
        const int shift = 5 * (in_word - 1 - k % 3) + 16 * hi;
        wtab[cc] = (uint32_t)(hi * NWH + k / 3) | ((uint32_t)shift << 8);       // the right half sits one iteration later
    }
    __syncthreads();
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= A.pairs) return;
    const long long pr = A.perm ? (long long)A.perm[q] : q;
    const long long p = A.pair0 + pr;
    if (A.fallback[p]) return;
    const int nthr = blockDim.x;
    const psa_batch_args& P = A.P;
    const PackConsts& C = A.C;
    const bool local = A.local != 0;
    const int g = C.g, h = C.h, go = C.g + C.h;
    psa_batch_item it = P.items[p];
    const bool pk2 = (P.a2 != nullptr);
    const int m = pk2 ? P.fixed_m : P.len_a[p], n = pk2 ? P.fixed_n : P.len_b[p];
    uint32_t* codes = s_dyn + threadIdx.x;
    uint32_t* a2 = codes + (size_t)(RS + 1) * NWH * nthr;
    uint32_t* b2 = a2 + (size_t)((A.m_cap + 15) / 16) * nthr;
    if (pk2) {
        for (int w = 0; w * 16 < m; ++w) a2[w * nthr] = __ldg(P.a2 + p * P.wa + w);
        for (int w = 0; w * 16 < n; ++w) b2[w * nthr] = __ldg(P.b2 + p * P.wb + w);
    } else {   // both sequences as 2-bit codes (flagged pairs never get here: every byte is one of ACGT)
        const uint8_t* sa = P.bases_a + P.off_a[p];
        const uint8_t* sb = P.bases_b + P.off_b[p];
        for (int w = 0; w * 16 < m; ++w) {
            uint32_t v = 0;
            const int e = min(16, m - w * 16);
            for (int x = 0; x < e; ++x) v |= (uint32_t)((sa[w * 16 + x] >> 1) & 3) << (2 * x);
            a2[w * nthr] = v;
        }
        for (int w = 0; w * 16 < n; ++w) {
            uint32_t v = 0;
            const int e = min(16, n - w * 16);
            for (int x = 0; x < e; ++x) v |= (uint32_t)((sb[w * 16 + x] >> 1) & 3) << (2 * x);
            b2[w * nthr] = v;
        }
    }
    auto code_a = [&](int r) -> int { return (int)(a2[(r >> 4) * nthr] >> (2 * (r & 15))) & 3; };     // 0-based
    auto code_b = [&](int c) -> int { return (int)(b2[(c >> 4) * nthr] >> (2 * (c & 15))) & 3; };
    const int half = (int)(pr & 1);
    const uint2* colck = A.ck + (pr >> 1) * A.ck_slot;
    const uint2* rowck = colck + A.ck_col;
    const int SC = (int)(A.ck_col / G);
    const uint32_t sel_own_lo = half ? 0x5432u : 0x5410u;    // (own half of a, LOW half of b)
    const uint32_t sel_own_own = half ? 0x7632u : 0x5410u;   // (own half of a, own half of b)
    uint32_t* ow = P.ops + p * P.ops_stride_words;

    int i = it.end_i, j = it.end_j, state = it.end_state;
    int v = it.score;
    int len = 0;
    uint32_t acc = 0;
    int r_first = 0, c0 = 0;
    bool done = !(i > 0 && j > 0);
    bool need = !done && ((state == 2 ? i : i - 1) > 0) && ((state == 3 ? j : j - 1) > 0);
    while (!done) {
        if (need) {
            // ---------------- recompute tile (strip t, checkpoint interval c), rows r_first .. r ----------------
            const int r = ((state == 2) ? i : i - 1) - 1, t = (((state == 3) ? j : j - 1) - 1) / K;
            const int c = (r + t) / RS;
            r_first = max(0, RS * c - t);
            c0 = t * K;
            const int nrows = r - r_first + 1;
            PackCols<KH> L;
#pragma unroll
            for (int k = 0; k < KH; ++k) {
                const int j0 = c0 + k, j1 = c0 + KH + k;
                int cl = 8, ch = 8;
                if (j0 < n) cl = code_b(j0);
                if (KH + k < K && j1 < n) ch = 4 + code_b(j1);
                L.sel[k] = (uint32_t)cl | 0x80u | ((uint32_t)ch << 8) | 0x8000u;
            }
            if (c == 0) {
#pragma unroll
                for (int k = 0; k < KH; ++k) {       // row 0 (cpp:222-224), as the fill initialises it
                    const int hb0 = local ? C.bias : C.bias - h - g * (c0 + k + 1);
                    const int hb1 = local ? C.bias : C.bias - h - g * (c0 + KH + k + 1);
                    L.hgo[k] = ((uint32_t)(hb0 - go) & 0xffffu) | ((uint32_t)(hb1 - go) << 16);
                    L.f[k] = 0u;
                }
            } else {
                const uint4* rp = reinterpret_cast<const uint4*>(rowck + ((long long)(c - 1) * G + t) * KP);
                uint4 w[KP / 2];
#pragma unroll
                for (int x = 0; x < KP / 2; ++x) w[x] = __ldg(rp + x);
                auto hg = [&](int k) -> uint32_t { return (k & 1) ? w[k / 2].z : w[k / 2].x; };
                auto ff = [&](int k) -> uint32_t { return (k & 1) ? w[k / 2].w : w[k / 2].y; };
#pragma unroll
                for (int k = 0; k < KH; ++k) {
                    const bool two = KH + k < K;
                    L.hgo[k] = prmt(hg(k), two ? hg(two ? KH + k : 0) : 0u, sel_own_own);
                    L.f[k] = prmt(ff(k), two ? ff(two ? KH + k : 0) : 0u, sel_own_own);
                }
            }
            const uint2* lbp = colck + (long long)t * SC + (r_first + t);       // lane t received row r at step r + t
            // H[r_first-1][c0] - (g+h): the diagonal of the left half's first cell
            uint32_t diag;
            if (r_first == 0) diag = (uint32_t)(((local || c0 == 0) ? C.bias : C.bias - h - g * c0) - go);
            else { const uint32_t w = __ldg(&lbp[-1].x); diag = half ? (w >> 16) : (w & 0xffffu); }
            uint32_t prev_h = L.hgo[KH - 1], prev_e = 0u;      // low halves feed the right half one iteration later
            uint32_t t_hi = C.go4;
            uint2 lb = __ldg(lbp);
            uint32_t* cw = codes;
            for (int itx = 0; itx <= nrows; ++itx) {
                const uint2 lb_cur = lb;
                const uint32_t t_lo = C.go4 + (1u << (8 * code_a(min(r_first + itx, r))));
                if (itx + 1 < nrows) lb = __ldg(lbp + itx + 1);          // next row's boundary words in flight
                uint32_t hl = prmt(lb_cur.x, prev_h, sel_own_lo);
                uint32_t el = prmt(lb_cur.y, prev_e, sel_own_lo);
                const uint32_t hl0 = hl;
                uint32_t words[NWH], rowkey = 0, cap[1];
                if (itx == 0) {
                    // the right half has no row yet: run the step for the left half, then put the right half's top
                    // boundary back
                    uint32_t oh[KH], of[KH];
#pragma unroll
                    for (int k = 0; k < KH; ++k) { oh[k] = L.hgo[k]; of[k] = L.f[k]; }
                    pack_step<KH, false, true, false>(L, hl, el, diag, t_lo, t_hi, C, words, rowkey, -1, -1, cap);
                    prev_h = L.hgo[KH - 1]; prev_e = el;
#pragma unroll
                    for (int k = 0; k < KH; ++k) { L.hgo[k] = prmt(L.hgo[k], oh[k], 0x7610u); L.f[k] = prmt(L.f[k], of[k], 0x7610u); }
                } else {
                    pack_step<KH, false, true, false>(L, hl, el, diag, t_lo, t_hi, C, words, rowkey, -1, -1, cap);
                    prev_h = L.hgo[KH - 1]; prev_e = el;
                }
#pragma unroll
                for (int w = 0; w < NWH; ++w) cw[w * nthr] = words[w];
                cw += NWH * nthr;
                diag = hl0;
                t_hi = t_lo;
            }
        }
        // ---------------- walk while the source cell stays inside the tile ----------------
        for (;;) {
            const int si = (state == 2) ? i : i - 1, sj = (state == 3) ? j : j - 1;
            const bool border = (si == 0 || sj == 0);
            const int cc = sj - 1 - c0, rr = si - 1 - r_first;
            if (!border && (cc < 0 || rr < 0)) { need = true; break; }        // another tile (the path only moves up / left)
            acc |= (uint32_t)state << (2 * (len & 15));
            if ((len & 15) == 15) { ow[len >> 4] = acc; acc = 0; }
            ++len;
            if (local && state == 1) {
                const int f = (code_a(i - 1) == code_b(j - 1)) ? 1 : 0;
                if (v == f) { done = true; break; }             // T1[i][j] == f: the 0 floor, first column of the alignment
                v -= f;
            }
            if (border) { done = true; break; }                 // predecessor on the border: dropped node (cpp:170)
            const uint32_t we = wtab[cc];
            const uint32_t w = codes[(rr * NWH + (int)(we & 0xffu)) * nthr];
            const int ns = lutb[(state - 1) * 32 + ((w >> (we >> 8)) & 31u)];
            if (state != 1) v += (ns == state) ? g : g + h;
            state = ns; i = si; j = sj;
        }
    }
    if (len & 15) ow[len >> 4] = acc;
    it.aln_len = len;
    it.start_i = len ? i : 0; it.start_j = len ? j : 0;
    P.items[p] = it;
}

// Visiting order of the tile-recompute walk: chunk-relative pair indices sorted by descending expected path length
// (local: the score; global: (m + n) / 2) into 32 buckets -- a counting sort in two small grid-wide passes with
// warp-aggregated atomics (pass 0: histogram into hist[0..31]; pass 1: scatter, cursors in hist[32..63]).
__global__ void __launch_bounds__(256) psa_pack_perm_kernel(const psa_batch_item* items, const int32_t* len_a, const int32_t* len_b,
                                                             long long pair0, int pairs, int local, int span, int* hist, int* perm,
                                                             int pass) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = q < pairs;
    int b = 0;
    if (ok) {
        const long long p = pair0 + q;
        const int key = local ? items[p].score : (len_a ? (len_a[p] + len_b[p]) / 2 : span);
        b = 31 - min(max((int)((long long)key * 32 / (span + 1)), 0), 31);     // bucket 0 = longest
    }
    const unsigned peers = __match_any_sync(0xffffffffu, ok ? b : -1);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1, rank = __popc(peers & ((1u << lane) - 1u));
    if (pass == 0) {
        if (ok && lane == leader) atomicAdd(&hist[b], __popc(peers));
        return;
    }
    int base = 0;
    if (ok && lane == leader) {
        for (int x = 0; x < b; ++x) base += hist[x];
        base += atomicAdd(&hist[32 + b], __popc(peers));
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (ok) perm[base + rank] = q;
}

template <int G, int K>
int launch_fill(psa_ctx* ctx, const PackArgs& A, int mode, int tb, cudaStream_t st) {
    constexpr int GPW = 32 / G;
    const int wpb = 4;
    const size_t smem = (size_t)wpb * GPW * A.m_cap * sizeof(uint2) +
                        (tb == TB_CODES ? (size_t)wpb * STAGE_BYTES : (tb == TB_CKPT ? (size_t)wpb * ck_stage_bytes(K) : 0));
    const long long n_pp = (A.pairs + 1) / 2;
    const long long warps = (n_pp + GPW - 1) / GPW;
    auto go = [&](auto kern) -> int {
        if (smem > (size_t)ctx->smem_optin) return psa_fail(ctx, PSA_ERR_RANGE, "packed kernel does not fit");
        const int orc = psa_kernel_optin_smem(ctx, (const void*)kern);
        if (orc) return orc;
        int per_sm = 0;
        PSA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, wpb * 32, smem));
        if (per_sm < 1) return psa_fail(ctx, PSA_ERR_RANGE, "packed kernel does not fit");
        if (ctx->opt.pack_ctas_per_sm > 0) per_sm = std::max(1, std::min(per_sm, ctx->opt.pack_ctas_per_sm));
        long long grid = std::min<long long>((warps + wpb - 1) / wpb, (long long)per_sm * ctx->sm_count);
        if (grid < 1) grid = 1;
        kern<<<(int)grid, wpb * 32, smem, st>>>(A);
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
        return PSA_OK;
    };
    if (mode == PSA_LOCAL) {
        if (tb == TB_CKPT) return go(psa_pack_fill_kernel<G, K, PSA_LOCAL, TB_CKPT>);
        return tb ? go(psa_pack_fill_kernel<G, K, PSA_LOCAL, TB_CODES>) : go(psa_pack_fill_kernel<G, K, PSA_LOCAL, TB_NONE>);
    }
    if (tb == TB_CKPT) return go(psa_pack_fill_kernel<G, K, PSA_GLOBAL, TB_CKPT>);
    return tb ? go(psa_pack_fill_kernel<G, K, PSA_GLOBAL, TB_CODES>) : go(psa_pack_fill_kernel<G, K, PSA_GLOBAL, TB_NONE>);
}

// Bias B: every stored half must stay >= g+h so that the plain 32-bit adds never carry between the
// two pairs.  True values are >= -(2h + g(m+n)) in global mode and >= -(g+h) on real cells in local
// mode; PADDING cells (rows/columns past a member's own m, n, computed because the two members
// and the warp's groups run in lockstep) keep decaying by at most g per step, g+h once per
// direction -- hence the extra g(m+n) + 2(g+h).
long long pack_bias(int mode, int g, int h, int max_m, int max_n) {
    const long long decay = (long long)g * (max_m + max_n) + 2 * (g + h);
    if (mode == PSA_LOCAL) return (g + h) + 16 + decay;
    return (long long)g * (max_m + max_n) + 2 * h + (g + h) + 16 + decay;
}

struct Shape { int G, K; };
bool pick_shape(int max_n, Shape& s) {
    if (max_n <= 32) s = {8, 4};
    else if (max_n <= 64) s = {8, 8};
    else if (max_n <= 96) s = {8, 12};
    else if (max_n <= 128) s = {8, 16};
    else if (max_n <= 152) s = {8, 19};
    else if (max_n <= 160) s = {8, 20};
    else if (max_n <= 192) s = {16, 12};
    else if (max_n <= 256) s = {16, 16};
    else return false;
    return true;
}

// Calls f(integral_constant<int, G>, integral_constant<int, K>) for the shape pick_shape chose: the one list of the
// (G, K) instantiations of the fill and walk kernels.
template <class F>
int with_shape(const Shape& s, F&& f) {
    using std::integral_constant;
    switch (s.G * 100 + s.K) {
        case 804: return f(integral_constant<int, 8>{}, integral_constant<int, 4>{});
        case 808: return f(integral_constant<int, 8>{}, integral_constant<int, 8>{});
        case 812: return f(integral_constant<int, 8>{}, integral_constant<int, 12>{});
        case 816: return f(integral_constant<int, 8>{}, integral_constant<int, 16>{});
        case 819: return f(integral_constant<int, 8>{}, integral_constant<int, 19>{});
        case 820: return f(integral_constant<int, 8>{}, integral_constant<int, 20>{});
        case 1612: return f(integral_constant<int, 16>{}, integral_constant<int, 12>{});
        default: return f(integral_constant<int, 16>{}, integral_constant<int, 16>{});
    }
}

}  // namespace

bool psa_pack_supported(int max_m, int max_n, int mode, int g, int h) {
    Shape s;
    if (!pick_shape(max_n, s) || max_m > 512 || max_m < 1 || max_n < 1) return false;
    if (h > 2 || g + h + 1 > 120) return false;
    if (mode == PSA_LOCAL && g + h < 1) return false;   // padding cells can only tie the best when g+h == 0
    const long long bias = pack_bias(mode, g, h, max_m, max_n);
    const long long top = bias + std::min(max_m, max_n) + g + h + 2;
    if (mode == PSA_LOCAL) return top * 32 + 31 < 65536;
    return top < 32000;
}

namespace {

constexpr int kInFlight = 4;     // chunks in flight: rings, perm buffers and aux streams (DESIGN.md section 5)
constexpr int kCounters = 4096;  // flagged-pair counters, one per chunk

// What every chunk of one packed batch shares, decided once per call by pack_plan: the kernel shape and constants,
// the traceback flavour and the scratch in ctx->d_work.  Chunk c uses ring and perm buffer c % kInFlight and, for
// byte input, flagged-pair counter c.
struct PackPlan {
    psa_batch_args args;               // device view of the whole batch
    int max_m, max_n, mode;
    int flavour;                       // TB_NONE (score only), TB_CODES or TB_CKPT
    Shape sh;
    PackConsts C;
    uint8_t* flags;                    // fallback bytes of the WHOLE batch (indexed by absolute pair)
    int* counters;                     // [kCounters]
    uint32_t* rings[kInFlight];        // direction codes or checkpoints of one chunk
    int* perms[kInFlight];             // visiting order of the tile-recompute walk (TB_CKPT only, else null)
    long long slot_words;              // ring words per pair-of-pairs
};

long long pairs_cap_round(long long pairs) { return (pairs + 63) / 64 * 64; }

template <int G, int K>
int launch_walk(psa_ctx* ctx, const PackPlan& P, const uint32_t* ring, int* perm, long long pair0, long long pairs,
                cudaStream_t st) {
    const psa_batch_args& args = P.args;
    const bool local = P.mode == PSA_LOCAL;
    if (P.flavour == TB_CODES) {
        PackTbArgs T;
        T.P = args; T.C = P.C; T.dirs = ring; T.dirs_slot_words = P.slot_words; T.pair0 = pair0; T.pairs = pairs;
        T.fallback = P.flags; T.local = local;
        pack_tb_lut(P.C.h, T.lut);
        psa_pack_tb_kernel<G, K><<<(int)((pairs + 127) / 128), 128, 0, st>>>(T);
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
        return PSA_OK;
    }
    // visiting order, then the tile-recompute walk
    const int span = local ? std::min(P.max_m, P.max_n) : (P.max_m + P.max_n) / 2;
    int* hist = perm + pairs_cap_round(pairs);          // 64 ints behind the permutation
    PSA_CUDA_OK(ctx, cudaMemsetAsync(hist, 0, 64 * sizeof(int), st));
    for (int pass = 0; pass < 2; ++pass)
        psa_pack_perm_kernel<<<(int)((pairs + 255) / 256), 256, 0, st>>>(args.items, args.len_a, args.len_b, pair0, (int)pairs,
                                                                          local ? 1 : 0, span, hist, perm, pass);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    PackWalkArgs W;
    W.P = args; W.C = P.C; W.ck = reinterpret_cast<const uint2*>(ring); W.ck_slot = P.slot_words / 2; W.ck_col = ck_col_u2(P.max_m, G);
    W.pair0 = pair0; W.pairs = pairs; W.fallback = P.flags; W.perm = perm; W.local = local;
    pack_tb_lut(P.C.h, W.lut);
    W.m_cap = P.max_m;
    const size_t smem = rwalk_smem_words(K, P.max_m, P.max_n) * 128 * sizeof(uint32_t);
    if (smem + 1024 > (size_t)ctx->smem_optin) return psa_fail(ctx, PSA_ERR_RANGE, "tile-recompute walk does not fit in shared memory");
    auto kern = psa_pack_rwalk_kernel<G, K>;
    const int orc = psa_kernel_optin_smem(ctx, (const void*)kern);
    if (orc) return orc;
    kern<<<(int)((pairs + 127) / 128), 128, smem, st>>>(W);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 3;
    return PSA_OK;
}

// Chunk c, the pairs [pair0, pair0 + pairs) of the planned batch, on stream `st`: fill, traceback walk and, for byte
// input, the generic kernel on the members the fill flagged.  fill_after / fill_done optionally order the fills of
// consecutive chunks that run on different streams (option pack_serial_fills).
int pack_chunk(psa_ctx* ctx, const PackPlan& P, int c, long long pair0, long long pairs, cudaStream_t st,
               cudaEvent_t fill_after = nullptr, cudaEvent_t fill_done = nullptr) {
    const bool bytes = P.args.a2 == nullptr;         // 2-bit input is plain ACGT: nothing can be flagged
    const bool traceback = P.flavour != TB_NONE;
    uint32_t* ring = P.rings[c % kInFlight];
    int* flag_count = (bytes && c < kCounters) ? P.counters + c : nullptr;
    PackArgs A;
    A.P = P.args; A.C = P.C; A.m_cap = P.max_m;
    A.dirs = traceback ? ring : nullptr;
    A.dirs_slot_words = P.slot_words; A.pair0 = pair0; A.pairs = pairs;
    A.fallback = P.flags;
    A.flag_count = flag_count;
    if (flag_count) PSA_CUDA_OK(ctx, cudaMemsetAsync(flag_count, 0, sizeof(int), st));
    if (fill_after) PSA_CUDA_OK(ctx, cudaStreamWaitEvent(st, fill_after, 0));
    int rc = with_shape(P.sh, [&](auto G, auto K) {
        return launch_fill<decltype(G)::value, decltype(K)::value>(ctx, A, P.mode, P.flavour, st);
    });
    if (rc) return rc;
    if (fill_done) PSA_CUDA_OK(ctx, cudaEventRecord(fill_done, st));
    // opt.pack_skip_walk: measurement hook (psa_internal.h) -- bench.py times the fill launches alone with it
    if (traceback && !ctx->opt.pack_skip_walk) {
        rc = with_shape(P.sh, [&](auto G, auto K) {
            return launch_walk<decltype(G)::value, decltype(K)::value>(ctx, P, ring, P.perms[c % kInFlight], pair0, pairs, st);
        });
        if (rc) return rc;
    }
    if (!bytes) return PSA_OK;
    // members flagged by the fill (non-ACGT bytes, zero lengths) are recomputed by the generic kernel
    psa_batch_args sub = P.args;
    sub.off_a += pair0; sub.len_a += pair0; sub.off_b += pair0; sub.len_b += pair0; sub.items += pair0;
    if (sub.ops) sub.ops += pair0 * P.args.ops_stride_words;
    sub.n_pairs = pairs;
    sub.flagged_count = flag_count;
    return psa_launch_short_flagged(ctx, sub, P.max_m, P.max_n, P.mode, traceback, P.flags + pair0, st);
}

// Plans a batch: shape, constants and traceback flavour, and the scratch in ctx->d_work (fallback flags, counters and
// kInFlight rings and perm buffers of one chunk each).
int pack_plan(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback, PackPlan& P) {
    P.args = args; P.max_m = max_m; P.max_n = max_n; P.mode = mode;
    P.flavour = !traceback ? TB_NONE : (ctx->opt.pack_traceback == 1 ? TB_CKPT : TB_CODES);
    if (!pick_shape(max_n, P.sh)) return psa_fail(ctx, PSA_ERR_RANGE, "packed kernel: n > 256");
    const int NWP = pad_words(words_for(P.sh.K));
    const int g = args.g, h = args.h;
    PackConsts& C = P.C;
    C.g = g; C.h = h;
    C.bias = (int)pack_bias(mode, g, h, max_m, max_n);
    C.ng2 = (uint32_t)((-g) & 0xffff) * 0x00010001u;
    C.go2 = (uint32_t)(g + h) * 0x00010001u;
    C.go4 = (uint32_t)(g + h) * 0x01010101u;
    C.mul32 = 32u;
    C.m1 = 0xffffffffu; C.m3 = 0xfffdfffdu;
    for (int x = 0; x < 3; ++x) {
        const uint32_t sc = x == 0 ? 1u : (x == 1 ? 32u : 1024u);
        C.cH[x] = 11u * sc; C.cT[x] = 0u - sc; C.cE[x] = 0u - 2u * sc; C.cF[x] = 0u - 8u * sc;
    }
    P.slot_words = P.flavour == TB_CKPT ? 2 * ck_slot_u2(max_m, P.sh.G, P.sh.K) : dirs_slot_words_for(max_m, P.sh.G, NWP);
    const long long chunk = std::min<long long>(ctx->opt.pack_chunk, args.n_pairs);
    const size_t ring_bytes = traceback ? ((size_t)((chunk + 1) / 2) * (size_t)P.slot_words * 4 + 255) / 256 * 256 : 0;
    const size_t perm_bytes = P.flavour == TB_CKPT ? ((size_t)(pairs_cap_round(chunk) + 64) * sizeof(int) + 255) / 256 * 256 : 0;
    const size_t o_cnt = ((size_t)args.n_pairs + 255) / 256 * 256;
    const size_t o_perm = o_cnt + kCounters * sizeof(int);
    const size_t o_d0 = o_perm + (size_t)kInFlight * perm_bytes;
    const size_t total = o_d0 + (size_t)kInFlight * ring_bytes + 256;
    if (total > ctx->d_work_bytes) {
        if (ctx->d_work) cudaFree(ctx->d_work);
        ctx->d_work = nullptr; ctx->d_work_bytes = 0;
        if (cudaMalloc(&ctx->d_work, total) != cudaSuccess) { cudaGetLastError(); return psa_fail(ctx, PSA_ERR_NOMEM, "packed kernel scratch"); }
        ctx->d_work_bytes = total;
    }
    uint8_t* d = (uint8_t*)ctx->d_work;
    P.flags = d;
    P.counters = (int*)(d + o_cnt);
    for (int k = 0; k < kInFlight; ++k) {
        P.rings[k] = (uint32_t*)(d + o_d0 + (size_t)k * ring_bytes);
        P.perms[k] = perm_bytes ? (int*)(d + o_perm + (size_t)k * perm_bytes) : nullptr;
    }
    return PSA_OK;
}

// events of one pipeline call (destroyed when the call returns, on every path)
struct EventList {
    std::vector<cudaEvent_t> ev;
    int create(psa_ctx* ctx, size_t n) {
        ev.assign(n, nullptr);
        for (auto& e : ev) PSA_CUDA_OK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        return PSA_OK;
    }
    cudaEvent_t at(size_t k) const { return k < ev.size() ? ev[k] : nullptr; }
    ~EventList() { for (auto e : ev) if (e) cudaEventDestroy(e); }
};

int psa_ensure_aux(psa_ctx* ctx) {
    if (!ctx->aux_stream[0]) {
        for (int k = 0; k < kInFlight; ++k) PSA_CUDA_OK(ctx, cudaStreamCreateWithFlags(&ctx->aux_stream[k], cudaStreamNonBlocking));
        PSA_CUDA_OK(ctx, cudaStreamCreateWithFlags(&ctx->post_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 3; ++k) PSA_CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->aux_event[k], cudaEventDisableTiming));
    }
    return PSA_OK;
}

// Chunk schedule of the host pipelines: full-size chunks in the middle, ramped down to chunk/8 at both ends -- the
// first chunk's H2D copy and the last chunk's D2H copy are the only transfers nothing overlaps.
std::vector<long long> chunk_sizes(long long chunk, long long n) {
    const long long ramp[3] = {chunk / 8, chunk / 4, chunk / 2};
    const long long ramp_sum = ramp[0] + ramp[1] + ramp[2];
    const bool ramped = n >= 2 * ramp_sum + chunk && chunk >= 8192;
    std::vector<long long> sizes;
    if (ramped) sizes.assign(ramp, ramp + 3);
    for (long long mid = ramped ? n - 2 * ramp_sum : n; mid > 0; mid -= chunk) sizes.push_back(std::min(chunk, mid));
    if (ramped) sizes.insert(sizes.end(), {ramp[2], ramp[1], ramp[0]});
    return sizes;
}

// The per-chunk steps in which the host pipelines differ.  Each gets the chunk index, its pairs [p0, p0 + cnt) and
// its stream, and returns a psa_status.
struct ChunkSteps {
    std::function<int(size_t n_chunks)> begin;                        // once, before the first chunk (may be empty)
    std::function<int(int c, long long p0, long long cnt, cudaStream_t st)> inputs, records, outputs;   // records may be empty
    bool post = false;                                                // `records` enqueues work on ctx->post_stream
};

// Host-buffer pipeline: chunk c's H2D copies, fill, traceback, records and D2H copies all go to aux stream
// c % kInFlight, so that the copies of one chunk overlap the kernels of the others.  Returns when every chunk's
// results are on the host.
int pack_pipeline(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback, const ChunkSteps& s) {
    PackPlan P;
    int rc = pack_plan(ctx, args, max_m, max_n, mode, traceback, P);
    if (rc) return rc;
    rc = psa_ensure_aux(ctx);
    if (rc) return rc;
    const std::vector<long long> sizes = chunk_sizes(ctx->opt.pack_chunk, args.n_pairs);
    EventList fills, marks;
    rc = fills.create(ctx, ctx->opt.pack_serial_fills ? sizes.size() : 0);
    if (rc) return rc;
    if (s.begin && (rc = s.begin(sizes.size()))) return rc;
    const bool tl = ctx->opt.timing >= 2;      // debugging aid: GPU-side timeline of every chunk
    auto mark = [&](cudaStream_t st) {
        if (tl) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); marks.ev.push_back(e); }
    };
    const auto t0 = std::chrono::steady_clock::now();
    long long p0 = 0;
    for (int c = 0; c < (int)sizes.size(); p0 += sizes[c], ++c) {
        cudaStream_t st = ctx->aux_stream[c % kInFlight];
        const long long cnt = sizes[c];
        mark(st);
        if ((rc = s.inputs(c, p0, cnt, st))) return rc;
        mark(st);
        if ((rc = pack_chunk(ctx, P, c, p0, cnt, st, c > 0 ? fills.at(c - 1) : nullptr, fills.at(c)))) return rc;
        mark(st);
        if (s.records && (rc = s.records(c, p0, cnt, st))) return rc;
        mark(st);
        if ((rc = s.outputs(c, p0, cnt, st))) return rc;
        mark(st);
    }
    const auto t_enq = std::chrono::steady_clock::now();
    for (int k = 0; k < kInFlight; ++k) PSA_CUDA_OK(ctx, cudaStreamSynchronize(ctx->aux_stream[k]));
    if (s.post) PSA_CUDA_OK(ctx, cudaStreamSynchronize(ctx->post_stream));
    if (tl) {
        for (size_t c = 0; c < sizes.size(); ++c) {
            float t[5];
            for (int q = 0; q < 5; ++q) cudaEventElapsedTime(&t[q], marks.ev[0], marks.ev[5 * c + q]);
            fprintf(stderr, "  chunk %2d (%6lld pairs): h2d %.3f-%.3f  fill+walk -%.3f  records -%.3f  d2h -%.3f\n", (int)c,
                    sizes[c], t[0], t[1], t[2], t[3], t[4]);
        }
    }
    if (ctx->opt.timing)
        fprintf(stderr, "psa_pack_pipeline: %d chunks enqueued in %.3f ms, drained %.3f ms later\n", (int)sizes.size(),
                std::chrono::duration<double, std::milli>(t_enq - t0).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_enq).count());
    return PSA_OK;
}

}  // namespace

// The whole device-resident batch, chunk by chunk on the kInFlight aux streams, so that the traceback of one chunk
// overlaps the fills of the others; fork / join around `user`, no host synchronisation.  Without traceback the batch
// is one chunk on `user`.
int psa_launch_pack(psa_ctx* ctx, const psa_batch_args& args, int max_m, int max_n, int mode, bool traceback,
                    cudaStream_t user) {
    PackPlan P;
    int rc = pack_plan(ctx, args, max_m, max_n, mode, traceback, P);
    if (rc) return rc;
    const long long chunk = traceback ? ctx->opt.pack_chunk : args.n_pairs;
    const bool split = args.n_pairs > chunk;
    if (split) {
        rc = psa_ensure_aux(ctx);
        if (rc) return rc;
        PSA_CUDA_OK(ctx, cudaEventRecord(ctx->aux_event[0], user));
        for (int k = 0; k < kInFlight; ++k) PSA_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->aux_stream[k], ctx->aux_event[0], 0));
    }
    int c = 0;
    for (long long p0 = 0; p0 < args.n_pairs; p0 += chunk, ++c) {
        rc = pack_chunk(ctx, P, c, p0, std::min<long long>(chunk, args.n_pairs - p0), split ? ctx->aux_stream[c % kInFlight] : user);
        if (rc) return rc;
    }
    if (split) {
        for (int k = 0; k < kInFlight; ++k) {          // join: one event, re-recorded per stream, waited on in order
            PSA_CUDA_OK(ctx, cudaEventRecord(ctx->aux_event[1], ctx->aux_stream[k]));
            PSA_CUDA_OK(ctx, cudaStreamWaitEvent(user, ctx->aux_event[1], 0));
        }
    }
    return PSA_OK;
}

// Byte input (psa_align_batch): `h` = host arrays, `args` = their device mirror (same layout).  The offsets are
// ascending and back to back, so a chunk's bases are one contiguous range.
int psa_pack_pipeline(psa_ctx* ctx, const psa_batch_args& args, const psa_batch_args& h, size_t bytes_a, size_t bytes_b,
                      int max_m, int max_n, int mode, bool traceback) {
    const long long n = args.n_pairs, stride = args.ops_stride_words;
    ChunkSteps s;
    s.inputs = [&](int, long long p0, long long cnt, cudaStream_t st) -> int {
        const long long p1 = p0 + cnt;
        const size_t a0 = (size_t)h.off_a[p0], a1 = (p1 < n) ? (size_t)h.off_a[p1] : bytes_a;
        const size_t b0 = (size_t)h.off_b[p0], b1 = (p1 < n) ? (size_t)h.off_b[p1] : bytes_b;
        if (a1 > a0) PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.bases_a + a0), h.bases_a + a0, a1 - a0, cudaMemcpyHostToDevice, st));
        if (b1 > b0) PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.bases_b + b0), h.bases_b + b0, b1 - b0, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.off_a + p0), h.off_a + p0, cnt * 8, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.off_b + p0), h.off_b + p0, cnt * 8, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.len_a + p0), h.len_a + p0, cnt * 4, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.len_b + p0), h.len_b + p0, cnt * 4, cudaMemcpyHostToDevice, st));
        return PSA_OK;
    };
    s.outputs = [&](int, long long p0, long long cnt, cudaStream_t st) -> int {
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(h.items + p0, args.items + p0, cnt * sizeof(psa_batch_item), cudaMemcpyDeviceToHost, st));
        if (traceback)
            PSA_CUDA_OK(ctx, cudaMemcpyAsync(h.ops + p0 * stride, args.ops + p0 * stride, cnt * stride * 4, cudaMemcpyDeviceToHost, st));
        return PSA_OK;
    };
    return pack_pipeline(ctx, args, max_m, max_n, mode, traceback, s);
}

// ---- 2-bit packed fixed-stride batches (psa_align_batch_packed) ------------------------------
namespace {
__global__ void __launch_bounds__(256) psa_compact_items_kernel(const psa_batch_item* in, psa_packed_item* out, long long n) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const psa_batch_item it = in[k];
    out[k] = packed_item(it);
}

// PSA_OPS_COMPACT: the op words of a chunk, back to back in pair order (pair k uses ceil(aln_len/16) words), packed on
// the device so that only the words that carry ops cross PCIe (a 150 bp read pair needs 6 - 11 of its 20-word stride).
// Two launches per chunk, one more than the fixed-stride path:
//   psa_compact_items_scan_kernel: the 40 -> 16 byte records (packed_item) + per-CTA exclusive scan of
//                                  the word counts -> offs[k] (CTA-local) and sums[cta]
//   psa_ops_pack_kernel:           every CTA adds up the sums of the scan blocks before its pairs (at most 128) and the
//                                  chunk's base (= end of the previous chunk, chained through `bases`), then one warp
//                                  per 32 pairs copies their words to dst[base + offs]; the last CTA publishes the end
//                                  of the chunk to `bases` and to the host's page-locked mirror
// Both run as 128-thread CTAs of 1 024 pairs: while fills are in flight the SMs' register files are full, and only
// CTAs as small as the walk kernels' find a slot between two fill CTAs (1 024-thread CTAs were held back until the
// whole pipeline had drained).
constexpr int SCAN_T = 1024;         // pairs per CTA
constexpr int SCAN_CT = 128;         // threads per CTA
__global__ void __launch_bounds__(SCAN_CT) psa_compact_items_scan_kernel(const psa_batch_item* in, psa_packed_item* out, int n,
                                                                         unsigned* offs, unsigned* sums) {
    __shared__ unsigned s_w[SCAN_CT / 32];
    unsigned carry = 0u;
    for (int r = 0; r < SCAN_T / SCAN_CT; ++r) {
        const int k = blockIdx.x * SCAN_T + r * SCAN_CT + threadIdx.x;
        unsigned v = 0u;
        if (k < n) {
            const psa_batch_item it = in[k];
            out[k] = packed_item(it);
            v = (unsigned)((it.aln_len + 15) >> 4);
        }
        unsigned x = v;                                     // inclusive scan inside the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= d) x += y; }
        if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = x;
        __syncthreads();
        unsigned warp_base = 0u, total = 0u;
#pragma unroll
        for (int w = 0; w < SCAN_CT / 32; ++w) { const unsigned t = s_w[w]; if (w < (int)(threadIdx.x >> 5)) warp_base += t; total += t; }
        if (k < n) offs[k] = carry + warp_base + x - v;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[blockIdx.x] = carry;
}
// A warp gathers the words of 32 pairs into shared memory and writes the contiguous range out as whole 128-byte lines --
// `dst` is the caller's page-locked buffer itself when there is one (zero-copy: the stores leave as full PCIe write
// packets, nothing is enqueued late, no host round trip for the size), else a device buffer copied out at the end.
// The grid is small on purpose (PACK_CTAS CTAs looping over the 128-pair groups): the kernel runs at PCIe speed
// whatever its size, and every CTA it keeps resident costs the fill of the next chunk a quarter of an SM.
constexpr int PACK_CTAS = 64;
__global__ void __launch_bounds__(SCAN_CT) psa_ops_pack_kernel(const psa_packed_item* items16, const uint32_t* ops, long long stride, int n,
                                                               const unsigned* offs, const unsigned* sums, int n_sums, unsigned long long* bases,
                                                               unsigned long long* h_bases, int chunk, uint32_t* dst) {
    extern __shared__ uint32_t s_words[];                    // [warps][32 * stride]
    __shared__ unsigned long long s_prefix[SCAN_CT];         // words of the scan blocks (1 024 pairs each) before block t
    const unsigned long long chunk_base = bases[chunk];
    if ((int)threadIdx.x < n_sums) {                         // n_sums <= 128 = SCAN_CT
        unsigned long long acc = 0ull;
        for (int j = 0; j < (int)threadIdx.x; ++j) acc += sums[j];
        s_prefix[threadIdx.x] = acc;
        if ((int)threadIdx.x == n_sums - 1 && blockIdx.x == 0) {
            const unsigned long long end = chunk_base + acc + sums[threadIdx.x];
            bases[chunk + 1] = end;
            *reinterpret_cast<volatile unsigned long long*>(h_bases + chunk + 1) = end;
            __threadfence_system();
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* sw = s_words + (size_t)warp * 32 * stride;
    for (int grp = blockIdx.x; grp * SCAN_CT < n; grp += gridDim.x) {
        const int k0 = grp * SCAN_CT + warp * 32;
        if (k0 >= n) break;
        const unsigned long long base = chunk_base + s_prefix[(grp * SCAN_CT) / SCAN_T];
        // lane i holds pair i's word count and offset, the warp copies pair after pair
        const int kl = k0 + lane;
        const int my_words = kl < n ? (items16[kl].aln_len + 15) >> 4 : 0;
        const unsigned my_off = kl < n ? offs[kl] : 0u;
        const unsigned off0 = __shfl_sync(0xffffffffu, my_off, 0);
        const int last_lane = min(31, n - 1 - k0);                                             // the warp's last pair that exists
        const unsigned total = __shfl_sync(0xffffffffu, my_off + (unsigned)my_words, last_lane) - off0;
#pragma unroll 8
        for (int i = 0; i < 32; ++i) {
            const int words = __shfl_sync(0xffffffffu, my_words, i);
            const unsigned rel = __shfl_sync(0xffffffffu, my_off, i) - off0;
            const uint32_t* src = ops + (long long)(k0 + i) * stride;
            for (int w = lane; w < words; w += 32) sw[rel + w] = src[w];
        }
        __syncwarp();
        const unsigned long long g0 = base + off0, g1 = g0 + total;
        for (unsigned long long gw = (g0 & ~31ull) + lane; gw < g1; gw += 32)
            if (gw >= g0) dst[gw] = sw[gw - g0];
        __syncwarp();
    }
}
}  // namespace

// 2-bit input (psa_align_batch_packed): per chunk H2D of the two packed read arrays (fixed stride: one contiguous range
// each, no offsets or lengths), fill + traceback, 40 -> 16 byte result records, D2H of records and op words.  `args` =
// device mirror (a2/b2/items/ops device pointers).
int psa_pack_pipeline_packed(psa_ctx* ctx, const psa_batch_args& args, const uint32_t* h_a2, const uint32_t* h_b2,
                             psa_packed_item* d_items16, psa_packed_item* h_items16, uint32_t* h_ops, int mode, bool traceback,
                             bool compact, uint8_t* d_compact /* scan scratch | bases | (staging buffer) */) {
    const long long stride = args.ops_stride_words;
    // compact ops: the GPU packs each chunk's words back to back -- straight into the caller's buffer when that is
    // page-locked (zero-copy, whole 128-byte lines), else into a device buffer that is copied out once at the end
    compact = compact && traceback;
    unsigned* d_offs = nullptr; unsigned* d_sums = nullptr; unsigned long long* d_bases = nullptr;
    uint32_t* d_stage = nullptr;
    uint32_t* cdst = nullptr;
    bool zero_copy = false;
    unsigned long long* h_bases = nullptr;
    unsigned long long* dh_bases = nullptr;
    size_t n_chunks = 0;
    EventList chain;
    const size_t pack_smem = (size_t)(SCAN_CT / 32) * 32 * stride * 4;
    ChunkSteps s;
    s.post = compact;
    s.begin = [&](size_t nc) -> int {
        n_chunks = nc;
        if (!compact) return PSA_OK;
        if (nc + 1 > 4096) return psa_fail(ctx, PSA_ERR_RANGE, "compact ops: too many chunks");
        if (pack_smem > 48 * 1024) return psa_fail(ctx, PSA_ERR_RANGE, "compact ops: ops_stride_words too large");
        const size_t n_up = ((size_t)args.n_pairs + 255) / 256 * 256;
        d_offs = (unsigned*)d_compact;
        d_sums = (unsigned*)(d_compact + n_up * 4);                              // [chunks][128] scan-block sums
        d_bases = (unsigned long long*)(d_compact + n_up * 4 + 4096 * 128 * 4);
        d_stage = (uint32_t*)(d_compact + n_up * 4 + 4096 * 128 * 4 + 4096 * 8 + 256);
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, h_ops) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer != nullptr) {
            zero_copy = true; cdst = (uint32_t*)pa.devicePointer;
        } else { cudaGetLastError(); cdst = d_stage; }
        if (ctx->h_pinned_bytes < 4096 * 8) {               // page-locked mirror of the chunk ends (the total, for the caller)
            if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
            ctx->h_pinned = nullptr; ctx->h_pinned_bytes = 0;
            PSA_CUDA_OK(ctx, cudaHostAlloc(&ctx->h_pinned, 4096 * 8, cudaHostAllocMapped | cudaHostAllocPortable));
            ctx->h_pinned_bytes = 4096 * 8;
        }
        h_bases = (unsigned long long*)ctx->h_pinned;
        h_bases[0] = 0;
        PSA_CUDA_OK(ctx, cudaHostGetDevicePointer((void**)&dh_bases, ctx->h_pinned, 0));    // the GPU's view of the mirror
        PSA_CUDA_OK(ctx, cudaMemsetAsync(d_bases, 0, 8, ctx->post_stream));
        return chain.create(ctx, nc);
    };
    s.inputs = [&](int, long long p0, long long cnt, cudaStream_t st) -> int {
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.a2 + p0 * args.wa), h_a2 + p0 * args.wa, (size_t)cnt * args.wa * 4, cudaMemcpyHostToDevice, st));
        PSA_CUDA_OK(ctx, cudaMemcpyAsync((void*)(args.b2 + p0 * args.wb), h_b2 + p0 * args.wb, (size_t)cnt * args.wb * 4, cudaMemcpyHostToDevice, st));
        return PSA_OK;
    };
    s.records = [&](int c, long long p0, long long cnt, cudaStream_t st) -> int {
        const int n_cta = (int)((cnt + SCAN_T - 1) / SCAN_T);
        if (compact) {
            if (n_cta > 128) return psa_fail(ctx, PSA_ERR_RANGE, "compact ops: chunk larger than 131 072 pairs");
            psa_compact_items_scan_kernel<<<n_cta, SCAN_CT, 0, st>>>(args.items + p0, d_items16 + p0, (int)cnt, d_offs + p0, d_sums + (size_t)c * 128);
        } else {
            psa_compact_items_kernel<<<(int)((cnt + 255) / 256), 256, 0, st>>>(args.items + p0, d_items16 + p0, cnt);
        }
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
        if (!compact) return PSA_OK;
        // The packing runs on a stream of its own, chunk after chunk (a chunk's base is the end of the previous one):
        // chained inside the fill streams it made every later fill wait for the walks of ALL earlier chunks.
        PSA_CUDA_OK(ctx, cudaEventRecord(chain.ev[c], st));
        PSA_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->post_stream, chain.ev[c], 0));
        psa_ops_pack_kernel<<<(int)std::min<long long>((cnt + SCAN_CT - 1) / SCAN_CT, PACK_CTAS), SCAN_CT, pack_smem, ctx->post_stream>>>(
            d_items16 + p0, args.ops + p0 * stride, stride, (int)cnt, d_offs + p0, d_sums + (size_t)c * 128, n_cta, d_bases,
            dh_bases, c, cdst);
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
        return PSA_OK;
    };
    s.outputs = [&](int, long long p0, long long cnt, cudaStream_t st) -> int {
        PSA_CUDA_OK(ctx, cudaMemcpyAsync(h_items16 + p0, d_items16 + p0, (size_t)cnt * sizeof(psa_packed_item), cudaMemcpyDeviceToHost, st));
        if (traceback && !compact)
            PSA_CUDA_OK(ctx, cudaMemcpyAsync(h_ops + p0 * stride, args.ops + p0 * stride, (size_t)cnt * stride * 4, cudaMemcpyDeviceToHost, st));
        return PSA_OK;
    };
    const int rc = pack_pipeline(ctx, args, args.fixed_m, args.fixed_n, mode, traceback, s);
    if (rc || !compact) return rc;
    const unsigned long long total = h_bases[n_chunks];
    if (!zero_copy && total) PSA_CUDA_OK(ctx, cudaMemcpy(h_ops, d_stage, (size_t)total * 4, cudaMemcpyDeviceToHost));
    return PSA_OK;
}
