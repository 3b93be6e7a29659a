// psa_systolic.cu -- column-stationary systolic wavefront for ONE long pair, score only
// (BASELINE config 4: 1 Mbp x 1 Mbp local score, one GPU or block-cyclic panels over several).
//
// A warp owns a strip of 32*KC columns for ALL m rows: lane t owns KC columns, the lanes sweep the rows as a skewed
// wavefront (the chain value of the column to the left arrives from lane t-1 by shuffle).  Adjacent strips are
// chained through small rings of 8-byte entries in L2; a panel = all strips resident on the GPU at once, so the
// whole panel advances as ONE anti-diagonal wavefront whose critical path is m + (lag per strip) * strips lane
// steps -- no per-tile drain (the row-block kernel of psa_long.cu pays (m/R + n/W) tile sweeps).  What makes a step
// cheap here (the round-1 panel kernel needed 412 ns per row, this one ~50):
//   * in-band validity: a ring entry carries a 1-bit lap tag in its spare top bit and is written with ONE 8-byte
//     store -- no flag word, no fence, no release/acquire pair.  The consumer prefetches a 32-row block one block
//     ahead and only spins if a tag is still the previous lap's;
//   * rows are numbered cumulatively across calls (per-ring totals kept in device memory), so a ring never needs
//     clearing and consecutive calls / panels flow through it back to back;
//   * back-pressure by a consumed-rows counter the producer re-reads only when its ring is about to wrap;
//   * a one-instruction E chain: with TF = max(T1, F) - (g+h) (both known from the previous row),
//     E[j] = max(E[j-1] - g, TF[j-1]) -- one VIADDMNMX per cell on the row's dependency chain instead of
//     VIADDMNMX -> VIMNMX3 -> IADD; lanes hand over (TF, E) of their last column, so the lane boundary is one more
//     link of the same chain.
// Across GPUs the panels are dealt out block-cyclically (panel q -> rank q mod G): the last strip of a panel
// stores its entries straight into the next rank's ring over NVLink (peer-mapped pointer, system-scope stores);
// every GPU is busy on its own panel while the wavefront runs through all of them.
//
// Recurrence and borders as everywhere else (subproblem_alignment.cpp:229-292; psa_tile.cuh for the derivation);
// local end cell by the packed key T1*KM + (KM-1-k); global corner T1/T2/T3[m][n] captured by the owning lane.
#include <type_traits>

#include "psa_tile.cuh"

using namespace psa_tile;

namespace {

constexpr int SWPB = 4;              // warps (strips) per CTA
constexpr int RING = 1024;           // rows per ring between two strips of a panel (power of two)
constexpr int VBIAS = 1 << 30;       // entry word 0 = (TF + VBIAS) | tag << 31

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p, bool sys) {
    unsigned long long v;
    if (sys) asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    else asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v, bool sys) {
    if (sys) asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
    else asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned* p, bool sys) {
    unsigned v;
    if (sys) asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    else asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(unsigned* p, unsigned v, bool sys) {
    if (sys) asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
    else asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// One boundary between a producer strip and a consumer strip.  Rows are numbered cumulatively over the life of the
// buffer: row R lives in slot R % cap and carries tag ((R / cap) + 1) & 1 (fresh memory is all zero = tag 0 = never
// valid on the first lap).  prod_total / cons_total are private to their side; consumed_pub is the consumer's
// progress as the producer sees it.
struct Boundary {
    unsigned long long* slots;
    unsigned cap;              // rows
    unsigned* prod_total;      // producer side: rows written by all earlier launches
    unsigned* cons_total;      // consumer side: rows read by all earlier launches
    unsigned* consumed_pub;    // written by the consumer, polled by the producer when the ring is about to wrap
    int sys;                   // 1: the two sides are different GPUs (system-scope accesses)
};

struct SysJob {
    const uint8_t* a;
    const uint8_t* b;          // the WHOLE sequence B (global column j is b[j-1])
    int m, g, h;
    int col_begin;             // global index of the column left of the panel
    int n_cols;                // columns in this panel
    int n_total;
    int nstrips;
    int has_in, has_out;       // panel edges: 0 = matrix column 0 / nobody needs the right edge
    Boundary in, out;
    // rings between adjacent strips of the panel: ring w sits between strip w and strip w + 1
    unsigned long long* rings; // [nstrips][RING]
    unsigned* r_prod;          // [nstrips]
    unsigned* r_cons;
    unsigned* r_pub;
    unsigned long long* best;
    int* corner;
};

__device__ __forceinline__ unsigned long long pack_entry(int tf, int e, unsigned tag) {
    return (unsigned long long)(((unsigned)(tf + VBIAS)) | (tag << 31)) | ((unsigned long long)(unsigned)e << 32);
}

// One lane-step: the KC cells of one row.  H and T1 live in the "minus (g+h)" domain, E and F do not:
//   hg[k]  = H[i-1][j] - go      ff[k] = F[i-1][j]
//   tf_in / e_in: TF = max(T1, F) - go and E of the column to the left, this row
// Every recurrence is ONE VIADDMNMX: F = max(F' - g, H' - go) = viaddmax(ff, -g, hg);  TF = max(F - go, T1 - go) =
// viaddmax(F, -go, t1g);  E = viaddmax(E, -g, TF_left);  H - go = max(E - go, TF) = viaddmax(E, -go, TF).
// Out: tf_in / e_in of this lane's last column (for the next lane), rowkey (local).
template <int KC, bool LOCAL, bool CAP>
__device__ __forceinline__ void sys_step(int (&hg)[KC], int (&ff)[KC], const int (&b)[KC], const int (&ka)[KC],
                                         int& tf_in, int& e_in, int diag_hg, int a, int ng, int ngo, int km, int& rowkey,
                                         int kcap, int go, int& c1, int& c2, int& c3) {
    int t1g[KC], tfn[KC];
    // everything that depends only on the previous row first (off the E chain)
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        t1g[k] = (k == 0 ? diag_hg : hg[k - 1]) + (a == b[k] ? 1 : 0);        // T1 - go
        ff[k] = __viaddmax_s32(ff[k], ng, hg[k]);                            // F = max(F' - g, H' - go)
        tfn[k] = __viaddmax_s32(ff[k], ngo, t1g[k]);                         // TF = max(F, T1) - go
    }
    int key_prev = 0;
    int e = e_in, tf = tf_in;
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        e = __viaddmax_s32(e, ng, tf);                    // E[j] = max(E[j-1] - g, TF[j-1])     <- the only op on the chain
        tf = tfn[k];
        const int hgk = __viaddmax_s32(e, ngo, tf);       // H - go = max(E - go, TF)
        if (LOCAL) {
            const int key = t1g[k] * km + ka[k];
            if (k & 1) rowkey = __vimax3_s32(rowkey, key_prev, key);
            key_prev = key;
        }
        if (CAP) { if (k == kcap) { c1 = t1g[k] + go; c2 = e; c3 = ff[k]; } }
        hg[k] = hgk;
    }
    tf_in = tf; e_in = e;
}

__device__ __forceinline__ void st_relaxed_2xu64(unsigned long long* p, unsigned long long v0, unsigned long long v1, bool sys) {
    // two ring entries with one instruction; each 64-bit element is written atomically (aligned), which is all the tag needs
    if (sys) asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(v0), "l"(v1) : "memory");
    else asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(v0), "l"(v1) : "memory");
}

// RB rows x KC columns per lane and step: the per-step overhead (shuffles, boundary hand-over, loop control) is shared by
// RB*KC cells and the RB + KC - 1 anti-diagonals of the block give a lone warp the instruction-level parallelism a
// one-row step lacks.  Lane t works on row block s - t at step s; row counts are padded to a multiple of 4
// (padding rows never reach the result: their keys are masked, the corner is captured on row m).
template <int MODE, int KC, int RB>
__global__ void __launch_bounds__(SWPB * 32) psa_systolic_kernel(SysJob J) {
    constexpr bool LOCAL = (MODE == PSA_LOCAL);
    constexpr int W = 32 * KC, KM = key_mult(KC);
    static_assert(KC % 2 == 0, "the row key folds two cells per VIMNMX3");
    static_assert(RB == 1 || RB == 2 || RB == 4, "row characters of a block travel in one 32-bit word");
    __shared__ unsigned long long s_in[SWPB][2][32];          // the consumer's current / next 32-row block
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sidx = blockIdx.x * SWPB + wib;
    if (sidx >= J.nstrips) return;
    const int m = J.m, g = J.g, h = J.h, go = g + h, ng = -g, ngo = -go;
    // Padded rows: a multiple of 4 for every RB, the same count the ring totals advance by below.  Each ring row of
    // this launch must be written: a slot a lap skips still holds the tag of two laps back, which is the tag the next
    // lap waits for, so the consumer takes a stale entry as valid if it reads the slot before the producer rewrites it
    // (with rows padded to RB only, a 1-row launch at m = 5 skipped rows 5-7, and a later call on the same context
    // whose rows reached those slots one lap on could return a wrong corner).
    const int mp = (m + 3) & ~3;
    const int nblk = mp / RB;
    const int c0 = sidx * W + lane * KC;                  // panel-local 0-based first column of this lane
    const int cg = J.col_begin + c0;                      // global index of the column left of it
    const bool first = (sidx == 0), last = (sidx == J.nstrips - 1);

    // ---- boundaries of this strip ----
    Boundary bin, bout;
    const bool use_in = !first || J.has_in, use_out = !last || J.has_out;
    if (first) bin = J.in;
    else { bin.slots = J.rings + (size_t)(sidx - 1) * RING; bin.cap = RING; bin.prod_total = J.r_prod + sidx - 1;
           bin.cons_total = J.r_cons + sidx - 1; bin.consumed_pub = J.r_pub + sidx - 1; bin.sys = 0; }
    if (last) bout = J.out;
    else { bout.slots = J.rings + (size_t)sidx * RING; bout.cap = RING; bout.prod_total = J.r_prod + sidx;
           bout.cons_total = J.r_cons + sidx; bout.consumed_pub = J.r_pub + sidx; bout.sys = 0; }
    const bool in_sys = use_in && bin.sys, out_sys = use_out && bout.sys;
    // consumer cursor: slot / lap of the row this LANE loads next (row = 32-row block base + lane)
    unsigned cons_base = 0, in_slot = 0, in_lap = 0;
    if (use_in) {
        cons_base = *bin.cons_total;
        const unsigned r0 = cons_base + (unsigned)lane;
        in_slot = r0 % bin.cap; in_lap = r0 / bin.cap;
    }
    // producer cursor (lane 31 writes RB entries per step; totals are multiples of 4, so RB entries never straddle the wrap)
    unsigned prod_base = 0, out_slot = 0, out_lap = 0;
    int out_limit = 0x7fffffff;                           // rows (of this launch) lane 31 may write before re-reading consumed_pub
    if (use_out) {
        prod_base = *bout.prod_total;
        out_slot = prod_base % bout.cap; out_lap = prod_base / bout.cap;
        out_limit = (int)(ld_relaxed_u32(bout.consumed_pub, out_sys) - prod_base) + (int)bout.cap;
    }

    // ---- column state (row 0: subproblem_alignment.cpp:222-224) ----
    int hg[KC], ff[KC], b[KC], ka[KC];
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        const int jl = c0 + k;
        const bool valid = jl < J.n_cols;
        b[k] = valid ? (int)J.b[cg + k] : 256;
        const int H0 = valid ? border_row0_H<MODE>(cg + k + 1, g, h) : (LOCAL ? 0 : PSA_KNEG);
        hg[k] = H0 - go; ff[k] = PSA_KNEG;
        ka[k] = valid ? (KM - 1 - k) : -(1 << 30);
    }
    int diag_hg = border_row0_H<MODE>(cg, g, h) - go;     // H[0][cg] - go
    int recv_tf[RB], recv_e[RB];
#pragma unroll
    for (int q = 0; q < RB; ++q) { recv_tf[q] = PSA_KNEG; recv_e[q] = PSA_KNEG; }
    int bestkey = -(1 << 30), besti = 0;
    int c1 = PSA_KNEG, c2 = PSA_KNEG, c3 = PSA_KNEG;
    const int kcap = (!LOCAL && J.n_total > cg && J.n_total <= cg + KC) ? (J.n_total - 1 - cg) : -1;

    // first block of the left boundary in flight
    unsigned long long nxt = 0ull;
    if (use_in && lane < mp) nxt = ld_relaxed_u64(bin.slots + in_slot, in_sys);
    // row characters of a block: RB bytes in one word (rows past m read as 0: no match with any column)
    auto load_chars = [&](int blk) -> uint32_t {
        uint32_t w = 0;
        const int r0 = blk * RB;
        if (RB == 4 && r0 + 4 <= m) return *reinterpret_cast<const uint32_t*>(J.a + r0);      // a is 4-byte aligned (checked by the launcher)
#pragma unroll
        for (int q = 0; q < RB; ++q) if (r0 + q < m) w |= (uint32_t)J.a[r0 + q] << (8 * q);
        return w;
    };
    uint32_t aw_next = (lane == 0) ? load_chars(0) : 0u;

    const int steps = nblk + 31;
    // One step.  STEADY = every lane has a full row block inside the matrix (no range checks, no row masks, no corner
    // capture, aligned character words): the body is one straight-line block the scheduler can interleave across rows.
    auto step = [&](int st, auto steady_c) {
        constexpr bool STEADY = decltype(steady_c)::value;
        const int row0 = st * RB;                         // first row lane 0 works on at this step
        // ---- every 32 rows of lane 0: the next 32 rows of the left boundary (lane L <- row row0 + L) ----
        if ((row0 & 31) == 0 && row0 < mp) {
            if (use_in) {
                const int row = row0 + lane;
                const unsigned want = (in_lap + 1u) & 1u;
                for (;;) {
                    const bool ok = row >= mp || (unsigned)((nxt >> 31) & 1ull) == want;
                    if (__all_sync(0xffffffffu, ok)) break;
                    if (!ok) nxt = ld_relaxed_u64(bin.slots + in_slot, in_sys);
                }
                s_in[wib][(row0 >> 5) & 1][lane] = nxt;
                // rows < row0 are consumed: tell the producer (relaxed: it only gates slot reuse, and the entries of those
                // rows were read into registers a block ago)
                if (lane == 0 && row0 > 0) st_relaxed_u32(bin.consumed_pub, cons_base + (unsigned)row0, in_sys);
                // prefetch the block after this one
                in_slot += 32; if (in_slot >= bin.cap) { in_slot -= bin.cap; in_lap += 1; }
                if (row + 32 < mp) nxt = ld_relaxed_u64(bin.slots + in_slot, in_sys);
            } else {
                const int i = row0 + lane + 1;            // matrix column 0 (cpp:282-292): TF = H[i][0] - go, E = -inf
                s_in[wib][(row0 >> 5) & 1][lane] = pack_entry(border_col0_H<MODE>(i, g, h) - go, PSA_KNEG, 0u);
            }
            __syncwarp();
        }
        // ---- ring space for the rows lane 31 writes at this step (block st - 31) ----
        if (use_out && (st - 31) * RB + RB > out_limit) {
            unsigned ns = 64;
            for (;;) {                                    // every lane polls the same word: the warp stays converged
                out_limit = (int)(ld_relaxed_u32(bout.consumed_pub, out_sys) - prod_base) + (int)bout.cap;
                if ((st - 31) * RB + RB <= out_limit) break;
                __nanosleep(ns); if (ns < 2048) ns <<= 1;
            }
        }
        const int blk = st - lane;
        int tf_io[RB], e_io[RB];
        {
            // lane 0 takes its input from the staged block; the load is unconditional (every lane reads the same words)
            const unsigned long long* sp = &s_in[wib][(row0 >> 5) & 1][row0 & 31];
#pragma unroll
            for (int q = 0; q < RB; ++q) {
                const unsigned long long ent = sp[q];
                const int tfs = (int)((unsigned)ent & 0x7fffffffu) - VBIAS, es = (int)(unsigned)(ent >> 32);
                tf_io[q] = lane == 0 ? tfs : recv_tf[q];
                e_io[q] = lane == 0 ? es : recv_e[q];
            }
        }
        const bool active = STEADY || (blk >= 0 && blk < nblk);
        if (active) {
            const uint32_t aw = aw_next;
            if (STEADY) aw_next = *reinterpret_cast<const uint32_t*>(J.a + (blk + 1) * RB);    // RB == 4 in the steady phase
            else if (blk + 1 < nblk) aw_next = load_chars(blk + 1);
            const int r0 = blk * RB;
#pragma unroll
            for (int q = 0; q < RB; ++q) {
                const int a = (int)((aw >> (8 * q)) & 0xffu);
                const int hg_left = __viaddmax_s32(e_io[q], ngo, tf_io[q]);      // H[row][c0] - go: next row's diagonal
                int rowkey = -(1 << 30);
                if (!STEADY && !LOCAL && r0 + q == m - 1 && kcap >= 0)
                    sys_step<KC, LOCAL, true>(hg, ff, b, ka, tf_io[q], e_io[q], diag_hg, a, ng, ngo, KM, rowkey, kcap, go, c1, c2, c3);
                else
                    sys_step<KC, LOCAL, false>(hg, ff, b, ka, tf_io[q], e_io[q], diag_hg, a, ng, ngo, KM, rowkey, -1, go, c1, c2, c3);
                diag_hg = hg_left;
                if (LOCAL) {
                    const bool up = rowkey > (bestkey | (KM - 1)) && (STEADY || r0 + q < m);
                    bestkey = up ? rowkey : bestkey;
                    besti = up ? (r0 + q + 1) : besti;
                }
            }
        } else if (blk == -1) {
            aw_next = load_chars(0);                      // this lane's first row block is next
        }
#pragma unroll
        for (int q = 0; q < RB; ++q) {
            recv_tf[q] = __shfl_up_sync(0xffffffffu, tf_io[q], 1);
            recv_e[q] = __shfl_up_sync(0xffffffffu, e_io[q], 1);
        }
        if (lane == 31 && use_out && active) {
            const unsigned tag = (out_lap + 1u) & 1u;
            if (RB == 1) st_relaxed_u64(bout.slots + out_slot, pack_entry(tf_io[0], e_io[0], tag), out_sys);
            else {
#pragma unroll
                for (int q = 0; q < RB; q += 2)
                    st_relaxed_2xu64(bout.slots + out_slot + q, pack_entry(tf_io[q], e_io[q], tag),
                                     pack_entry(tf_io[q + 1 < RB ? q + 1 : q], e_io[q + 1 < RB ? q + 1 : q], tag), out_sys);
            }
            out_slot += RB; if (out_slot >= bout.cap) { out_slot = 0; out_lap += 1; }
        }
    };
    {
        int st = 0;
        // steady phase: every lane's block and the block whose characters it prefetches are full 4-row blocks inside the matrix
        const int steady_end = (RB == 4) ? (m / RB - 1) : 0;
        for (; st < steps && st < 31; ++st) step(st, std::false_type{});
        for (; st < steady_end; ++st) step(st, std::true_type{});
        for (; st < steps; ++st) step(st, std::false_type{});
    }
    // ---- totals for the next launch that uses these boundaries (padded to 4 rows so that entry pairs stay aligned) ----
    const unsigned adv = (unsigned)mp;
    if (use_in && lane == 0) { st_relaxed_u32(bin.consumed_pub, cons_base + adv, in_sys); *bin.cons_total = cons_base + adv; }
    if (use_out && lane == 31) *bout.prod_total = prod_base + adv;

    if (LOCAL) {
        // bestkey = (T1 - go) * KM + (KM - 1 - k)
        int t1v = 0, kk = 0;
        if (bestkey > -(1 << 29)) {
            const int q = (bestkey >= 0) ? bestkey / KM : -((-bestkey + KM - 1) / KM);   // floor division
            kk = KM - 1 - (bestkey - q * KM);
            t1v = q + go;
        }
        const int j = cg + kk + 1;
        unsigned long long key = 0ull;
        if (t1v > 0 && j <= J.n_total)
            key = best_key(t1v, besti, j);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, key, off);
            key = o > key ? o : key;
        }
        if (lane == 0 && key != 0ull) atomicMax(J.best, key);
    } else if (kcap >= 0) {
        J.corner[0] = c1; J.corner[1] = c2; J.corner[2] = c3;
    }
}

// Result record of a systolic run: the local best / the global corner accumulated by the panel launches.
__global__ void psa_systolic_result_kernel(const unsigned long long* best, const int* corner, int mode, int m, int n_total,
                                           int has_corner, psa_batch_item* item) {
    if (mode == PSA_LOCAL) { *item = local_item_from_key(*best); return; }
    const int c1 = has_corner ? corner[0] : PSA_KNEG, c2 = has_corner ? corner[1] : PSA_KNEG, c3 = has_corner ? corner[2] : PSA_KNEG;
    *item = global_item(c1, c2, c3, m, n_total, 0, -1);      // untyped: h is not read
}

struct SysLayout {
    size_t o_rings, o_prod, o_cons, o_pub, o_self[2], o_selfctr[2], o_xprod, o_misc, total;
};
SysLayout sys_layout(int strips, size_t self_rows) {
    auto up = [](size_t x) { return (x + 255) / 256 * 256; };
    SysLayout L;
    size_t o = 0;
    L.o_rings = o; o += up((size_t)strips * RING * 8);
    L.o_prod = o; o += up((size_t)strips * 4);
    L.o_cons = o; o += up((size_t)strips * 4);
    L.o_pub = o; o += up((size_t)strips * 4);
    for (int k = 0; k < 2; ++k) { L.o_self[k] = o; o += up(self_rows * 8); }
    for (int k = 0; k < 2; ++k) { L.o_selfctr[k] = o; o += 256; }       // prod_total @0, cons_total @64, consumed_pub @128
    L.o_xprod = o; o += 256;                                            // prod_total of the outgoing inter-GPU ring
    L.o_misc = o; o += 256;                                             // best @0, corner @16
    L.total = o;
    return L;
}

}  // namespace

// Rows of the boundary buffer between two GPUs.  It must hold a WHOLE column (>= m rows): a rank's consecutive panels
// run one after the other, so the panel feeding rank r's NEXT panel has to be able to finish before that one starts
// (a shorter ring deadlocks as soon as a rank owns more than one panel).  Power of two: see ensure_sys.
static unsigned xbuf_rows(size_t m_cap) {
    unsigned r = 8192;
    while ((size_t)r < m_cap) r <<= 1;
    return r;
}
size_t psa_systolic_xbuf_bytes(size_t m_cap) { return 256 + (size_t)xbuf_rows(m_cap) * 8; }

int psa_systolic_capacity(psa_ctx* ctx) {
    const int wpsm = ctx->opt.systolic_warps_per_sm > 0 ? ctx->opt.systolic_warps_per_sm : 8;
    return std::max(SWPB, wpsm / SWPB * SWPB) * ctx->sm_count;
}

// Persistent state of the systolic kernel (rings and their cumulative row counters must survive between launches;
// a fresh or regrown allocation starts from all-zero, which is a consistent state).
static int ensure_sys(psa_ctx* ctx, int strips, size_t self_rows, SysLayout* L) {
    // capacities are powers of two so that the cumulative row numbering survives the wrap of its 32-bit counters
    // and at least 32: a launch writes its rows padded to 4, and the producer waits while they exceed the capacity (the
    // consumer of a self boundary is the next panel's launch, so at m = 1 or 2 a 1- or 2-row buffer never drained)
    size_t pow2 = 32;
    while (pow2 < self_rows) pow2 <<= 1;
    self_rows = pow2;
    const bool fits = ctx->d_sys != nullptr && strips <= ctx->sys_strips && self_rows <= ctx->sys_self_rows;
    if (!fits) {
        if (ctx->d_sys) cudaFree(ctx->d_sys);
        ctx->d_sys = nullptr;
        const int s2 = std::max(strips, ctx->sys_strips);
        const size_t r2 = std::max(self_rows, ctx->sys_self_rows);
        const SysLayout L2 = sys_layout(s2, r2);
        if (cudaMalloc(&ctx->d_sys, L2.total) != cudaSuccess) {
            cudaGetLastError();
            ctx->sys_strips = 0; ctx->sys_self_rows = 0;
            return psa_fail(ctx, PSA_ERR_NOMEM, "systolic kernel state (" + std::to_string(L2.total >> 20) + " MiB)");
        }
        PSA_CUDA_OK(ctx, cudaMemset(ctx->d_sys, 0, L2.total));
        ctx->sys_strips = s2; ctx->sys_self_rows = r2;
    }
    *L = sys_layout(ctx->sys_strips, ctx->sys_self_rows);
    return PSA_OK;
}

// The panels `first_panel, first_panel + panel_step, ...` of one pair; panel q covers the global columns
// [q*PW, min((q+1)*PW, n_total)), PW = panel_strips * 32 * KC.  xin / xout: inter-GPU rings (this GPU's incoming
// buffer, the next GPU's incoming buffer peer-mapped) -- both null on a single GPU, where consecutive panels hand
// over through two full-length local buffers instead.
int psa_launch_systolic(psa_ctx* ctx, const uint8_t* d_a, const uint8_t* d_b, int m, int n_total, int mode, int g, int h,
                        int first_panel, int panel_step, int panel_strips, void* xin, void* xout, size_t x_m_cap,
                        psa_batch_item* d_item, cudaStream_t st) {
    if (m <= 0 || n_total <= 0) return psa_fail(ctx, PSA_ERR_ARG, "systolic path needs m, n >= 1");
    if (m >= 0x1FFFFF || n_total >= 0x1FFFFF) return psa_fail(ctx, PSA_ERR_RANGE, "long path: lengths must be < 2^21 - 1");
    const int KC = ctx->opt.systolic_kc == 4 ? 4 : 8;        // = psa_long_strip_columns() / 32
    int RB = ctx->opt.systolic_rb;
    if (RB != 1 && RB != 2 && RB != 4) RB = 4;
    if (RB == 4 && ((uintptr_t)d_a & 3u)) RB = 2;          // the 4-row step reads the row characters as aligned words
    const int W = 32 * KC;
    const int cap = psa_systolic_capacity(ctx);
    if (panel_strips <= 0) panel_strips = cap;
    if (panel_strips > cap) return psa_fail(ctx, PSA_ERR_RANGE, "panel wider than the resident strip capacity");
    const long long PW = (long long)panel_strips * W;
    const int npanels = (int)((n_total + PW - 1) / PW);
    const bool multi = (xin != nullptr || xout != nullptr || panel_step > 1);
    if (multi && (size_t)m > x_m_cap) return psa_fail(ctx, PSA_ERR_ARG, "m exceeds the row capacity the inter-GPU buffers were created with");
    SysLayout L;
    int rc = ensure_sys(ctx, panel_strips, multi ? 1 : (size_t)m, &L);
    if (rc) return rc;
    uint8_t* d = (uint8_t*)ctx->d_sys;
    PSA_CUDA_OK(ctx, cudaMemsetAsync(d + L.o_misc, 0, 64, st));
    SysJob J;
    J.a = d_a; J.b = d_b; J.m = m; J.g = g; J.h = h; J.n_total = n_total;
    J.rings = (unsigned long long*)(d + L.o_rings);
    J.r_prod = (unsigned*)(d + L.o_prod); J.r_cons = (unsigned*)(d + L.o_cons); J.r_pub = (unsigned*)(d + L.o_pub);
    J.best = (unsigned long long*)(d + L.o_misc);
    J.corner = (int*)(d + L.o_misc + 16);
    auto self_boundary = [&](int k) {
        Boundary B;
        B.slots = (unsigned long long*)(d + L.o_self[k]); B.cap = (unsigned)ctx->sys_self_rows;
        B.prod_total = (unsigned*)(d + L.o_selfctr[k]); B.cons_total = (unsigned*)(d + L.o_selfctr[k] + 64);
        B.consumed_pub = (unsigned*)(d + L.o_selfctr[k] + 128); B.sys = 0;
        return B;
    };
    auto x_boundary = [&](void* x, bool producer_side) {
        Boundary B;
        uint8_t* p = (uint8_t*)x;
        B.slots = (unsigned long long*)(p + 256); B.cap = xbuf_rows(x_m_cap);
        B.prod_total = producer_side ? (unsigned*)(d + L.o_xprod) : nullptr;
        B.cons_total = (unsigned*)p;                       // consumer-private (only the consumer side dereferences it)
        B.consumed_pub = (unsigned*)(p + 64); B.sys = 1;
        return B;
    };
    int has_corner = 0, launched = 0;
    for (int q = first_panel; q < npanels; q += panel_step, ++launched) {
        J.col_begin = (int)(q * PW);
        J.n_cols = (int)std::min<long long>(PW, n_total - q * PW);
        J.nstrips = (J.n_cols + W - 1) / W;
        J.has_in = q > 0; J.has_out = q + 1 < npanels;
        if (J.has_in) { if (multi && !xin) return psa_fail(ctx, PSA_ERR_ARG, "panel needs an incoming inter-GPU ring"); J.in = multi ? x_boundary(xin, false) : self_boundary((q - 1) & 1); }
        if (J.has_out) { if (multi && !xout) return psa_fail(ctx, PSA_ERR_ARG, "panel needs an outgoing inter-GPU ring"); J.out = multi ? x_boundary(xout, true) : self_boundary(q & 1); }
        if (q == npanels - 1) has_corner = 1;
        const int grid = (J.nstrips + SWPB - 1) / SWPB;
        auto go_k = [&](auto kern) { kern<<<grid, SWPB * 32, 0, st>>>(J); };
        const bool loc = (mode == PSA_LOCAL);
        switch (KC * 10 + RB) {
            case 41: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 4, 1>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 4, 1>); break;
            case 42: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 4, 2>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 4, 2>); break;
            case 81: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 8, 1>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 8, 1>); break;
            case 82: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 8, 2>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 8, 2>); break;
            case 84: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 8, 4>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 8, 4>); break;
            default: if (loc) go_k(psa_systolic_kernel<PSA_LOCAL, 4, 4>); else go_k(psa_systolic_kernel<PSA_GLOBAL, 4, 4>); break;
        }
        PSA_CUDA_OK(ctx, cudaGetLastError());
        ctx->launches += 1;
    }
    psa_systolic_result_kernel<<<1, 1, 0, st>>>(J.best, J.corner, mode, m, n_total, has_corner, d_item);
    PSA_CUDA_OK(ctx, cudaGetLastError());
    ctx->launches += 1;
    return PSA_OK;
}
