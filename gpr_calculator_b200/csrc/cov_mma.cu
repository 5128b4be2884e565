// cov_mma.cu — covariance blocks K_ff, K_ef/K_fe on the FP64 tensor pipe (DMMA.8x8x4) of sm_100a.
//
// Replaces rbf_kff_many / rbf_kff_many_with_grad / dot_kff_many and rbf_kef_many(_with_grad) /
// dot_kef_many of the reference (rbf_kernel.cpp:101-253, 341-640; dot_kernel.cpp:58-130, 217-336).
//
// Algebra (SURVEY.md §7.1).  With x^ = x/|x|, A~ = (I - x^x^T) dx/dr / |x| precomputed per row
// (pack.cu), every quantity the reference derives per pair from a d x d matrix is one entry of
//        [x^_a ; A~_a^T] (4 x d)  .  [x^_b ; B~_b^T]^T (d x 4)
//   s = x^_a.x^_b     p_c = A~_a[:,c].x^_b     q_e = x^_a.B~_b[:,e]     G_ce = A~_a[:,c].B~_b[:,e]
//   K_ff[3I+c,3J+e] = sum_{a in I, b in J}  g (beta G_ce + gamma p_c q_e)
// so a block of 8 x 8 atom pairs is 16 m8n8k4 accumulator tiles.  Rows are laid out
// component-major (tile = 8 rows of one component), which puts the complete 4x4 result of the
// pairs (a = lane/4, b = 2*(lane%4)+{0,1}) into the registers of ONE thread: the scalar epilogue
// (exp, powers, rank-1 correction) needs no shuffles.
//
// Generation 2 execution model (DESIGN.md §7):
//  * FLAT tiles: rows of neighbouring groups share 8-row tiles on both sides, so no DMMA work is
//    spent on per-group padding.  Column tiles carry a record of their group segments; a tile that
//    straddles a group boundary is multiplied once and accumulated once per segment with masked
//    weights.  Row tiles are handled by a segmented reduction (static per-thread predicates).
//  * one CTA = 12 warps = 96 consecutive rows; the row tiles live in shared memory (TMA bulk copy
//    at start) so that the kernel fits 168 registers and every scheduler has 3 warps to overlap
//    one warp's scalar epilogue with the other warps' DMMAs (DMMA and DFMA share the FP64 pipe).
//  * column tiles stream through a ring of TMA stages (cp.async.bulk + mbarrier); the warp that
//    releases a stage last refills it — no producer warp and no CTA-wide barrier in the main loop.
//  * flush at the end of a column group: transposing butterfly over the 4 lanes of a row, segmented
//    suffix sum over the 8 rows of the warp, head rows to one of four shared-memory buffers, one
//    mbarrier arrival per warp.  Two flushes later every warp adds the per-warp partials of its share
//    of the outputs in a fixed order and writes them (deterministic; no atomics on the critical path,
//    no designated finisher).
//    Row groups that continue in a neighbouring CTA are combined with fp64 atomics into the
//    pre-zeroed output (two addends: still order independent).
#include "cov_common.cuh"
#pragma nv_diag_suppress 128   // the 4x4-block path below the two-stage branch is unreachable in the two-stage instantiations
#include <cstdint>
#include <cmath>
#include <cstdlib>

namespace {

constexpr int WARPS = 12;
constexpr int THREADS = WARPS * 32;
constexpr int STAGES = 2;
constexpr int CH = GPRB_CHUNK_TILES;
constexpr int REC = GPRB_REC_INTS;
constexpr int MAXROWS = WARPS * 8;
constexpr int BIG_WARPS = 6, BIG_CH = 2;   // CTA shape of the 9..16 k-step kernels (d = 33..64)
constexpr int NFB = 4;                 // flush buffers: partials of flush k are summed two flushes later



__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded waits: a protocol error must surface as a launch failure (trap), never as a hung GPU.
constexpr long long SPIN_LIMIT_CYCLES = 8000000000LL;     // ~4 s at 1.9 GHz
__device__ __noinline__ void spin_timeout(int what) {
    printf("libgpr_b200: cov_mma_kernel wait %d timed out (block %d,%d thread %d)\n", what, blockIdx.x, blockIdx.y, threadIdx.x);
    __trap();
}
__device__ __forceinline__ bool mbar_try(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try(bar, parity))
        if (clock64() - t0 > SPIN_LIMIT_CYCLES) spin_timeout(1);
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Flush of the per-thread sums `out[NT]` when column group J is complete: transposing butterfly over the 4 lanes of a
// row, segmented suffix sum over the 8 rows of the warp, head rows to flush buffer flush_idx & 3, one mbarrier arrival per
// warp; the final sums of flush k are taken two flushes later (finish).  A macro so that the 4x4-block path and the
// two-stage path expand the very same statements.
#define COV_FLUSH_GROUP(J) \
    do { \
                if (flush_idx >= 2) finish(flush_idx - 2, J2); \
                const int fb = flush_idx & (NFB - 1); \
                const bool b0 = lane & 1, b1 = lane & 2; \
                double wv[N1], zv[N2]; \
_Pragma("unroll") \
                for (int i = 0; i < N1; i++) { \
                    const double lo = out[2 * i], hi = (2 * i + 1 < NT) ? out[(2 * i + 1 < NT) ? 2 * i + 1 : 0] : 0.0; \
                    const double keep = b0 ? hi : lo, send = b0 ? lo : hi; \
                    wv[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1); \
                } \
_Pragma("unroll") \
                for (int i = 0; i < N2; i++) { \
                    const double lo = wv[2 * i], hi = (2 * i + 1 < N1) ? wv[(2 * i + 1 < N1) ? 2 * i + 1 : 0] : 0.0; \
                    const double keep = b1 ? hi : lo, send = b1 ? lo : hi; \
                    zv[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2); \
                } \
_Pragma("unroll") \
                for (int i = 0; i < N2; i++) { \
                    double tv = __shfl_down_sync(0xffffffffu, zv[i], 4); \
                    zv[i] += p1 ? tv : 0.0; \
                    tv = __shfl_down_sync(0xffffffffu, zv[i], 8); \
                    zv[i] += p2 ? tv : 0.0; \
                    tv = __shfl_down_sync(0xffffffffu, zv[i], 16); \
                    zv[i] += p4 ? tv : 0.0; \
                } \
                if (is_head) { \
                    double *dst = sRow + (size_t)(fb * MAXROWS_K + arow_local) * NT + q4; \
_Pragma("unroll") \
                    for (int i = 0; i < N2; i++) \
                        if (4 * i + q4 < NT) dst[4 * i] = zv[i]; \
                } \
_Pragma("unroll") \
                for (int i = 0; i < NT; i++) out[i] = 0.0; \
                __syncwarp(); \
                if (lane == 0) mbar_arrive(&barFlush[fb]); \
                J2 = J1; J1 = J; \
                flush_idx++; \
    } while (0)

// NB = component tiles per column tile: 4 = force columns against force rows (K_ff), 1 = energy columns against force
// rows (K_fe / K_ef), 0 = energy columns against ENERGY rows (K_ee: one component on both sides, two CTAs per SM)
template <int NB, int KS_T, int KERNEL, bool GRAD, int ZI, bool MULTI, bool TWO, bool BIG>
__global__ void __launch_bounds__(BIG ? BIG_WARPS * 32 : THREADS, NB == 0 ? 2 : 1) cov_mma_kernel(const CovParams P) {
    // BIG: descriptors of 33..64 entries (9..16 k-steps): the row tiles of 12 warps no longer fit the shared memory, so 6 warps per CTA and
    // 2-tile column chunks (functional path for e.g. SO3(nmax=4, lmax=4), d = 50; the benchmarked descriptor has d = 30)
    constexpr int WARPS_K = BIG ? BIG_WARPS : WARPS, CH_K = BIG ? BIG_CH : CH, MAXROWS_K = WARPS_K * 8;
    constexpr bool FF = (NB == 4), EE = (NB == 0);
    constexpr int NA = EE ? 1 : 4, NBC = EE ? 1 : NB;        // component tiles of a row tile / of a column tile
    constexpr int NOUT = FF ? 9 : (EE ? 1 : 3);
    constexpr int NT = GRAD ? 2 * NOUT : NOUT;
    constexpr int N1 = (NT + 1) / 2, N2 = (N1 + 1) / 2;      // values left after each transposing butterfly step
    const int KS = KS_T ? KS_T : P.ks;
    const int a_tile_d = NA * KS * 32, b_tile_d = NBC * KS * 32;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *sA = reinterpret_cast<double *>(smem_raw);                  // [WARPS_K][a_tile_d]
    double *sB = sA + WARPS_K * a_tile_d;                                  // [STAGES][CH_K][b_tile_d]
    double *sRow = sB + STAGES * CH_K * b_tile_d;                          // [NFB][MAXROWS_K][NT] flush partials
    double *sTab = sRow + NFB * MAXROWS_K * NT;                            // [EXP_TAB]
    int4 *sEnt = reinterpret_cast<int4 *>(sTab + EXP_TAB);               // [MAXROWS_K]
    int *sRec = reinterpret_cast<int *>(sEnt + MAXROWS_K);                 // [STAGES][CH_K][REC]
    uint64_t *sBar = reinterpret_cast<uint64_t *>(sRec + STAGES * CH_K * REC);   // full[STAGES], A, flush[NFB]
    uint64_t *barFlush = sBar + STAGES + 1;
    int *sCnt = reinterpret_cast<int *>(barFlush + NFB);                 // consumed[STAGES]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int4 blk = P.sched[blockIdx.x];
    const int tile0 = blk.x, ntiles = blk.y, ent0 = blk.z, nent = blk.w;

    // column group range of this CTA -> column tiles / chunks
    int ga, gb;
    {
        const int G = P.n_groupsB;
        const int first_group = P.sched_ent[ent0].x, last_group = P.sched_ent[ent0 + nent - 1].x;
        // the column groups this row block sweeps, cut evenly over the n_splits CTAs of the block
        int lo = 0, hi = G;
        if (P.mode == GPRB_FF_SYMMETRIC || P.mode == GPRB_FF_UPPER) lo = first_group;
        if (P.mode == GPRB_FF_DIAG) { lo = first_group; hi = last_group + 1; }
        ga = lo + (int)((long long)(hi - lo) * blockIdx.y / P.n_splits);
        gb = lo + (int)((long long)(hi - lo) * (blockIdx.y + 1) / P.n_splits);
    }
    if (gb <= ga) return;
    const int cr0 = P.row_ptrB[ga], cr1 = P.row_ptrB[gb];
    if (cr1 <= cr0) return;
    const int tb0 = cr0 >> 3, tb1 = (cr1 + 7) >> 3;
    const int c_begin = tb0 / CH_K, c_end = (tb1 + CH_K - 1) / CH_K;

    if (tid < nent) sEnt[tid] = P.sched_ent[ent0 + tid];
    for (int i = tid; i < EXP_TAB; i += blockDim.x) sTab[i] = d_exp2_tab[i];
    if (tid == 0) {
        for (int s = 0; s <= STAGES; s++) mbar_init(&sBar[s], 1);
        for (int s = 0; s < NFB; s++) mbar_init(&barFlush[s], ntiles);     // one arrival per active warp and flush
        for (int s = 0; s < STAGES; s++) sCnt[s] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const uint32_t b_chunk_bytes = (uint32_t)(CH_K * b_tile_d * 8), rec_chunk_bytes = (uint32_t)(CH_K * REC * 4);
    auto issue = [&](int ci, int buf) {
        mbar_expect_tx(&sBar[buf], b_chunk_bytes + rec_chunk_bytes);
        bulk_g2s(sB + (size_t)buf * CH_K * b_tile_d, P.PB + (size_t)ci * CH_K * b_tile_d, b_chunk_bytes, &sBar[buf]);
        bulk_g2s(sRec + buf * CH_K * REC, P.recB + (size_t)ci * CH_K * REC, rec_chunk_bytes, &sBar[buf]);
    };
    if (tid == 0) {
        const uint32_t a_bytes = (uint32_t)(ntiles * a_tile_d * 8);
        mbar_expect_tx(&sBar[STAGES], a_bytes);
        bulk_g2s(sA, P.PA + (size_t)tile0 * a_tile_d, a_bytes, &sBar[STAGES]);
        for (int s = 0; s < STAGES; s++)
            if (c_begin + s < c_end) issue(c_begin + s, s);
    }
    if (warp >= ntiles) return;          // no CTA-wide barrier below this line
    const int n_active = ntiles;

    // static per-thread row data: species, window, segment structure of the warp's 8 rows
    const int ra = lane >> 2, q4 = lane & 3;
    const int arow_local = warp * 8 + ra;
    const int arow = (tile0 + warp) * 8 + ra;
    int ele_a = P.eleA[arow];
    if (arow < P.win_r0 || arow >= P.win_r1) ele_a = -1;
    const int g_a = P.row_groupA[arow];
    // (shuffles first, unconditionally: every lane must take part in a full-mask shuffle)
    const int g_d1 = __shfl_down_sync(0xffffffffu, g_a, 4), g_d2 = __shfl_down_sync(0xffffffffu, g_a, 8);
    const int g_d4 = __shfl_down_sync(0xffffffffu, g_a, 16), g_u1 = __shfl_up_sync(0xffffffffu, g_a, 4);
    const bool p1 = (ra + 1 < 8) && (g_d1 == g_a);
    const bool p2 = (ra + 2 < 8) && (g_d2 == g_a);
    const bool p4 = (ra + 4 < 8) && (g_d4 == g_a);
    const bool is_head = (ra == 0) || (g_u1 != g_a);

    double out[NT];
#pragma unroll
    for (int i = 0; i < NT; i++) out[i] = 0.0;
    double Z[TWO ? 3 : 1][TWO ? 4 : 1][2];      // two-stage path: Z_e[ra][8 t + 2 q4 + {0, 1}] of the current column group
#pragma unroll
    for (int e = 0; e < (TWO ? 3 : 1); e++)
#pragma unroll
        for (int t = 0; t < (TWO ? 4 : 1); t++) { Z[e][t][0] = 0.0; Z[e][t][1] = 0.0; }
    int flush_idx = 0, J1 = 0, J2 = 0;      // J1 / J2: column groups of the previous two flushes

    // Final sums of flush kk (column group J): every warp adds the per-warp partials of ITS share of the
    // (row group, component) outputs in a fixed order and writes them.  Called two flushes later, when the
    // partials of all warps have long been delivered (mbarrier per flush buffer; no atomics, no designated
    // finisher warp, deterministic).  Buffer reuse is safe with NFB = 4: a warp overwrites buffer k & 3 at
    // flush k only after it has seen flush k-2 complete, i.e. after every warp has summed its share of k-4.
    auto finish = [&](int kk, int J) {
        const int fb = kk & (NFB - 1);
        mbar_wait(&barFlush[fb], (kk / NFB) & 1);
        const int total = nent * NT;
        for (int idx = lane * n_active + warp; idx < total; idx += 32 * n_active) {
            const int en = idx / NT, o = idx - en * NT;
            const int4 E4 = sEnt[en];
            const int I = E4.x;
            const double *src = sRow + (size_t)fb * MAXROWS_K * NT + o;
            double v = src[E4.y * NT];
            for (int r = (E4.y & ~7) + 8; r < E4.z; r += 8) v += src[r * NT];
            const bool shared = E4.w != 0;
            const bool isgrad = GRAD && o >= NOUT;
            const int oo = isgrad ? o - NOUT : o;
            if (FF) {
                const int c = oo / 3, e = oo - 3 * c;
                double *dst = isgrad ? P.dK : P.K;
                const long long ld = isgrad ? P.lddk : P.ldk;
                if (P.mode == GPRB_FF_DIAG) {
                    if (I == J && c == e) {
                        double *qd = dst + 3 * (I - P.grp_begin) + c;
                        if (shared) atomicAdd(qd, v); else *qd = v;
                    }
                } else if (!((P.mode == GPRB_FF_SYMMETRIC || P.mode == GPRB_FF_UPPER) && J < I)) {
                    const long long off = (long long)(3 * (I - P.grp_begin) + c) * ld + 3 * J + e;
                    double *qd = dst + off;
                    if (shared) atomicAdd(qd, v); else *qd = v;
                    if (MULTI && !isgrad) {
#pragma unroll
                        for (int p = 0; p < GPRB_MAX_DST - 1; p++)
                            if (p < P.n_extra) { double *qp = P.Kx[p] + off; if (shared) atomicAdd(qp, v); else *qp = v; }
                    }
                    if (P.mode == GPRB_FF_SYMMETRIC && J > I) {
                        double *qt = dst + (long long)(3 * J + e) * ld + 3 * I + c;
                        if (shared) atomicAdd(qt, v); else *qt = v;
                    }
                }
            } else if (EE) {
                // K_ee[I, J] = 1 / (n_I n_J) sum k   (rbf_kernel.py:56-70, dot_kernel.py:46).  Symmetric mode writes
                // J >= I only and gprb_kee mirrors afterwards: a group split over three or more CTAs is summed by
                // atomics in arrival order, which can differ between K[I, J] and K[J, I] in the last bits.
                const double nn = (double)P.group_rowsA[I] * (double)P.group_rowsB[J];
                const double val = nn > 0 ? v / nn : 0.0;
                double *dst = isgrad ? P.dK : P.K;
                const long long ld = isgrad ? P.lddk : P.ldk;
                if (!(P.mode == GPRB_FF_SYMMETRIC && J < I)) {
                    double *qd = dst + (long long)(I - P.grp_begin) * ld + J;
                    if (shared) atomicAdd(qd, val); else *qd = val;
                }
            } else {
                // a side = force group I (window), b side = energy group J; K_ef = -(1/n_J) sum
                const int nJ = P.group_rowsB[J];
                const double val = nJ > 0 ? -v / (double)nJ : 0.0;
                const long long row = 3 * (I - P.grp_begin) + oo;
                double *fe = isgrad ? P.dK : P.K;
                const long long ldfe = isgrad ? P.lddk : P.ldk;
                double *ef = isgrad ? P.dK2 : P.K2;
                const long long ldef = isgrad ? P.lddk2 : P.ldk2;
                if (fe) {
                    const long long off = row * ldfe + J;
                    double *qd = fe + off;
                    if (shared) atomicAdd(qd, val); else *qd = val;
                    if (MULTI && !isgrad) {
#pragma unroll
                        for (int p = 0; p < GPRB_MAX_DST - 1; p++)
                            if (p < P.n_extra) { double *qp = P.Kx[p] + off; if (shared) atomicAdd(qp, val); else *qp = val; }
                    }
                }
                if (ef) { double *qd = ef + (long long)J * ldef + row; if (shared) atomicAdd(qd, val); else *qd = val; }
            }
        }
    };

    mbar_wait(&sBar[STAGES], 0);         // row tiles have landed
    const double *pa = sA + (size_t)warp * a_tile_d + lane;

    for (int ci = c_begin; ci < c_end; ci++) {
        const int it = ci - c_begin, buf = it % STAGES;
        mbar_wait(&sBar[buf], (it / STAGES) & 1);
        for (int tt = 0; tt < CH_K; tt++) {
            const int t = ci * CH_K + tt;
            if (t < tb0 || t >= tb1) continue;
            const int *rec = sRec + (buf * CH_K + tt) * REC;
            const double *pb = sB + (size_t)(buf * CH_K + tt) * b_tile_d + lane;

            if constexpr (TWO) {
                // Two-stage contraction (no gradient, d in 29..32; design: profiles/experiments/README.md and
                // two_stage_emulation.py; parity: test_two_stage_path_matches_block_path).  Stage 1: x^(a) . [x^; B~_e](b) -> s, q_e
                // (32 DMMAs).  Stage 2, per column segment: Z_e[a, :] += W1 B~_e + (W2 q_e) x^ with the stage-1 accumulator
                // registers as A fragments (k order b = 2 q4 + j) and the B fragments read from the same slabs (48 DMMAs).
                // Per column group: out_ce = A~_c(a) . Z_e(a), then the common flush.
                static_assert(!TWO || (NB == 4 && KS_T == 8 && !GRAD), "two-stage path: K_ff without gradient, 8 k-steps");
                double a1[4][2];
#pragma unroll
                for (int e = 0; e < 4; e++) { a1[e][0] = 0.0; a1[e][1] = 0.0; }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const double af = pa[k * 32];
#pragma unroll
                    for (int e = 0; e < 4; e++) dmma(a1[e][0], a1[e][1], af, pb[(e * 8 + k) * 32]);
                }
                const int2 eb2 = *reinterpret_cast<const int2 *>(rec + 2 * q4);
                double tw1[2], tw2[2];
                bool tvalid[2];
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const int ele_b = j ? eb2.y : eb2.x;
                    tvalid[j] = (ele_a == ele_b) && (ele_a >= 0);
                    double du1 = 0.0, du2 = 0.0;
                    tw2[j] = 0.0;
                    pair_weights<KERNEL, false, true, ZI>(P, sTab, a1[0][j], tvalid[j], tw1[j], tw2[j], du1, du2);
                }
                const double *pbt = pb - lane;                      // tile base: stage 2 addresses the slabs by (row b, column)
                const int nseg2 = rec[8];
                for (int sg = 0; sg < nseg2; sg++) {
                    const int J = rec[10 + 2 * sg], mf = rec[11 + 2 * sg];
                    if (J < ga || J >= gb) continue;
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        const bool on = tvalid[j] && ((mf >> (2 * q4 + j)) & 1);
                        const double W1 = on ? tw1[j] : 0.0;
                        double V[3];
#pragma unroll
                        for (int e = 0; e < 3; e++) V[e] = on ? tw2[j] * a1[1 + e][j] : 0.0;
#pragma unroll
                        for (int t = 0; t < 4; t++) {
                            // B fragment of n-tile t: element (k = q4 -> row b = 2 q4 + j, n = ra -> column 8 t + ra)
                            const int off = (2 * t + (ra >> 2)) * 32 + (2 * q4 + j) * 4 + (ra & 3);
                            const double bx = pbt[off];
#pragma unroll
                            for (int e = 0; e < 3; e++) {
                                dmma(Z[e][t][0], Z[e][t][1], W1, pbt[(1 + e) * 8 * 32 + off]);
                                dmma(Z[e][t][0], Z[e][t][1], V[e], bx);
                            }
                        }
                    }
                    if (!(mf & 0x100)) continue;
                    // column group J is complete: out_ce = sum over this thread's 8 columns of A~_c[ra, col] Z_e[ra, col]
                    const double *par = pa - lane;                  // row tile base (component c + 1 holds A~_c)
#pragma unroll
                    for (int c = 0; c < 3; c++) {
#pragma unroll
                        for (int t = 0; t < 4; t++) {
                            // columns 8 t + 2 q4 + {0, 1}: k-step 2 t + (q4 >> 1), kk = 2 (q4 & 1) + {0, 1} (adjacent: one 16-byte read)
                            const double2 av = *reinterpret_cast<const double2 *>(
                                par + ((c + 1) * 8 + 2 * t + (q4 >> 1)) * 32 + ra * 4 + 2 * (q4 & 1));
#pragma unroll
                            for (int e = 0; e < 3; e++) out[c * 3 + e] = fma(av.x, Z[e][t][0], fma(av.y, Z[e][t][1], out[c * 3 + e]));
                        }
                    }
#pragma unroll
                    for (int e = 0; e < 3; e++)
#pragma unroll
                        for (int t = 0; t < 4; t++) { Z[e][t][0] = 0.0; Z[e][t][1] = 0.0; }
                    COV_FLUSH_GROUP(J);
                }
                continue;
            }

            // species of this thread's two pairs (a = ra, b = 2*q4 + j): read after the DMMAs, except for K_ee
            bool valid[2];
            if (EE) {
                const int2 eb = *reinterpret_cast<const int2 *>(rec + 2 * q4);
                valid[0] = (ele_a == eb.x) && (ele_a >= 0);
                valid[1] = (ele_a == eb.y) && (ele_a >= 0);
                // energy rows of one structure are usually ordered by species (all Mg, all O, ...): a pair of tiles without any
                // same-species pair contributes nothing (rbf_kernel.cpp:26-37) -- skip its DMMAs and exp; a group that ends in
                // the tile still has to be flushed
                if (!__any_sync(0xffffffffu, valid[0] || valid[1])) {
                    const int nseg0 = rec[8];
                    for (int sg = 0; sg < nseg0; sg++) {
                        const int J = rec[10 + 2 * sg], mf = rec[11 + 2 * sg];
                        if (J < ga || J >= gb || !(mf & 0x100)) continue;
                        COV_FLUSH_GROUP(J);
                    }
                    continue;
                }
            }
            double acc[NA][NBC][2];
#pragma unroll
            for (int c = 0; c < NA; c++)
#pragma unroll
                for (int e = 0; e < NBC; e++) { acc[c][e][0] = 0.0; acc[c][e][1] = 0.0; }
            if (KS_T) {
#pragma unroll
                for (int k = 0; k < (KS_T ? KS_T : 1); k++) {
                    double af[NA], bf[NBC];
#pragma unroll
                    for (int c = 0; c < NA; c++) af[c] = pa[(c * KS_T + k) * 32];
#pragma unroll
                    for (int e = 0; e < NBC; e++) bf[e] = pb[(e * KS_T + k) * 32];
#pragma unroll
                    for (int c = 0; c < NA; c++)
#pragma unroll
                        for (int e = 0; e < NBC; e++) dmma(acc[c][e][0], acc[c][e][1], af[c], bf[e]);
                }
            } else {
                for (int k = 0; k < KS; k++) {
                    double af[NA], bf[NBC];
#pragma unroll
                    for (int c = 0; c < NA; c++) af[c] = pa[(c * KS + k) * 32];
#pragma unroll
                    for (int e = 0; e < NBC; e++) bf[e] = pb[(e * KS + k) * 32];
#pragma unroll
                    for (int c = 0; c < NA; c++)
#pragma unroll
                        for (int e = 0; e < NBC; e++) dmma(acc[c][e][0], acc[c][e][1], af[c], bf[e]);
                }
            }

            // weights of this thread's two pairs, once per tile
            if (!EE) {
                const int2 eb = *reinterpret_cast<const int2 *>(rec + 2 * q4);
                valid[0] = (ele_a == eb.x) && (ele_a >= 0);
                valid[1] = (ele_a == eb.y) && (ele_a >= 0);
            }
            double w1[2], w2[2], u1[2], u2[2];
#pragma unroll
            for (int j = 0; j < 2; j++) {
                w2[j] = 0.0; u1[j] = 0.0; u2[j] = 0.0;
                pair_weights<KERNEL, GRAD, FF, ZI, EE>(P, sTab, acc[0][0][j], valid[j], w1[j], w2[j], u1[j], u2[j]);
            }

            const int nseg = rec[8];
            for (int sg = 0; sg < nseg; sg++) {
                const int J = rec[10 + 2 * sg], mf = rec[11 + 2 * sg];
                if (J < ga || J >= gb) continue;
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const bool on = valid[j] && ((mf >> (2 * q4 + j)) & 1);
                    const double W1 = on ? w1[j] : 0.0;
                    if (EE) {
                        out[0] += W1;
                        if (GRAD) out[NOUT] += on ? u1[j] : 0.0;
                    } else if (FF) {
                        const double W2 = on ? w2[j] : 0.0, U1 = on ? u1[j] : 0.0, U2 = on ? u2[j] : 0.0;
#pragma unroll
                        for (int c = 0; c < 3; c++) {
                            const double pc = acc[(NA == 4) ? c + 1 : 0][0][j];
                            const double t2 = W2 * pc;
                            const double t3 = GRAD ? U2 * pc : 0.0;
#pragma unroll
                            for (int e = 0; e < 3; e++) {
                                const double G = acc[(NA == 4) ? c + 1 : 0][(NB == 4) ? e + 1 : 0][j];
                                const double qe = acc[0][(NB == 4) ? e + 1 : 0][j];
                                out[c * 3 + e] = fma(W1, G, fma(t2, qe, out[c * 3 + e]));
                                if (GRAD) out[NOUT + c * 3 + e] = fma(U1, G, fma(t3, qe, out[NOUT + c * 3 + e]));
                            }
                        }
                    } else {
                        const double U1 = on ? u1[j] : 0.0;
#pragma unroll
                        for (int c = 0; c < 3; c++) {
                            const double pc = acc[(NA == 4) ? c + 1 : 0][0][j];
                            out[c] = fma(W1, pc, out[c]);
                            if (GRAD) out[NOUT + c] = fma(U1, pc, out[NOUT + c]);
                        }
                    }
                }
                if (!(mf & 0x100)) continue;

                COV_FLUSH_GROUP(J);      // column group J is complete
            }
        }
        // release the stage; the warp that arrives last refills it
        __syncwarp();
        if (lane == 0) {
            const int old = atomicAdd(&sCnt[buf], 1);
            if ((old + 1) % n_active == 0 && ci + STAGES < c_end) issue(ci + STAGES, buf);
        }
    }
    // the sums of the last two flushes
    if (flush_idx >= 2) finish(flush_idx - 2, J2);
    if (flush_idx >= 1) finish(flush_idx - 1, J1);
}

size_t cov_smem_bytes(int nb, int ks, bool grad, bool big) {
    const int nt = (nb == 4 ? 9 : (nb == 0 ? 1 : 3)) * (grad ? 2 : 1);
    const int na = nb == 0 ? 1 : 4, nbc = nb == 0 ? 1 : nb;
    const int warps = big ? BIG_WARPS : WARPS, ch = big ? BIG_CH : CH, maxrows = warps * 8;
    return (size_t)(warps * na * ks * 32 + STAGES * ch * nbc * ks * 32 + NFB * maxrows * nt + EXP_TAB) * 8 +
           (size_t)maxrows * 16 + (size_t)STAGES * ch * REC * 4 + (STAGES + 1 + NFB) * 8 + STAGES * 4 + 128;
}

// Row-side schedule for the window [g0, g1): blocks of <= WARPS consecutive flat tiles and, per block, the
// groups it holds {group, first row, one past last row (block-local), continues in a neighbouring block}.
int build_sched(gprb_pack *a, int g0, int g1, cudaStream_t st) {
    const int wpc = a->ks > GPRB_MAX_KS ? BIG_WARPS : WARPS;       // row tiles per CTA of the kernels this pack runs (fixed by its ks)
    if (a->sched_g0 == g0 && a->sched_g1 == g1 && a->sched) return GPRB_OK;
    std::vector<int4> blocks, ents;
    const int r0 = a->row_ptr[g0], r1 = a->row_ptr[g1];
    if (r1 > r0) {
        const int t0 = r0 / 8, t1 = (r1 + 7) / 8;
        int g = g0;
        for (int tb = t0; tb < t1; tb += wpc) {
            const int nt = t1 - tb < wpc ? t1 - tb : wpc;
            const int lo = tb * 8 > r0 ? tb * 8 : r0, hi = (tb + nt) * 8 < r1 ? (tb + nt) * 8 : r1;
            const int e0 = (int)ents.size();
            while (g < g1 && a->row_ptr[g + 1] <= lo) g++;      // groups that ended before this block (or empty)
            int gg = g;
            while (gg < g1 && a->row_ptr[gg] < hi) {
                const int s = a->row_ptr[gg] > lo ? a->row_ptr[gg] : lo;
                const int e = a->row_ptr[gg + 1] < hi ? a->row_ptr[gg + 1] : hi;
                if (e > s) {
                    const int shared = (a->row_ptr[gg] < lo || a->row_ptr[gg + 1] > hi) ? 1 : 0;
                    ents.push_back(make_int4(gg, s - tb * 8, e - tb * 8, shared));
                }
                gg++;
            }
            if ((int)ents.size() > e0) blocks.push_back(make_int4(tb, nt, e0, (int)ents.size() - e0));
        }
    }
    if (a->sched) { GPRB_CUDA(cudaFreeAsync(a->sched, st)); a->sched = nullptr; }
    if (a->sched_ent) { GPRB_CUDA(cudaFreeAsync(a->sched_ent, st)); a->sched_ent = nullptr; }
    a->sched_host = blocks; a->sched_ent_host = ents;
    a->sched_n = (int)blocks.size();
    a->sched_g0 = g0; a->sched_g1 = g1;
    if (!blocks.empty()) {
        GPRB_CUDA(cudaMallocAsync((void **)&a->sched, blocks.size() * sizeof(int4), st));
        GPRB_CUDA(cudaMallocAsync((void **)&a->sched_ent, ents.size() * sizeof(int4), st));
        GPRB_CUDA(cudaMemcpyAsync(a->sched, a->sched_host.data(), blocks.size() * sizeof(int4), cudaMemcpyHostToDevice, st));
        GPRB_CUDA(cudaMemcpyAsync(a->sched_ent, a->sched_ent_host.data(), ents.size() * sizeof(int4), cudaMemcpyHostToDevice, st));
    }
    return GPRB_OK;
}

template <int NB, int KS_T, int KERNEL, bool GRAD, int ZI, bool MULTI, bool TWO = false, bool BIG = false>
int launch_cov_m(const CovParams &P, int n_blocks, cudaStream_t st) {
    auto kern = cov_mma_kernel<NB, KS_T, KERNEL, GRAD, ZI, MULTI, TWO, BIG>;
    static bool configured[MAX_DEV] = {};
    int dev = 0;
    { int rc = current_device(&dev); if (rc) return rc; }
    if (!configured[dev]) {
        GPRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)cov_smem_bytes(NB, BIG ? 2 * GPRB_MAX_KS : GPRB_MAX_KS, GRAD, BIG)));
        configured[dev] = true;
    }
    dim3 grid(n_blocks, P.n_splits);
    kern<<<grid, BIG ? BIG_WARPS * 32 : THREADS, cov_smem_bytes(NB, P.ks, GRAD, BIG), st>>>(P);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

// the single-destination kernels carry no peer-store code at all (MULTI = false)
template <int NB, int KS_T, int KERNEL, bool GRAD, int ZI, bool BIG = false>
int launch_cov(const CovParams &P, int n_blocks, cudaStream_t st) {
    if constexpr (BIG)
        return P.n_extra > 0 ? launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, true, false, true>(P, n_blocks, st)
                             : launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, false, false, true>(P, n_blocks, st);
    if constexpr (NB == 4 && KS_T == 8 && !GRAD) {
        if (P.two_stage)
            return P.n_extra > 0 ? launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, true, true>(P, n_blocks, st)
                                 : launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, false, true>(P, n_blocks, st);
    }
    return P.n_extra > 0 ? launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, true>(P, n_blocks, st)
                         : launch_cov_m<NB, KS_T, KERNEL, GRAD, ZI, false>(P, n_blocks, st);
}

template <int NB, int KS_T, int ZI, bool BIG = false>
int dispatch_kernel(int kernel, bool grad, const CovParams &P, int n_blocks, cudaStream_t st) {
    if (kernel == GPRB_KERNEL_RBF) return grad ? launch_cov<NB, KS_T, GPRB_KERNEL_RBF, true, ZI, BIG>(P, n_blocks, st)
                                               : launch_cov<NB, KS_T, GPRB_KERNEL_RBF, false, ZI, BIG>(P, n_blocks, st);
    return launch_cov<NB, KS_T, GPRB_KERNEL_DOT, false, ZI, BIG>(P, n_blocks, st);
}

template <int NB>
int dispatch_cov(int kernel, bool grad, const CovParams &P, int n_blocks, cudaStream_t st) {
    const bool z2 = P.zi == 2;
    if (P.ks > GPRB_MAX_KS) return dispatch_kernel<NB, 0, 0, true>(kernel, grad, P, n_blocks, st);     // d = 33..64
    if (P.ks == 8) return z2 ? dispatch_kernel<NB, 8, 2>(kernel, grad, P, n_blocks, st) : dispatch_kernel<NB, 8, 0>(kernel, grad, P, n_blocks, st);
    return z2 ? dispatch_kernel<NB, 0, 2>(kernel, grad, P, n_blocks, st) : dispatch_kernel<NB, 0, 0>(kernel, grad, P, n_blocks, st);
}

int choose_splits(int n_blocks, int n_groupsB) {
    int sms = 148;
    int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // enough CTAs (24 per SM) that the longest one is a small fraction of the launch: a row block's sweep
    // can take tens of milliseconds, and whole-sweep CTAs would leave a long partially filled last wave
    int want = (24 * sms + n_blocks - 1) / (n_blocks > 0 ? n_blocks : 1);
    if (want < 1) want = 1;
    if (want > n_groupsB) want = n_groupsB;
    if (want < 1) want = 1;
    if (want > 65535) want = 65535;
    return want;
}

// Checks every covariance builder makes.  Side A is the pack whose group window [grp_begin, grp_end) gives the rows
// the kernel runs over, with ncols_a columns (0 energy, 3 force); side B has ncols_b.  The descriptor limit is not
// checked here: gprb_pack_create refuses descriptors the kernels cannot run.
int check_cov_args(const char *who, int kernel, const gprb_pack *a, int ncols_a, const gprb_pack *b, int ncols_b,
                   int grp_begin, int grp_end, bool has_out, bool has_dk) {
    GPRB_REQUIRE(a && b && has_out, "%s: NULL argument", who);
    { int rcd = gprb_check_device(a, who); if (rcd || (rcd = gprb_check_device(b, who))) return rcd; }
    auto kind = [](int ncols) { return ncols ? "force" : "energy"; };
    GPRB_REQUIRE(a->ncols == ncols_a, "%s: need %s rows, got %s rows", who, kind(ncols_a), kind(a->ncols));
    GPRB_REQUIRE(b->ncols == ncols_b, "%s: need %s columns, got %s columns", who, kind(ncols_b), kind(b->ncols));
    GPRB_REQUIRE(a->d == b->d, "%s: descriptor length mismatch %d vs %d", who, a->d, b->d);
    GPRB_REQUIRE(kernel == GPRB_KERNEL_RBF || kernel == GPRB_KERNEL_DOT, "%s: unknown kernel %d", who, kernel);
    GPRB_REQUIRE(0 <= grp_begin && grp_begin <= grp_end && grp_end <= a->n_groups, "%s: bad window [%d,%d)", who, grp_begin, grp_end);
    GPRB_REQUIRE(!(has_dk && kernel == GPRB_KERNEL_DOT), "%s: Dot has no dK output (closed form, see header)", who);
    return GPRB_OK;
}

// dst[0] is this GPU's output (the caller decides whether it may be NULL), dst[1..n_dst) the same row slab in peer matrices
int check_dst(const char *who, int n_dst, double *const *dst) {
    GPRB_REQUIRE(n_dst >= 1 && n_dst <= GPRB_MAX_DST && dst, "%s: need 1..%d destination matrices", who, GPRB_MAX_DST);
    for (int p = 1; p < n_dst; p++) GPRB_REQUIRE(dst[p], "%s: NULL destination %d", who, p);
    return GPRB_OK;
}

// kernel constants, side A (rows, schedule of build_sched), side B (columns) and the row window
int init_cov_params(CovParams &P, int kernel, double p0, double p1, double zeta, const gprb_pack *a, const gprb_pack *b,
                    int grp_begin, int grp_end) {
    int rc = fill_kernel_params(P, kernel, p0, p1, zeta);
    if (rc) return rc;
    P.PA = a->P; P.eleA = a->elep; P.row_groupA = a->row_group; P.sched = a->sched; P.sched_ent = a->sched_ent;
    P.PB = b->P; P.recB = b->tile_rec; P.row_ptrB = b->d_row_ptr; P.group_rowsB = b->d_group_rows;
    P.n_groupsB = b->n_groups; P.ks = a->ks;
    P.win_r0 = a->row_ptr[grp_begin]; P.win_r1 = a->row_ptr[grp_end];
    P.grp_begin = grp_begin;
    P.n_splits = choose_splits(a->sched_n, b->n_groups);
    return GPRB_OK;
}

// zeroes rows x cols doubles of a matrix with leading dimension ld; a NULL output is skipped
cudaError_t zero2d(double *M, long long ld, size_t cols, int rows, cudaStream_t st) {
    return M ? cudaMemset2DAsync(M, ld * sizeof(double), 0, cols * sizeof(double), rows, st) : cudaSuccess;
}

}  // namespace

// n_dst > 1: K_dst[1..] are the same row slab in peer matrices (fused all-gather); the outputs are then NOT
// zeroed here (every GPU zeroes its own matrix before the ranks synchronise, see dist.PeerMatrix)
static int kff_impl(int kernel, const gprb_pack *f1_, const gprb_pack *f2, double p0, double p1, double zeta,
                    int use_tol, double tol, int mode, int grp_begin, int grp_end,
                    int n_dst, double *const *K_dst, long long ldk, double *dK, long long lddk, cudaStream_t st) {
    gprb_pack *f1 = const_cast<gprb_pack *>(f1_);
    int rc = check_dst("gprb_kff", n_dst, K_dst);
    if (rc) return rc;
    double *K = K_dst[0];
    if ((rc = check_cov_args("gprb_kff", kernel, f1, 3, f2, 3, grp_begin, grp_end, K != nullptr, dK != nullptr))) return rc;
    GPRB_REQUIRE(mode >= 0 && mode <= 3, "gprb_kff: unknown mode %d", mode);
    if (mode == GPRB_FF_SYMMETRIC)
        GPRB_REQUIRE(f1 == f2 && grp_begin == 0 && grp_end == f1->n_groups, "gprb_kff: symmetric mode needs f1 == f2 and the full window");
    if (mode == GPRB_FF_DIAG || mode == GPRB_FF_UPPER) GPRB_REQUIRE(f1 == f2, "gprb_kff: diag / upper mode needs f1 == f2");
    if (grp_begin == grp_end || f2->n_groups == 0) return GPRB_OK;
    if ((rc = build_sched(f1, grp_begin, grp_end, st))) return rc;
    // the output is pre-zeroed: groups without rows stay zero and row groups shared by two CTAs are
    // combined with atomics (UPPER leaves the blocks left of the diagonal zero)
    const int rows = 3 * (grp_end - grp_begin);
    if (mode == GPRB_FF_DIAG) {
        GPRB_REQUIRE(n_dst == 1, "gprb_kff_multi: diag mode has a single destination");
        GPRB_CUDA(cudaMemsetAsync(K, 0, (size_t)rows * sizeof(double), st));
    } else {
        GPRB_CUDA(zero2d(n_dst == 1 ? K : nullptr, ldk, (size_t)3 * f2->n_groups, rows, st));
        GPRB_CUDA(zero2d(dK, lddk, (size_t)3 * f2->n_groups, rows, st));
    }
    if (f1->sched_n == 0 || f2->n_rows == 0) return GPRB_OK;
    // RBF with gradient over a whole pack: the factored build when the pack's rows share atoms (cov_factored.cu)
    if (kernel == GPRB_KERNEL_RBF && dK && f1 == f2 && grp_begin == 0 && grp_end == f1->n_groups && n_dst == 1) {
        bool done = false;
        if ((rc = gprb_kff_factored(f1, p0, p1, zeta, mode, K, ldk, dK, lddk, st, &done))) return rc;
        if (done) return GPRB_OK;
    }
    CovParams P = {};
    if ((rc = init_cov_params(P, kernel, p0, p1, zeta, f1, f2, grp_begin, grp_end))) return rc;
    P.tol = tol; P.use_tol = use_tol; P.mode = mode;
    P.K = K; P.ldk = ldk; P.dK = dK; P.lddk = lddk;
    P.n_extra = n_dst - 1;
    for (int p = 1; p < n_dst; p++) P.Kx[p - 1] = K_dst[p];
    // no-gradient K_ff with 8 k-steps (d = 29..32, the default descriptor): two-stage contraction, 1.44x the 4x4-block path
    // (profiles/r02_two_stage.txt); GPRB_KFF_TWO_STAGE=0 selects the block path for the A/B parity test
    const char *two_env = getenv("GPRB_KFF_TWO_STAGE");
    P.two_stage = (!dK && mode != GPRB_FF_DIAG && f1->ks == GPRB_MAX_KS && !(two_env && two_env[0] == '0')) ? 1 : 0;
    if (mode == GPRB_FF_DIAG) P.n_splits = 1;
    return dispatch_cov<4>(kernel, dK != nullptr, P, f1->sched_n, st);
}

extern "C" int gprb_kff(int kernel, const gprb_pack *f1, const gprb_pack *f2, double p0, double p1, double zeta,
                        int use_tol, double tol, int mode, int grp_begin, int grp_end,
                        double *K, long long ldk, double *dK, long long lddk, void *stream) {
    double *dst[1] = {K};
    return kff_impl(kernel, f1, f2, p0, p1, zeta, use_tol, tol, mode, grp_begin, grp_end, 1, dst, ldk, dK, lddk, (cudaStream_t)stream);
}

extern "C" int gprb_kff_multi(int kernel, const gprb_pack *f1, const gprb_pack *f2, double p0, double p1, double zeta,
                              int use_tol, double tol, int mode, int grp_begin, int grp_end,
                              int n_dst, double *const *K_dst_host, long long ldk, double *dK, long long lddk, void *stream) {
    GPRB_REQUIRE(mode == GPRB_FF_FULL || mode == GPRB_FF_UPPER, "gprb_kff_multi: mode must be FULL or UPPER");
    return kff_impl(kernel, f1, f2, p0, p1, zeta, use_tol, tol, mode, grp_begin, grp_end, n_dst, K_dst_host, ldk, dK, lddk,
                    (cudaStream_t)stream);
}

// the rows are the force groups of the window, the columns the energy groups: K_fe is written as it is computed and
// K_ef as its transpose
static int kef_impl(int kernel, const gprb_pack *e, const gprb_pack *f_, double p0, double p1, double zeta,
                    int grp_begin, int grp_end,
                    double *Kef, long long ld_ef, int n_dst, double *const *Kfe_dst, long long ld_fe,
                    double *dKef, long long ld_def, double *dKfe, long long ld_dfe, cudaStream_t st) {
    gprb_pack *f = const_cast<gprb_pack *>(f_);
    int rc = check_dst("gprb_kfe_multi", n_dst, Kfe_dst);
    if (rc) return rc;
    double *Kfe = Kfe_dst[0];
    const bool grad = dKef || dKfe;
    if ((rc = check_cov_args("gprb_kef", kernel, f, 3, e, 0, grp_begin, grp_end, Kef || Kfe, grad))) return rc;
    if (grp_begin == grp_end || e->n_groups == 0) return GPRB_OK;
    if ((rc = build_sched(f, grp_begin, grp_end, st))) return rc;
    const int rows = 3 * (grp_end - grp_begin);
    GPRB_CUDA(zero2d(n_dst == 1 ? Kfe : nullptr, ld_fe, e->n_groups, rows, st));
    GPRB_CUDA(zero2d(dKfe, ld_dfe, e->n_groups, rows, st));
    GPRB_CUDA(zero2d(Kef, ld_ef, rows, e->n_groups, st));
    GPRB_CUDA(zero2d(dKef, ld_def, rows, e->n_groups, st));
    if (f->sched_n == 0 || e->n_rows == 0) return GPRB_OK;
    // RBF with gradient over a whole force pack: the factored build when the pack's rows share atoms (cov_factored.cu)
    if (kernel == GPRB_KERNEL_RBF && grad && grp_begin == 0 && grp_end == f->n_groups && n_dst == 1) {
        bool done = false;
        if ((rc = gprb_kef_factored(e, f, p0, p1, zeta, Kef, ld_ef, Kfe, ld_fe, dKef, ld_def, dKfe, ld_dfe, st, &done))) return rc;
        if (done) return GPRB_OK;
    }
    CovParams P = {};
    if ((rc = init_cov_params(P, kernel, p0, p1, zeta, f, e, grp_begin, grp_end))) return rc;
    P.mode = GPRB_FF_FULL;
    P.K = Kfe; P.ldk = ld_fe; P.dK = dKfe; P.lddk = ld_dfe;
    P.K2 = Kef; P.ldk2 = ld_ef; P.dK2 = dKef; P.lddk2 = ld_def;
    P.n_extra = n_dst - 1;
    for (int p = 1; p < n_dst; p++) P.Kx[p - 1] = Kfe_dst[p];
    return dispatch_cov<1>(kernel, grad, P, f->sched_n, st);
}

extern "C" int gprb_kef(int kernel, const gprb_pack *e, const gprb_pack *f, double p0, double p1, double zeta,
                        int grp_begin, int grp_end,
                        double *Kef, long long ld_ef, double *Kfe, long long ld_fe,
                        double *dKef, long long ld_def, double *dKfe, long long ld_dfe, void *stream) {
    double *dst[1] = {Kfe};
    return kef_impl(kernel, e, f, p0, p1, zeta, grp_begin, grp_end, Kef, ld_ef, 1, dst, ld_fe, dKef, ld_def, dKfe, ld_dfe,
                    (cudaStream_t)stream);
}

extern "C" int gprb_kfe_multi(int kernel, const gprb_pack *e, const gprb_pack *f, double p0, double p1, double zeta,
                              int grp_begin, int grp_end, int n_dst, double *const *Kfe_dst_host, long long ld_fe,
                              double *dKfe, long long ld_dfe, void *stream) {
    GPRB_REQUIRE(Kfe_dst_host && n_dst >= 1 && Kfe_dst_host[0], "gprb_kfe_multi: NULL destination");
    return kef_impl(kernel, e, f, p0, p1, zeta, grp_begin, grp_end, nullptr, 0, n_dst, Kfe_dst_host, ld_fe, nullptr, 0, dKfe, ld_dfe,
                    (cudaStream_t)stream);
}

// K_ee on the same tile machinery (NB = 0: one component per side, 8 DMMAs per 8 x 8 pairs, table exp, tiles without a
// same-species pair skipped).  Replaces rbf_kee_many / rbf_kee_many_with_grad (rbf_kernel.cpp:5-98) and dot_kee_many
// (dot_kernel.cpp:5-56) with the wrappers' 1 / (n_I n_J) (rbf_kernel.py:56-70, dot_kernel.py:46).
extern "C" int gprb_kee(int kernel, const gprb_pack *e1_, const gprb_pack *e2, double p0, double p1, double zeta,
                        int grp_begin, int grp_end, double *K, long long ldk, double *dK, long long lddk, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    gprb_pack *e1 = const_cast<gprb_pack *>(e1_);
    int rc = check_cov_args("gprb_kee", kernel, e1, 0, e2, 0, grp_begin, grp_end, K != nullptr, dK != nullptr);
    if (rc) return rc;
    if (grp_begin == grp_end || e2->n_groups == 0) return GPRB_OK;
    if ((rc = build_sched(e1, grp_begin, grp_end, st))) return rc;
    const int rows = grp_end - grp_begin;
    GPRB_CUDA(zero2d(K, ldk, e2->n_groups, rows, st));
    GPRB_CUDA(zero2d(dK, lddk, e2->n_groups, rows, st));
    if (e1->sched_n == 0 || e2->n_rows == 0) return GPRB_OK;
    CovParams P = {};
    if ((rc = init_cov_params(P, kernel, p0, p1, zeta, e1, e2, grp_begin, grp_end))) return rc;
    P.group_rowsA = e1->d_group_rows;
    // the training block is symmetric: evaluate the J >= I group pairs once, then mirror them
    P.mode = (e1 == e2 && grp_begin == 0 && grp_end == e1->n_groups) ? GPRB_FF_SYMMETRIC : GPRB_FF_FULL;
    P.K = K; P.ldk = ldk; P.dK = dK; P.lddk = lddk;
    rc = dispatch_cov<0>(kernel, dK != nullptr, P, e1->sched_n, st);
    if (rc || P.mode != GPRB_FF_SYMMETRIC) return rc;
    rc = gprb_symmetrize(K, ldk, e1->n_groups, st);
    if (rc == GPRB_OK && dK) rc = gprb_symmetrize(dK, lddk, e1->n_groups, st);
    return rc;
}
