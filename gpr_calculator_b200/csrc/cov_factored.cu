// cov_factored.cu — K_ff with dK/dl over the atoms a structure's force centres share (DESIGN.md §2, §7).
//
// Every force row is the descriptor of an atom of its structure: row a of group I is (I, j) with x^_a = x^(j), and only
// A~ is specific to the row.  The per-pair weights W1, W2 (and U1, U2 of dK/dl) depend on s = x^(j).x^(k) and the
// species only, so the pairwise sum regroups exactly:
//     K_ce(I,J) = sum_j A~_c(I,j) . Z_e(J,j)        Z_e(J,j) = sum_k W1(j,k) B~_e(J,k) + W2(j,k) (x^(j).B~_e(J,k)) x^(k)
// and dK/dl the same with Z' built from (U1, U2).  The weights are formed once per ATOM pair and Z is shared by every
// centre I of the structure.
//
// Atom plan (built once per pack, on the first call that can use it): the groups are cut into clusters of consecutive
// groups whose distinct rows (64-bit hash of the raw x bits and the species code, written by prep_rows_kernel) number
// at most A_MAX; a row maps to (cluster, slot).  Every row is compared bit for bit (x^ and species code) with its
// slot's representative on the device; a mismatch -- a hash collision -- gets a slot of its own.  Two rows of one group
// in the same slot have their A~ summed.  Per cluster S the plan holds X^_S [npad_S x 32] and
//     Acal_S [(3 m_S) x (npad_S * 32)]   row 3(I - I0) + c, column 32 j + d: A~_c(I, j)[d], zero where group I has no row j.
// Per cluster pair (S, T), in batches of pairs that bound the workspace:
//   kff_z_kernel        s, the weights, q_e = x^(j).B~_e(J,k), then Z and Z' -> workspace [6 m_T] x [npad_S * 32]
//   kff_contract_kernel [K | dK](3I+c, 3J+e) = Acal_S . [Z | Z']^T, stored with the UPPER / SYMMETRIC rules of cov_mma.cu
// Both are FP64 m8n8k4 MMA kernels; every output entry is written by exactly one thread with a fixed summation order, so
// the build is bitwise reproducible.
//
// K_fe / K_ef with dK/dl regroup the same way over the force side's atoms (the energy side needs no plan): for energy group
// I (rows a) and force group J of cluster T,
//     K_fe(3J+c, I) = -(1/n_I) sum_k A~_c(J,k) . Y_I(k)      Y_I(k) = sum_{a in I} W1(a,k) x^(a)
// and dK/dl with Y' built from U1.  Per cluster T, in batches of clusters that bound the workspace:
//   kef_y_kernel                 s, the weights, then Y and Y' -> workspace [2 NE] x [npad_T * 32]
//   kff_contract_kernel<true>    [K_fe | dK_fe](3J+c, I) = Acal_T . [Y | Y']^T, stored to K_fe, K_ef and their dK/dl
#include "cov_common.cuh"
#include <cstdlib>
#include <cstring>
#include <vector>
#include <algorithm>

namespace {

constexpr int A_MAX = 128;                 // slots per cluster (S4's 108-atom structures fit)
constexpr int MAX_CLUSTER_GROUPS = 4096;   // groups per cluster: bounds the workspace of one cluster pair
constexpr long long WS_BYTES = 1LL << 30;  // Z workspace of one batch of cluster pairs
constexpr double MIN_GAIN = 2.0;           // the factored path runs when the pairwise kernel executes >= 2x its DMMAs
constexpr double MIN_PAIRWISE_DMMA = 67108864.0;   // below ~1 ms of pairwise work the plan's host round trip does not pay

struct ClusterDev { long long aoff; int grp0, m, npad, slot0; };
struct GroupDev { long long arow; int fr_off, npad; };
struct Batch { int p0, np, max_mt, max_jb, max_mb, max_nb; long long zdoubles; };

struct PairList {
    bool built = false;
    int2 *d_pairs = nullptr;
    long long *d_zoff = nullptr;          // Z offset of each pair inside its batch's workspace (doubles)
    std::vector<Batch> batches;
    long long max_zdoubles = 0;
};

}  // namespace

struct gprb_atom_plan {
    int n_clusters = 0, tot_slots = 0;
    std::vector<ClusterDev> cl;
    ClusterDev *d_cl = nullptr;
    double *Xh = nullptr;                 // [tot_slots][32] x^ of each slot's representative (0 for padding slots)
    int *spec = nullptr;                  // [tot_slots] species code (-1 padding)
    double *Acal = nullptr;
    PairList lists[2];                    // [0] S <= T (UPPER, SYMMETRIC), [1] every pair (FULL)
    double pairwise_dmma[2] = {0, 0}, factored_dmma[2] = {0, 0};
    std::vector<int> cgrp, cslots;        // host copies of gprb_atom_plan_host's cluster_grp / cluster_slots (K_ef cost)
};

void gprb_atom_plan_free(gprb_atom_plan *pl, cudaStream_t st) {
    if (!pl) return;
    gprb_pool_free(pl->d_cl, st); gprb_pool_free(pl->Xh, st); gprb_pool_free(pl->spec, st); gprb_pool_free(pl->Acal, st);
    for (auto &L : pl->lists) { gprb_pool_free(L.d_pairs, st); gprb_pool_free(L.d_zoff, st); }
    delete pl;
}

// ------------------------------------------------------------------------------------------------------------------
// host part of the plan (no device calls: the CPU tests drive it directly)

extern "C" int gprb_atom_plan_host(int n_groups, const int *row_ptr, const unsigned long long *hash, const int *code,
                                   const unsigned char *unique, int a_max, int max_groups,
                                   int *n_clusters, int *cluster_grp, int *cluster_slots, int *row_slot, int *slot_rep) {
    GPRB_REQUIRE(n_groups >= 0 && row_ptr && n_clusters && cluster_grp && cluster_slots, "gprb_atom_plan_host: NULL argument");
    GPRB_REQUIRE(a_max >= 1 && a_max <= 4096 && max_groups >= 1, "gprb_atom_plan_host: bad limits a_max=%d max_groups=%d",
                 a_max, max_groups);
    const int n_rows = row_ptr[n_groups];
    GPRB_REQUIRE(n_rows == 0 || (hash && code && row_slot && slot_rep), "gprb_atom_plan_host: NULL row array");
    // open-addressing table of the current cluster's keys: (hash, code) -> slot
    const int TAB = 2 * 4096;
    std::vector<unsigned long long> th(TAB);
    std::vector<int> tc(TAB), ts(TAB, -1), used;
    auto find = [&](unsigned long long h, int c, bool insert, int slot) -> int {
        int i = (int)((h ^ (h >> 29)) & (TAB - 1));
        while (ts[i] >= 0) {
            if (th[i] == h && tc[i] == c) return ts[i];
            i = (i + 1) & (TAB - 1);
        }
        if (insert) { th[i] = h; tc[i] = c; ts[i] = slot; used.push_back(i); }
        return -1;
    };
    int nc = 0, slots = 0, groups = 0, rep0 = 0;     // current cluster: slots so far, groups, first slot_rep index
    std::vector<std::pair<unsigned long long, int>> gk;
    auto close = [&]() {
        if (groups == 0) return;
        cluster_slots[nc] = slots;
        nc++;
        rep0 += slots;
        slots = 0; groups = 0;
        for (int i : used) ts[i] = -1;
        used.clear();
    };
    for (int g = 0; g < n_groups; g++) {
        const int r0 = row_ptr[g], r1 = row_ptr[g + 1];
        GPRB_REQUIRE(r1 >= r0, "gprb_atom_plan_host: row_ptr not increasing at group %d", g);
        // distinct keys of the group and how many of them the current cluster already has
        gk.clear();
        int n_unique = 0;
        for (int r = r0; r < r1; r++) {
            if (unique && unique[r]) n_unique++;
            else gk.emplace_back(hash[r], code[r]);
        }
        std::sort(gk.begin(), gk.end());
        gk.erase(std::unique(gk.begin(), gk.end()), gk.end());
        const int distinct = (int)gk.size() + n_unique;
        if (distinct > a_max) { *n_clusters = 0; gprb_set_error("gprb_atom_plan_host: group %d has %d distinct rows > %d", g, distinct, a_max); return GPRB_ERR_UNSUPPORTED; }
        int shared = 0;
        for (auto &k : gk) shared += find(k.first, k.second, false, 0) >= 0;
        // a new cluster when the group shares no atom with the current one (next structure), or it would not fit
        if (groups > 0 && r1 > r0 && (shared == 0 || slots + distinct - shared > a_max || groups >= max_groups)) close();
        if (groups == 0) cluster_grp[nc] = g;
        groups++;
        for (int r = r0; r < r1; r++) {
            int s = -1;
            if (!(unique && unique[r])) s = find(hash[r], code[r], false, 0);
            if (s < 0) {
                s = slots++;
                slot_rep[rep0 + s] = r;
                if (!(unique && unique[r])) find(hash[r], code[r], true, s);
            }
            row_slot[r] = s;
        }
    }
    close();
    cluster_grp[nc] = n_groups;
    *n_clusters = nc;
    return GPRB_OK;
}

namespace {

int pad8(int n) { return (n + 7) & ~7; }

// DMMAs the two paths execute.  Pairwise (cov_mma_kernel<4, 8, RBF, grad>): 128 per pair of 8-row tiles.  Factored, per
// cluster pair: kff_z_kernel 128 per (J, 8 slots of S, 8 slots of T); kff_contract_kernel (3 m_S / 8)(6 m_T / 8)(8 npad_S).
void plan_costs(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows, int upper,
                double *pairwise, double *factored) {
    const double tiles = (double)((n_rows + 7) / 8);
    *pairwise = 128.0 * (upper ? 0.5 * tiles * (tiles + 1.0) : tiles * tiles);
    double f = 0.0;
    for (int S = 0; S < n_clusters; S++) {
        const double ns = pad8(cluster_slots[S]), ms = cluster_grp[S + 1] - cluster_grp[S];
        for (int T = upper ? S : 0; T < n_clusters; T++) {
            const double nt = pad8(cluster_slots[T]), mt = cluster_grp[T + 1] - cluster_grp[T];
            f += 128.0 * mt * (ns / 8) * (nt / 8) + std::ceil(3 * ms / 8) * std::ceil(6 * mt / 8) * 8 * ns;
        }
    }
    *factored = f;
}

// The same for K_fe + dK/dl against an energy pack of ne_rows rows in ne groups.  Pairwise (cov_mma_kernel<1, 8, RBF,
// grad>): 32 per pair of 8-row tiles (4 component tiles x 8 k-steps).  Factored, per cluster T: kef_y_kernel 24 per
// (energy tile, 8 slots of T); kff_contract_kernel<true> (3 m_T / 8)(2 NE / 8)(8 npad_T).
void plan_costs_kef(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows, int ne_rows, int ne,
                    double *pairwise, double *factored) {
    const double etiles = (double)((ne_rows + 7) / 8);
    *pairwise = 32.0 * (double)((n_rows + 7) / 8) * etiles;
    double f = 0.0;
    for (int T = 0; T < n_clusters; T++) {
        const double nt = pad8(cluster_slots[T]), mt = cluster_grp[T + 1] - cluster_grp[T];
        f += 24.0 * etiles * (nt / 8) + std::ceil(3 * mt / 8) * std::ceil(2.0 * ne / 8) * 8 * nt;
    }
    *factored = f;
}

}  // namespace

extern "C" int gprb_atom_plan_cost(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows, int upper,
                                   double *pairwise_dmma, double *factored_dmma) {
    GPRB_REQUIRE(n_clusters >= 0 && (n_clusters == 0 || (cluster_grp && cluster_slots)) && pairwise_dmma && factored_dmma,
                 "gprb_atom_plan_cost: NULL argument");
    plan_costs(n_clusters, cluster_grp, cluster_slots, n_rows, upper, pairwise_dmma, factored_dmma);
    return GPRB_OK;
}

extern "C" int gprb_atom_plan_cost_kef(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows,
                                       int n_energy_rows, int n_energy_groups, double *pairwise_dmma, double *factored_dmma) {
    GPRB_REQUIRE(n_clusters >= 0 && (n_clusters == 0 || (cluster_grp && cluster_slots)) && pairwise_dmma && factored_dmma,
                 "gprb_atom_plan_cost_kef: NULL argument");
    GPRB_REQUIRE(n_rows >= 0 && n_energy_rows >= 0 && n_energy_groups >= 0, "gprb_atom_plan_cost_kef: negative size");
    plan_costs_kef(n_clusters, cluster_grp, cluster_slots, n_rows, n_energy_rows, n_energy_groups, pairwise_dmma,
                   factored_dmma);
    return GPRB_OK;
}

namespace {

// ------------------------------------------------------------------------------------------------------------------
// plan kernels (once per pack).  Pack slab of row r, component c (0 = x^, 1..3 = A~ columns), entry k (ks = 8):
__device__ __forceinline__ size_t slab(int r, int c, int k) {
    return ((size_t)((r >> 3) * 4 + c) * GPRB_MAX_KS + (k >> 2)) * 32 + (r & 7) * 4 + (k & 3);
}

__global__ void plan_gather_x_kernel(int tot_slots, const int *__restrict__ rep, const double *__restrict__ P,
                                     const int *__restrict__ elep, double *__restrict__ Xh, int *__restrict__ spec) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)tot_slots * 32) return;
    const int s = (int)(i >> 5), k = (int)(i & 31), r = rep[s];
    Xh[i] = r >= 0 ? P[slab(r, 0, k)] : 0.0;
    if (k == 0) spec[s] = r >= 0 ? elep[r] : -1;
}

// every row against its slot: species code and x^ bit for bit
__global__ void plan_verify_kernel(int n_rows, const int *__restrict__ row_gslot, const double *__restrict__ P,
                                   const int *__restrict__ elep, const double *__restrict__ Xh, const int *__restrict__ spec,
                                   unsigned char *__restrict__ bad, int *__restrict__ n_bad) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int s = row_gslot[r];
    bool ok = elep[r] == spec[s];
    for (int k = 0; k < 32; k++)
        ok = ok && __double_as_longlong(P[slab(r, 0, k)]) == __double_as_longlong(Xh[(size_t)s * 32 + k]);
    bad[r] = ok ? 0 : 1;
    if (!ok) atomicAdd(n_bad, 1);
}

// one block per group: Acal rows 3(I - I0) + c, A~ of the group's rows summed per slot in row order
__global__ void plan_gather_a_kernel(const GroupDev *__restrict__ gd, const int *__restrict__ first_row,
                                     const int *__restrict__ next_row, const double *__restrict__ P, double *__restrict__ Acal) {
    const GroupDev g = gd[blockIdx.x];
    const int n = 3 * g.npad * 32;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = i / (g.npad * 32), rem = i - c * g.npad * 32, j = rem >> 5, k = rem & 31;
        double v = 0.0;
        for (int r = first_row[g.fr_off + j]; r >= 0; r = next_row[r]) v += P[slab(r, 1 + c, k)];
        Acal[g.arow + i] = v;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// build kernels

struct FactArgs {
    const ClusterDev *cl; const int2 *pairs; const long long *zoff;
    const double *Xh; const int *spec; const double *Acal; double *Zw;
};

// CTA = (cluster pair, group J of T, up to 4 tiles of 8 slots of S); warp = one 8-slot tile j of S, all 32 columns d.
// Per 8 slots k of T: s (8 DMMAs) and q_e (24) with the x^(j) fragments as A operand, the weights of this thread's two
// (j, k) pairs, then Z_e += W1 B~_e + (W2 q_e) x^ and Z'_e likewise (96): the accumulator fragment of s / q is the A
// fragment of the second product with the k order k0 + 2 q4 + jj (the two-stage idea of cov_mma.cu).
template <int ZI>
__global__ void __launch_bounds__(128) kff_z_kernel(const FactArgs A, const CovParams P, int p0) {
    __shared__ double sTab[EXP_TAB];
    if (threadIdx.x < EXP_TAB) sTab[threadIdx.x] = d_exp2_tab[threadIdx.x];
    __syncthreads();
    const int2 st = A.pairs[p0 + blockIdx.x];
    const ClusterDev cS = A.cl[st.x], cT = A.cl[st.y];
    const int J = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, ra = lane >> 2, q4 = lane & 3;
    const int jt = blockIdx.z * 4 + warp;
    if (J >= cT.m || jt * 8 >= cS.npad) return;

    const double *XT = A.Xh + (size_t)cT.slot0 * 32;
    const int *spT = A.spec + cT.slot0;
    const size_t ldA = (size_t)cT.npad * 32;
    const double *BT = A.Acal + cT.aoff + (size_t)(3 * J) * ldA;     // B~_e(J, k)[d] = BT[e ldA + 32 k + d]
    double xa[8];
    {
        const double *XS = A.Xh + (size_t)(cS.slot0 + jt * 8 + ra) * 32 + q4;
#pragma unroll
        for (int ks = 0; ks < 8; ks++) xa[ks] = XS[4 * ks];
    }
    const int ea = A.spec[cS.slot0 + jt * 8 + ra];
    double Z[2][3][4][2];
#pragma unroll
    for (int w = 0; w < 2; w++)
#pragma unroll
        for (int e = 0; e < 3; e++)
#pragma unroll
            for (int t = 0; t < 4; t++) { Z[w][e][t][0] = 0.0; Z[w][e][t][1] = 0.0; }

    for (int k0 = 0; k0 < cT.npad; k0 += 8) {
        double s[2] = {0.0, 0.0}, q[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
        {
            const double *xb = XT + (size_t)(k0 + ra) * 32 + q4;
#pragma unroll
            for (int ks = 0; ks < 8; ks++) dmma(s[0], s[1], xa[ks], xb[4 * ks]);
#pragma unroll
            for (int e = 0; e < 3; e++) {
                const double *bb = BT + e * ldA + (size_t)(k0 + ra) * 32 + q4;
#pragma unroll
                for (int ks = 0; ks < 8; ks++) dmma(q[e][0], q[e][1], xa[ks], bb[4 * ks]);
            }
        }
#pragma unroll
        for (int jj = 0; jj < 2; jj++) {
            const int eb = spT[k0 + 2 * q4 + jj];
            bool valid = (ea == eb) && (ea >= 0);
            double w1 = 0.0, w2 = 0.0, u1 = 0.0, u2 = 0.0;
            pair_weights<GPRB_KERNEL_RBF, true, true, ZI>(P, sTab, s[jj], valid, w1, w2, u1, u2);
            const double W1 = valid ? w1 : 0.0, W2 = valid ? w2 : 0.0, U1 = valid ? u1 : 0.0, U2 = valid ? u2 : 0.0;
            // k-step over the slots k0 + 2 q4 + jj: B fragment element (k = q4, n = ra) is row k0 + 2 q4 + jj, column 8 t + ra
            const double *xr = XT + (size_t)(k0 + 2 * q4 + jj) * 32 + ra;
            const double *br = BT + (size_t)(k0 + 2 * q4 + jj) * 32 + ra;
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const double bx = xr[8 * t];
#pragma unroll
                for (int e = 0; e < 3; e++) {
                    const double bb = br[e * ldA + 8 * t];
                    dmma(Z[0][e][t][0], Z[0][e][t][1], W1, bb);
                    dmma(Z[0][e][t][0], Z[0][e][t][1], W2 * q[e][jj], bx);
                    dmma(Z[1][e][t][0], Z[1][e][t][1], U1, bb);
                    dmma(Z[1][e][t][0], Z[1][e][t][1], U2 * q[e][jj], bx);
                }
            }
        }
    }
    // Z rows: [w][3 J + e] of the pair's [6 m_T] x [npad_S * 32] block
    const size_t ldz = (size_t)cS.npad * 32;
    double *zp = A.Zw + A.zoff[p0 + blockIdx.x] + (size_t)(jt * 8 + ra) * 32 + 2 * q4;
#pragma unroll
    for (int w = 0; w < 2; w++)
#pragma unroll
        for (int e = 0; e < 3; e++)
#pragma unroll
            for (int t = 0; t < 4; t++)
                *reinterpret_cast<double2 *>(zp + (size_t)(w * 3 * cT.m + 3 * J + e) * ldz + 8 * t) =
                    make_double2(Z[w][e][t][0], Z[w][e][t][1]);
}

// Energy side of the K_ef build: the energy pack's x^ slab (one component, ks = 8) in flat 8-row tiles and its groups.
struct KefE { const double *P; const int *elep; const int *row_ptr; int ne; };

// CTA = (energy group I, cluster T0 + blockIdx.y, up to 4 tiles of 8 slots of T); warp = one 8-slot tile k of T, all 32
// columns d.  Per energy tile holding rows of I: s^T = X^_T . x^_a^T (8 DMMAs) with the slots as A operand, the weights of
// this thread's two (k, a) pairs (rows of other groups masked), then Y += W1 x^ and Y' += U1 x^ (16): the accumulator
// fragment of s^T is the A fragment of the second product with the row order a = 2 q4 + jj.  A tile shared by two groups
// is multiplied once for each.
template <int ZI>
__global__ void __launch_bounds__(128) kef_y_kernel(const FactArgs A, const CovParams P, const KefE E, int T0) {
    __shared__ double sTab[EXP_TAB];
    if (threadIdx.x < EXP_TAB) sTab[threadIdx.x] = d_exp2_tab[threadIdx.x];
    __syncthreads();
    const int I = blockIdx.x, T = T0 + blockIdx.y;
    const ClusterDev cT = A.cl[T];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, ra = lane >> 2, q4 = lane & 3;
    const int kt = blockIdx.z * 4 + warp;
    if (kt * 8 >= cT.npad) return;

    double xa[8];
    {
        const double *XT = A.Xh + (size_t)(cT.slot0 + kt * 8 + ra) * 32 + q4;
#pragma unroll
        for (int ks = 0; ks < 8; ks++) xa[ks] = XT[4 * ks];
    }
    const int ek = A.spec[cT.slot0 + kt * 8 + ra];
    const int r0 = E.row_ptr[I], r1 = E.row_ptr[I + 1];
    double Y[2][4][2];
#pragma unroll
    for (int w = 0; w < 2; w++)
#pragma unroll
        for (int t = 0; t < 4; t++) { Y[w][t][0] = 0.0; Y[w][t][1] = 0.0; }

    for (int tile = r0 >> 3; tile * 8 < r1; tile++) {
        const double *pe = E.P + (size_t)tile * GPRB_MAX_KS * 32;     // fragment (k-step ks) = pe[32 ks + lane]
        double s[2] = {0.0, 0.0};
#pragma unroll
        for (int ks = 0; ks < 8; ks++) dmma(s[0], s[1], xa[ks], pe[32 * ks + lane]);
#pragma unroll
        for (int jj = 0; jj < 2; jj++) {
            const int a = tile * 8 + 2 * q4 + jj;
            bool valid = a >= r0 && a < r1 && ek >= 0 && ek == E.elep[a];
            double w1 = 0.0, w2 = 0.0, u1 = 0.0, u2 = 0.0;
            pair_weights<GPRB_KERNEL_RBF, true, false, ZI>(P, sTab, s[jj], valid, w1, w2, u1, u2);
            const double W1 = valid ? w1 : 0.0, U1 = valid ? u1 : 0.0;
#pragma unroll
            for (int t = 0; t < 4; t++) {
                // B fragment element (k = q4, n = ra) is x^(a)[8 t + ra]: k-step 2 t + ra / 4, entry ra % 4 of row 2 q4 + jj
                const double bx = pe[(2 * t + (ra >> 2)) * 32 + (2 * q4 + jj) * 4 + (ra & 3)];
                dmma(Y[0][t][0], Y[0][t][1], W1, bx);
                dmma(Y[1][t][0], Y[1][t][1], U1, bx);
            }
        }
    }
    // Y rows: [w][I] of the cluster's [2 NE] x [npad_T * 32] block (row-major, the contraction's B operand)
    const size_t ldy = (size_t)cT.npad * 32;
    double *yp = A.Zw + (size_t)2 * E.ne * 32 * (cT.slot0 - A.cl[T0].slot0) + (size_t)(kt * 8 + ra) * 32 + 2 * q4;
#pragma unroll
    for (int w = 0; w < 2; w++)
#pragma unroll
        for (int t = 0; t < 4; t++)
            *reinterpret_cast<double2 *>(yp + (size_t)(w * E.ne + I) * ldy + 8 * t) = make_double2(Y[w][t][0], Y[w][t][1]);
}

constexpr int CT = 64, CK = 32, SST = CK + 4;      // CTA tile, k chunk, shared-memory row stride (conflict-free fragments)
constexpr size_t CONTRACT_SMEM = (size_t)2 * 2 * CT * SST * sizeof(double);

// Outputs of kff_contract_kernel.  K_ff: K / dK with the UPPER / SYMMETRIC / FULL rules of `mode`.  K_ef: K = K_fe,
// dK = dK_fe/dl ([3 NF] x [NE]), K2 = K_ef, dK2 = dK_ef/dl ([NE] x [3 NF]), each written when not NULL.
struct ContractOut {
    double *K, *dK, *K2, *dK2;
    long long ldk, lddk, ldk2, lddk2;
    int mode, ne;
    const int *group_rowsE;          // K_ef: rows per energy group (the pairwise epilogue's -1 / n_I)
};

__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// C [3 m_S] x [N] = Acal_S . Zw^T (K-dimension npad_S * 32); CTA tile 64 x 64, 4 warps of 32 x 32, 2-stage cp.async ring.
// Grid: (unit, m tile, n tile).  K_ff (KEF = false): unit = cluster pair p0 + u (S, T), N = 6 m_T; column n < 3 m_T is K(3I+c, 3J+e), the rest dK/dl;
// UPPER / SYMMETRIC: group blocks J >= I only (and their mirror).
// K_ef (KEF = true): unit = cluster S = p0 + u, N = 2 NE; column n < NE is K_fe(3J+c, n), the rest dK_fe/dl.
template <bool KEF>
__global__ void __launch_bounds__(128) kff_contract_kernel(const FactArgs A, int p0, const ContractOut O) {
    extern __shared__ __align__(16) double smem_c[];
    const int u = blockIdx.x;
    int S, N;
    const double *Bb;
    ClusterDev cT = {};
    if (KEF) {
        S = p0 + u;
        N = 2 * O.ne;
        Bb = A.Zw + (size_t)2 * O.ne * 32 * (A.cl[S].slot0 - A.cl[p0].slot0);
    } else {
        const int2 st = A.pairs[p0 + u];
        S = st.x;
        cT = A.cl[st.y];
        N = 6 * cT.m;
        Bb = A.Zw + A.zoff[p0 + u];
    }
    const ClusterDev cS = A.cl[S];
    const int M = 3 * cS.m, Kd = cS.npad * 32;
    const int m0 = blockIdx.y * CT, n0 = blockIdx.z * CT;
    if (m0 >= M || n0 >= N) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ra = lane >> 2, q4 = lane & 3;
    const int wm = warp >> 1, wn = warp & 1;
    const bool active = m0 + 32 * wm < M && n0 + 32 * wn < N;
    const double *Ab = A.Acal + cS.aoff;
    double *sA = smem_c, *sB = smem_c + 2 * CT * SST;

    auto load = [&](int buf, int k0) {
        for (int i = tid; i < CT * CK / 2; i += 128) {
            const int row = i >> 4, col = (i & 15) * 2;
            const int ar = min(m0 + row, M - 1), br = min(n0 + row, N - 1);   // rows past the end feed outputs never stored
            cp_async16(sA + buf * CT * SST + row * SST + col, Ab + (size_t)ar * Kd + k0 + col);
            cp_async16(sB + buf * CT * SST + row * SST + col, Bb + (size_t)br * Kd + k0 + col);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    const int nk = Kd / CK;
    load(0, 0);
    for (int kc = 0; kc < nk; kc++) {
        if (kc + 1 < nk) {
            load((kc + 1) & 1, (kc + 1) * CK);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        if (active) {
            const double *a = sA + (kc & 1) * CT * SST + (32 * wm + ra) * SST + q4;
            const double *b = sB + (kc & 1) * CT * SST + (32 * wn + ra) * SST + q4;
#pragma unroll
            for (int kk = 0; kk < CK / 4; kk++) {
                double af[4], bf[4];
#pragma unroll
                for (int i = 0; i < 4; i++) { af[i] = a[i * 8 * SST + 4 * kk]; bf[i] = b[i * 8 * SST + 4 * kk]; }
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
        }
        __syncthreads();
    }
    if (!active) return;
    const int nG = KEF ? O.ne : 3 * cT.m;       // columns per output (K, then dK/dl)
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = m0 + 32 * wm + 8 * i + ra;
        if (r >= M) continue;
        const int I = cS.grp0 + r / 3, c = r % 3;
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int n = n0 + 32 * wn + 8 * j + 2 * q4 + h;
                if (n >= N) continue;
                const bool grad = n >= nG;
                const int nn = grad ? n - nG : n;
                const double v = acc[i][j][h];
                if (KEF) {
                    // force group I, energy group nn: K_fe = -(1 / n_nn) sum, as the pairwise NB = 1 epilogue
                    const int nE = O.group_rowsE[nn];
                    const double val = nE > 0 ? -v / (double)nE : 0.0;
                    double *fe = grad ? O.dK : O.K, *ef = grad ? O.dK2 : O.K2;
                    if (fe) fe[(long long)(3 * I + c) * (grad ? O.lddk : O.ldk) + nn] = val;
                    if (ef) ef[(long long)nn * (grad ? O.lddk2 : O.ldk2) + 3 * I + c] = val;
                } else {
                    const int J = cT.grp0 + nn / 3, e = nn % 3;
                    double *dst = grad ? O.dK : O.K;
                    const long long ld = grad ? O.lddk : O.ldk;
                    if (O.mode == GPRB_FF_FULL || J >= I) dst[(long long)(3 * I + c) * ld + 3 * J + e] = v;
                    if (O.mode == GPRB_FF_SYMMETRIC && J > I) dst[(long long)(3 * J + e) * ld + 3 * I + c] = v;
                }
            }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// host: plan construction and the build

#define FP_CUDA(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { gprb_set_error("%s:%d CUDA error %s", __FILE__, __LINE__, cudaGetErrorString(_e)); gprb_atom_plan_free(pl, st); return GPRB_ERR_CUDA; } } while (0)

template <typename T>
cudaError_t upload(T **dst, const std::vector<T> &v, cudaStream_t st) {
    cudaError_t e = cudaMallocAsync((void **)dst, (v.empty() ? 1 : v.size()) * sizeof(T), st);
    if (e == cudaSuccess && !v.empty()) e = cudaMemcpyAsync(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st);
    return e;
}

// *out = NULL (and GPRB_OK) when the pack has no plan: a group with more than A_MAX distinct rows, or collisions that do not
// resolve
int build_plan(gprb_pack *f, cudaStream_t st, gprb_atom_plan **out) {
    *out = nullptr;
    gprb_atom_plan *pl = new gprb_atom_plan();
    const int G = f->n_groups, R = f->n_rows;
    std::vector<unsigned long long> hash(R);
    std::vector<int> code(R);
    FP_CUDA(cudaMemcpyAsync(hash.data(), f->row_hash, (size_t)R * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    FP_CUDA(cudaMemcpyAsync(code.data(), f->elep, (size_t)R * sizeof(int), cudaMemcpyDeviceToHost, st));
    FP_CUDA(cudaStreamSynchronize(st));
    std::vector<unsigned char> unique(R, 0), bad(R);
    std::vector<int> cgrp(G + 1), cslots(G + 1), row_slot(R), slot_rep(R), row_gslot(R);
    int nc = 0;
    int *d_rep = nullptr, *d_row_gslot = nullptr, *d_nbad = nullptr;
    unsigned char *d_bad = nullptr;
    for (int attempt = 0;; attempt++) {
        int rc = gprb_atom_plan_host(G, f->row_ptr.data(), hash.data(), code.data(), unique.data(), A_MAX, MAX_CLUSTER_GROUPS,
                                     &nc, cgrp.data(), cslots.data(), row_slot.data(), slot_rep.data());
        if (rc == GPRB_ERR_UNSUPPORTED) { gprb_atom_plan_free(pl, st); return GPRB_OK; }
        if (rc) { gprb_atom_plan_free(pl, st); return rc; }
        pl->n_clusters = nc;
        pl->cl.assign(nc, {});
        std::vector<int> rep;
        long long aoff = 0;
        int slot0 = 0, rep0 = 0;
        for (int c = 0; c < nc; c++) {
            ClusterDev &C = pl->cl[c];
            C.grp0 = cgrp[c]; C.m = cgrp[c + 1] - cgrp[c]; C.npad = pad8(cslots[c] > 0 ? cslots[c] : 1);
            C.slot0 = slot0; C.aoff = aoff;
            for (int j = 0; j < C.npad; j++) rep.push_back(j < cslots[c] ? slot_rep[rep0 + j] : -1);
            for (int g = C.grp0; g < C.grp0 + C.m; g++)
                for (int r = f->row_ptr[g]; r < f->row_ptr[g + 1]; r++) row_gslot[r] = slot0 + row_slot[r];
            slot0 += C.npad; rep0 += cslots[c];
            aoff += (long long)3 * C.m * C.npad * 32;
        }
        pl->tot_slots = slot0;
        gprb_pool_free(pl->Xh, st); gprb_pool_free(pl->spec, st); gprb_pool_free(d_rep, st); gprb_pool_free(d_row_gslot, st);
        pl->Xh = nullptr; pl->spec = nullptr;
        FP_CUDA(upload(&d_rep, rep, st));
        FP_CUDA(upload(&d_row_gslot, row_gslot, st));
        FP_CUDA(cudaMallocAsync((void **)&pl->Xh, (size_t)slot0 * 32 * sizeof(double), st));
        FP_CUDA(cudaMallocAsync((void **)&pl->spec, (size_t)slot0 * sizeof(int), st));
        if (!d_bad) {
            FP_CUDA(cudaMallocAsync((void **)&d_bad, (size_t)(R > 0 ? R : 1), st));
            FP_CUDA(cudaMallocAsync((void **)&d_nbad, sizeof(int), st));
        }
        FP_CUDA(cudaMemsetAsync(d_nbad, 0, sizeof(int), st));
        {
            const long long n = (long long)slot0 * 32;
            plan_gather_x_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(slot0, d_rep, f->P, f->elep, pl->Xh, pl->spec);
            GPRB_LAUNCHED();
            FP_CUDA(cudaGetLastError());
        }
        if (R > 0) {
            plan_verify_kernel<<<(R + 255) / 256, 256, 0, st>>>(R, d_row_gslot, f->P, f->elep, pl->Xh, pl->spec, d_bad, d_nbad);
            GPRB_LAUNCHED();
            FP_CUDA(cudaGetLastError());
        }
        int nbad = 0;
        FP_CUDA(cudaMemcpyAsync(&nbad, d_nbad, sizeof(int), cudaMemcpyDeviceToHost, st));
        FP_CUDA(cudaStreamSynchronize(st));
        if (nbad == 0) break;
        // hash collisions: the rows that differ from their slot's representative get slots of their own
        if (attempt >= 1) {
            gprb_pool_free(d_rep, st); gprb_pool_free(d_row_gslot, st); gprb_pool_free(d_bad, st); gprb_pool_free(d_nbad, st);
            gprb_atom_plan_free(pl, st);
            return GPRB_OK;
        }
        FP_CUDA(cudaMemcpyAsync(bad.data(), d_bad, (size_t)R, cudaMemcpyDeviceToHost, st));
        FP_CUDA(cudaStreamSynchronize(st));
        for (int r = 0; r < R; r++) unique[r] |= bad[r];
    }
    gprb_pool_free(d_rep, st); gprb_pool_free(d_row_gslot, st); gprb_pool_free(d_bad, st); gprb_pool_free(d_nbad, st);

    // Acal: per group and slot the chain of its rows (increasing row order)
    std::vector<GroupDev> gd(G);
    std::vector<int> first_row, next_row(R > 0 ? R : 1, -1);
    for (int c = 0; c < nc; c++) {
        const ClusterDev &C = pl->cl[c];
        for (int g = C.grp0; g < C.grp0 + C.m; g++) {
            GroupDev &D = gd[g];
            D.npad = C.npad;
            D.fr_off = (int)first_row.size();
            D.arow = C.aoff + (long long)3 * (g - C.grp0) * C.npad * 32;
            first_row.resize(first_row.size() + C.npad, -1);
            for (int r = f->row_ptr[g + 1] - 1; r >= f->row_ptr[g]; r--) {
                int &head = first_row[D.fr_off + row_slot[r]];
                next_row[r] = head;
                head = r;
            }
        }
    }
    const long long a_total = nc > 0 ? pl->cl[nc - 1].aoff + (long long)3 * pl->cl[nc - 1].m * pl->cl[nc - 1].npad * 32 : 0;
    GroupDev *d_gd = nullptr;
    int *d_first = nullptr, *d_next = nullptr;
    FP_CUDA(upload(&d_gd, gd, st));
    FP_CUDA(upload(&d_first, first_row, st));
    FP_CUDA(upload(&d_next, next_row, st));
    FP_CUDA(upload(&pl->d_cl, pl->cl, st));
    FP_CUDA(cudaMallocAsync((void **)&pl->Acal, (size_t)(a_total > 0 ? a_total : 1) * sizeof(double), st));
    if (G > 0) {
        plan_gather_a_kernel<<<G, 256, 0, st>>>(d_gd, d_first, d_next, f->P, pl->Acal);
        GPRB_LAUNCHED();
        FP_CUDA(cudaGetLastError());
    }
    gprb_pool_free(d_gd, st); gprb_pool_free(d_first, st); gprb_pool_free(d_next, st);
    for (int u = 0; u < 2; u++)
        plan_costs(nc, cgrp.data(), cslots.data(), R, u == 0, &pl->pairwise_dmma[u], &pl->factored_dmma[u]);
    pl->cgrp.assign(cgrp.begin(), cgrp.begin() + nc + 1);
    pl->cslots.assign(cslots.begin(), cslots.begin() + nc);
    // the host vectors die at return: make the pageable copies explicit and surface faults of the plan kernels here
    FP_CUDA(cudaStreamSynchronize(st));
    *out = pl;
    return GPRB_OK;
}

int build_pairs(gprb_atom_plan *pl, int kind, cudaStream_t st) {
    PairList &L = pl->lists[kind];
    if (L.built) return GPRB_OK;
    std::vector<int2> pairs;
    std::vector<long long> zoff;
    Batch b = {0, 0, 0, 0, 0, 0, 0};
    auto flush = [&]() { if (b.np) { L.batches.push_back(b); L.max_zdoubles = std::max(L.max_zdoubles, b.zdoubles); } };
    for (int S = 0; S < pl->n_clusters; S++)
        for (int T = kind == 0 ? S : 0; T < pl->n_clusters; T++) {
            const ClusterDev &cS = pl->cl[S], &cT = pl->cl[T];
            const long long z = (long long)6 * cT.m * cS.npad * 32;
            if (b.np > 0 && (b.zdoubles + z) * (long long)sizeof(double) > WS_BYTES) {
                flush();
                b = {(int)pairs.size(), 0, 0, 0, 0, 0, 0};
            }
            pairs.push_back(make_int2(S, T));
            zoff.push_back(b.zdoubles);
            b.np++;
            b.zdoubles += z;
            b.max_mt = std::max(b.max_mt, cT.m);
            b.max_jb = std::max(b.max_jb, (cS.npad + 31) / 32);
            b.max_mb = std::max(b.max_mb, (3 * cS.m + CT - 1) / CT);
            b.max_nb = std::max(b.max_nb, (6 * cT.m + CT - 1) / CT);
        }
    flush();
    GPRB_CUDA(upload(&L.d_pairs, pairs, st));
    GPRB_CUDA(upload(&L.d_zoff, zoff, st));
    GPRB_CUDA(cudaStreamSynchronize(st));      // pageable sources
    L.built = true;
    return GPRB_OK;
}

constexpr int MAX_DEV_F = 64;

template <bool KEF>
int contract_config() {
    static bool configured[MAX_DEV_F] = {};
    int dev = 0;
    GPRB_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < MAX_DEV_F && !configured[dev]) {
        GPRB_CUDA(cudaFuncSetAttribute(kff_contract_kernel<KEF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)CONTRACT_SMEM));
        configured[dev] = true;
    }
    return GPRB_OK;
}

template <int ZI>
int run_batches(gprb_atom_plan *pl, PairList &L, const CovParams &P, const ContractOut &O, cudaStream_t st) {
    int rc = contract_config<false>();
    if (rc) return rc;
    FactArgs A = {pl->d_cl, L.d_pairs, L.d_zoff, pl->Xh, pl->spec, pl->Acal, nullptr};
    GPRB_CUDA(cudaMallocAsync((void **)&A.Zw, (size_t)L.max_zdoubles * sizeof(double), st));
    for (const Batch &b : L.batches) {
        kff_z_kernel<ZI><<<dim3(b.np, b.max_mt, b.max_jb), 128, 0, st>>>(A, P, b.p0);
        GPRB_LAUNCHED();
        kff_contract_kernel<false><<<dim3(b.np, b.max_mb, b.max_nb), 128, CONTRACT_SMEM, st>>>(A, b.p0, O);
        GPRB_LAUNCHED();
    }
    const cudaError_t e = cudaGetLastError();
    gprb_pool_free(A.Zw, st);
    GPRB_CUDA(e);
    return GPRB_OK;
}

// K_ef: batches of consecutive clusters whose Y workspace stays within WS_BYTES (and 65535 clusters: grid y)
template <int ZI>
int run_kef(gprb_atom_plan *pl, const KefE &E, const CovParams &P, const ContractOut &O, cudaStream_t st) {
    int rc = contract_config<true>();
    if (rc) return rc;
    struct KBatch { int T0, nT, max_kb, max_mb; };
    std::vector<KBatch> batches;
    const long long per_slot = (long long)2 * E.ne * 32;        // Y doubles per slot of a cluster
    long long ws = 0, max_ws = 0;
    for (int T = 0; T < pl->n_clusters; T++) {
        const ClusterDev &c = pl->cl[T];
        const long long y = per_slot * c.npad;
        if (batches.empty() || (ws + y) * (long long)sizeof(double) > WS_BYTES || batches.back().nT == 65535) {
            batches.push_back({T, 0, 0, 0});
            ws = 0;
        }
        KBatch &b = batches.back();
        b.nT++;
        b.max_kb = std::max(b.max_kb, (c.npad + 31) / 32);
        b.max_mb = std::max(b.max_mb, (3 * c.m + CT - 1) / CT);
        ws += y;
        max_ws = std::max(max_ws, ws);
    }
    const int nb = (2 * E.ne + CT - 1) / CT;
    FactArgs A = {pl->d_cl, nullptr, nullptr, pl->Xh, pl->spec, pl->Acal, nullptr};
    GPRB_CUDA(cudaMallocAsync((void **)&A.Zw, (size_t)max_ws * sizeof(double), st));
    for (const KBatch &b : batches) {
        kef_y_kernel<ZI><<<dim3(E.ne, b.nT, b.max_kb), 128, 0, st>>>(A, P, E, b.T0);
        GPRB_LAUNCHED();
        kff_contract_kernel<true><<<dim3(b.nT, b.max_mb, nb), 128, CONTRACT_SMEM, st>>>(A, b.T0, O);
        GPRB_LAUNCHED();
    }
    const cudaError_t e = cudaGetLastError();
    gprb_pool_free(A.Zw, st);
    GPRB_CUDA(e);
    return GPRB_OK;
}

// GPRB_KFF_FACTORED: '0' keeps the pairwise kernels, '1' takes a factored build whenever the pack has a plan (tests on
// small packs), unset leaves it to the cost model.  The switch governs K_ff and K_ef alike.
void factored_switch(bool *off, bool *force) {
    const char *env = getenv("GPRB_KFF_FACTORED");
    *off = env && env[0] == '0';
    *force = env && env[0] == '1';
}

// the pack's atom plan, built on the first call that can use it; NULL when the pack has none
int pack_plan(gprb_pack *f, cudaStream_t st, gprb_atom_plan **out) {
    if (!f->plan_tried) {
        f->plan_tried = true;
        int rc = build_plan(f, st, &f->plan);
        if (rc) return rc;
    }
    *out = f->plan && f->plan->n_clusters > 0 ? f->plan : nullptr;
    return GPRB_OK;
}

}  // namespace

// K_ff + dK/dl of pack f against itself over the full window with one destination (the caller checked that and zeroed K
// and dK).  *done = false: the pairwise kernel is to run (GPRB_KFF_FACTORED=0, no plan, or the plan does not pay).
int gprb_kff_factored(gprb_pack *f, double p0, double p1, double zeta, int mode, double *K, long long ldk, double *dK,
                      long long lddk, cudaStream_t st, bool *done) {
    *done = false;
    bool off, force;
    factored_switch(&off, &force);
    if (off || f->ks != GPRB_MAX_KS || f->n_rows == 0 || mode == GPRB_FF_DIAG) return GPRB_OK;
    const int kind = mode == GPRB_FF_FULL ? 1 : 0;
    if (!force) {
        const double tiles = (double)((f->n_rows + 7) / 8);
        if (128.0 * (kind ? tiles * tiles : 0.5 * tiles * (tiles + 1.0)) < MIN_PAIRWISE_DMMA) return GPRB_OK;
    }
    gprb_atom_plan *pl = nullptr;
    int rc = pack_plan(f, st, &pl);
    if (rc || !pl) return rc;
    if (!force && pl->pairwise_dmma[kind] < MIN_GAIN * pl->factored_dmma[kind]) return GPRB_OK;
    CovParams P = {};
    if ((rc = fill_kernel_params(P, GPRB_KERNEL_RBF, p0, p1, zeta))) return rc;
    if ((rc = build_pairs(pl, kind, st))) return rc;
    ContractOut O = {};
    O.K = K; O.ldk = ldk; O.dK = dK; O.lddk = lddk; O.mode = mode;
    rc = P.zi == 2 ? run_batches<2>(pl, pl->lists[kind], P, O, st) : run_batches<0>(pl, pl->lists[kind], P, O, st);
    if (rc) return rc;
    *done = true;
    return GPRB_OK;
}

// K_fe / K_ef + dK/dl of force pack f (full window, one destination, outputs zeroed by the caller; any of the four may be
// NULL) against energy pack e.  *done = false: the pairwise kernel is to run.
int gprb_kef_factored(const gprb_pack *e, gprb_pack *f, double p0, double p1, double zeta, double *Kef, long long ld_ef,
                      double *Kfe, long long ld_fe, double *dKef, long long ld_def, double *dKfe, long long ld_dfe,
                      cudaStream_t st, bool *done) {
    *done = false;
    bool off, force;
    factored_switch(&off, &force);
    if (off || f->ks != GPRB_MAX_KS || e->ks != GPRB_MAX_KS || f->n_rows == 0 || e->n_rows == 0) return GPRB_OK;
    if (!force && 32.0 * (double)((f->n_rows + 7) / 8) * (double)((e->n_rows + 7) / 8) < MIN_PAIRWISE_DMMA) return GPRB_OK;
    gprb_atom_plan *pl = nullptr;
    int rc = pack_plan(f, st, &pl);
    if (rc || !pl) return rc;
    if (!force) {
        double pw = 0.0, fa = 0.0;
        plan_costs_kef(pl->n_clusters, pl->cgrp.data(), pl->cslots.data(), f->n_rows, e->n_rows, e->n_groups, &pw, &fa);
        if (pw < MIN_GAIN * fa) return GPRB_OK;
    }
    CovParams P = {};
    if ((rc = fill_kernel_params(P, GPRB_KERNEL_RBF, p0, p1, zeta))) return rc;
    const KefE E = {e->P, e->elep, e->d_row_ptr, e->n_groups};
    ContractOut O = {};
    O.K = Kfe; O.ldk = ld_fe; O.dK = dKfe; O.lddk = ld_dfe;
    O.K2 = Kef; O.ldk2 = ld_ef; O.dK2 = dKef; O.lddk2 = ld_def;
    O.ne = e->n_groups; O.group_rowsE = e->d_group_rows;
    rc = P.zi == 2 ? run_kef<2>(pl, E, P, O, st) : run_kef<0>(pl, E, P, O, st);
    if (rc) return rc;
    *done = true;
    return GPRB_OK;
}
