// cov_common.cuh — what the covariance kernels of cov_mma.cu and cov_factored.cu share: the kernel constants (CovParams),
// the FP64 m8n8k4 MMA, the table exp and the per-pair weights, so that both paths evaluate the same formulas and quirks.
// Everything is in an anonymous namespace: each translation unit has its own exp table and uploads it itself.
#pragma once
#include "common.cuh"
#include <cmath>

namespace {

struct CovParams {
    const double *PA; const int *eleA; const int *row_groupA;
    const int4 *sched; const int4 *sched_ent;
    const double *PB; const int *recB; const int *row_ptrB; const int *group_rowsB;
    int n_groupsB, n_splits, ks;
    int win_r0, win_r1;                                   // row window on side A (flat rows)
    // k1 = sigma^2/(2 l^2), kz = k1*zeta, c = 1/(2 l^2), h0 = 1/l^3 - 2/l ; Dot: c_dot = sigma^2 zeta
    double k1, kz, c, c_il3, h0, zeta, tol, c_dot;
    double s2, s02;                                          // EE blocks: sigma^2 and (Dot) sigma0^2
    const int *group_rowsA;                                  // EE blocks: rows per group of side A (1 / (n_I n_J))
    int zi, use_tol, mode, grp_begin;
    double *K; long long ldk; double *dK; long long lddk;     // kff: K / dK/dl ; kfe: Kfe / dKfe
    double *K2; long long ldk2; double *dK2; long long lddk2; // kfe only: Kef / dKef (transposed copies)
    // fused all-gather (gprb_kff_multi / gprb_kfe_multi): every finished value of K is also stored into the
    // same slab of n_extra peer matrices (NVLink peer stores, pointers from gprb_peer_open); dK stays local
    double *Kx[GPRB_MAX_DST - 1]; int n_extra;
    int two_stage;                                            // two-stage contraction (no-gradient K_ff, 8 k-steps)
};

__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// exp(x) for x <= 0 (the RBF exponent -(1-D)/(2 l^2)): 2^(k/32) table + degree-5 polynomial on
// |r| <= ln2/64 (truncation 2e-15 relative), evaluated in Estrin form.  (Round 2 measured a variant with a 1024-entry
// table, degree 3, one-step reduction and an integer clamp -- 5 instead of 8 dependent FP64 steps: same kernel time,
// 1 812 vs 1 811 ms at S5, so the dependent chain is not what bounds the epilogue; profiles/experiments/README.md.)
constexpr int EXP_TAB = 32;
__device__ double d_exp2_tab[EXP_TAB];    // 2^(j / 32)

__device__ __forceinline__ double exp_neg(double x, const double *tab) {
    x = fmax(x, -700.0);                                     // exp(-700) ~ 1e-304: below anything that matters, no branch
    const double MAGIC = 6755399441055744.0;                 // 1.5 * 2^52: low word = round-to-nearest integer
    const double t = fma(x, 46.16624130844682903, MAGIC);    // 32 / ln 2
    const int ki = __double2loint(t);
    const double kf = t - MAGIC;
    double r = fma(kf, -0x1.62e42fe000000p-6, x);            // ln2/32, high 29 bits (kf * hi is exact)
    r = fma(kf, -0x1.f473de6af278fp-35, r);                   // ln2/32 - high part
    const double r2 = r * r;
    const double a = fma(r, 1.66666666666666657e-01, 0.5);
    const double b = fma(r, 8.33333333333333322e-03, 4.16666666666666644e-02);
    const double c1 = 1.0 + r;
    const double d = fma(r2, a, c1);
    const double r4 = r2 * r2;
    const double p = fma(r4, b, d);                           // 1 + r + r^2/2 + r^3/6 + r^4/24 + r^5/120
    const double v = tab[ki & 31] * p;
    return __hiloint2double(__double2hiint(v) + ((ki >> 5) << 20), __double2loint(v));
}

// s^(zeta-2): ZI = 2 is compile-time (the reference's default zeta, gaussianprocess.py:1027);
// ZI = 0 picks the small integer cases at run time and falls back to pow()
template <int ZI>
__device__ __forceinline__ double pow_zm2(double s, double zeta, int zi) {
    if (ZI == 2) return 1.0;
    if (zi == 2) return 1.0;
    if (zi == 3) return s;
    if (zi == 4) return s * s;
    if (zi == 1) return 1.0 / s;
    return pow(s, zeta - 2.0);
}

// Per-pair scalar weights.  out = w1*G + w2*p q^T ; grad: dout = u1*G + u2*p q^T
// (for NB == 1: out_c = w1 * p_c, dout_c = u1 * p_c).  `valid` may be cleared by the pair cut.
template <int KERNEL, bool GRAD, bool FF, int ZI, bool EE = false>
__device__ __forceinline__ void pair_weights(const CovParams &P, const double *tab, double s, bool &valid,
                                             double &w1, double &w2, double &u1, double &u2) {
    const double sm2 = pow_zm2<ZI>(s, P.zeta, P.zi);
    const double sm1 = s * sm2;
    if (EE) {
        // energy-energy pair: w1 = k(a, b), u1 = dk/dl = k (1 - D) / l^3   (rbf_kernel.cpp:40-47, 86-94; dot_kernel.cpp:38-44)
        const double D = s * sm1;
        if (KERNEL == GPRB_KERNEL_RBF) {
            w1 = P.s2 * exp_neg(fma(D, P.c, -P.c), tab);
            if (GRAD) u1 = w1 * fma(-P.c_il3, D, P.c_il3);
        } else {
            w1 = P.s2 * (D + P.s02);
        }
        return;
    }
    if (KERNEL == GPRB_KERNEL_RBF) {
        // every weight is E times a factor that does not depend on E: the factors are computed next to the exp
        // chain (instruction-level parallelism), one multiply each once E is known
        const double D = s * sm1;
        const double f1 = P.kz * sm1;                                  // w1 = g beta          = E f1
        const double q2 = f1 * (P.zeta * sm1);                         // g zeta^2 s^(2zeta-2) = E q2
        const double f2 = (ZI == 2) ? fma(q2, P.c, P.kz) : fma(q2, P.c, P.kz * (P.zeta - 1.0) * sm2);   // w2 = g gamma = E f2
        const double h = fma(-P.c_il3, D, P.h0);                       // (1-D)/l^3 - 2/l   (:622-630, :245-247)
        const double g1 = f1 * h, g2 = fma(f2, h, -(q2 * P.c_il3));
        const double E = exp_neg(fma(D, P.c, -P.c), tab);             // exp(-(1-D)/(2l^2))  rbf_kernel.cpp:393
        if (FF && !GRAD && P.use_tol) valid = valid && (E * P.k1 > P.tol);   // dK_dD > tol (:394-395), non-grad only
        w1 = E * f1;
        if (FF) w2 = E * f2;
        if (GRAD) {
            u1 = E * g1;
            if (FF) u2 = E * g2;
        }
    } else {   // Dot: sigma^2 zeta (s^(z-1) G + (z-1) s^(z-2) p q^T)   (dot_kernel.cpp:285-289, dot_kernel.py:256)
        w1 = P.c_dot * sm1;
        if (FF) w2 = P.c_dot * (P.zeta - 1.0) * sm2;
    }
}

int integer_zeta(double zeta) {
    int zi = (int)zeta;
    return ((double)zi == zeta && zi >= 1 && zi <= 4) ? zi : -1;
}

// per-device one-time state (a process may drive several GPUs): __constant__ tables and function attributes exist per device
constexpr int MAX_DEV = 64;
int current_device(int *dev) {
    GPRB_CUDA(cudaGetDevice(dev));
    GPRB_REQUIRE(*dev >= 0 && *dev < MAX_DEV, "device index %d out of range", *dev);
    return GPRB_OK;
}

int upload_tables() {
    static bool done[MAX_DEV] = {};
    int dev = 0;
    { int rc = current_device(&dev); if (rc) return rc; }
    if (done[dev]) return GPRB_OK;
    static double tab[EXP_TAB];
    for (int j = 0; j < EXP_TAB; j++) tab[j] = std::exp2((double)j / (double)EXP_TAB);
    GPRB_CUDA(cudaMemcpyToSymbol(d_exp2_tab, tab, sizeof tab));
    done[dev] = true;
    return GPRB_OK;
}

int fill_kernel_params(CovParams &P, int kernel, double p0, double p1, double zeta) {
    P.zeta = zeta;
    P.zi = integer_zeta(zeta);
    if (kernel == GPRB_KERNEL_RBF) {
        GPRB_REQUIRE(p1 > 0.0, "length scale l must be positive, got %g", p1);
        P.c = 1.0 / (2.0 * p1 * p1);
        P.k1 = p0 * p0 * P.c;
        P.kz = P.k1 * zeta;
        P.c_il3 = 1.0 / (p1 * p1 * p1);
        P.h0 = P.c_il3 - 2.0 / p1;
    } else {
        P.c = P.k1 = P.kz = P.c_il3 = P.h0 = 0.0;
    }
    P.c_dot = p0 * p0 * zeta;
    P.s2 = p0 * p0;
    P.s02 = kernel == GPRB_KERNEL_DOT ? p1 * p1 : 0.0;
    return upload_tables();
}

}  // namespace
