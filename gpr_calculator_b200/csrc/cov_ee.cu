// cov_ee.cu — the eps-regularised energy diagonal (prior variance of energy rows).
//
// Replaces the numpy K_ee_RBF / K_ee that the reference uses only in diag() (kernels/base.py:107-130,
// Dot_mb.py:177-202).  The energy-energy covariance K_ee itself is gprb_kee on the DMMA tile path (cov_mma.cu).
//
// A plain DFMA kernel, 2*d flops per pair: one CTA per group, threads over the pairs of its rows; fixed-order reductions.
#include "common.cuh"

namespace {

struct EEParams {
    const double *PA; const int *eleA; const int *row_ptrA; const int *rowsA;
    int ks;
    double c_sigma2, c_i2l2, c_sigma02, zeta;
    int zi, kernel;
    double *K;
};

__device__ __forceinline__ double pow_z(double s, double zeta, int zi) {
    if (zi == 2) return s * s;
    if (zi == 3) return s * s * s;
    if (zi == 1) return s;
    if (zi == 4) { double t = s * s; return t * t; }
    return pow(s, zeta);
}

// element k of flat row `prow` of an energy pack (ncomp = 1)
__device__ __forceinline__ const double *row_base(const double *P, int ks, int prow) {
    return P + (size_t)(prow >> 3) * ks * 32 + (prow & 7) * 4;
}

// diag(): energy rows, k(I,I) with norms (|x|+eps) and d = x1.x2 / (eps + n1 n2); no zero-norm drop.
__global__ void __launch_bounds__(128) kee_diag_kernel(const EEParams P, const double *normA, double eps) {
    const int I = blockIdx.x;
    const int row0 = P.row_ptrA[I], n = P.rowsA[I];
    double acc = 0.0;
    for (int pidx = threadIdx.x; pidx < n * n; pidx += blockDim.x) {
        const int a = pidx / n, b = pidx - a * n;
        int ea = P.eleA[row0 + a], eb = P.eleA[row0 + b];
        ea = ea >= 0 ? ea : -(ea + 2);
        eb = eb >= 0 ? eb : -(eb + 2);
        if (ea != eb) continue;
        const double *xa = row_base(P.PA, P.ks, row0 + a), *xb = row_base(P.PA, P.ks, row0 + b);
        double s = 0.0;
        for (int kk = 0; kk < P.ks; kk++)
            for (int q = 0; q < 4; q++) s = fma(xa[kk * 32 + q], xb[kk * 32 + q], s);
        const double na = normA[row0 + a], nb = normA[row0 + b];
        const double dd = s * na * nb / (eps + (na + eps) * (nb + eps));
        const double D = pow_z(dd, P.zeta, P.zi);
        if (P.kernel == GPRB_KERNEL_RBF) acc += P.c_sigma2 * exp((D - 1.0) * P.c_i2l2);
        else acc += P.c_sigma2 * (D + P.c_sigma02);
    }
    __shared__ double red[4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        const double nn = (double)n * (double)n;
        P.K[I] = nn > 0 ? (red[0] + red[1] + red[2] + red[3]) / nn : 0.0;
    }
}

int fill(EEParams &P, int kernel, double p0, double p1, double zeta) {
    P.kernel = kernel;
    P.zeta = zeta;
    int zi = (int)zeta;
    P.zi = ((double)zi == zeta && zi >= 1 && zi <= 4) ? zi : -1;
    P.c_sigma2 = p0 * p0;
    if (kernel == GPRB_KERNEL_RBF) {
        GPRB_REQUIRE(p1 > 0.0, "length scale l must be positive, got %g", p1);
        P.c_i2l2 = 1.0 / (2.0 * p1 * p1);
        P.c_sigma02 = 0.0;
    } else {
        P.c_i2l2 = 0.0;
        P.c_sigma02 = p1 * p1;
    }
    return GPRB_OK;
}

}  // namespace

extern "C" int gprb_kee_diag(int kernel, const gprb_pack *e, double p0, double p1, double zeta, double *out, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(e && out, "gprb_kee_diag: NULL argument");
    { int rcd = gprb_check_device(e, "gprb_kee_diag"); if (rcd) return rcd; }
    GPRB_REQUIRE(e->ncols == 0, "gprb_kee_diag: need an energy pack");
    if (e->n_groups == 0) return GPRB_OK;
    EEParams P = {};
    int rc = fill(P, kernel, p0, p1, zeta);
    if (rc) return rc;
    P.PA = e->P; P.eleA = e->elep; P.row_ptrA = e->d_row_ptr; P.rowsA = e->d_group_rows; P.ks = e->ks;
    P.K = out;
    kee_diag_kernel<<<e->n_groups, 128, 0, st>>>(P, e->norm, GPRB_EPS_NORM);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}
