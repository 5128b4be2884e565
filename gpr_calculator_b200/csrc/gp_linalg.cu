// gp_linalg.cu — the O(N^2) / O(N^3) GP algebra that follows the covariance build, kept on device.
//
// Replaces the scipy/numpy steps of GP.log_marginal_likelihood, GP.fit, GP.set_K_inv and
// GP.predict* (gaussianprocess.py:128-202, 286-317, 338-377, 880-908).  The factorisation and
// triangular solves are cuSOLVER / cuBLAS (potrf / potrs / trsm) and the K* K^-1 product is cuBLAS trmm:
// library calls, reported separately by bench.py and not optimised (north_star).  The
// bandwidth-bound pieces (noise, log-det, trace of (alpha alpha^T - K^-1) dK, fused mean/variance
// row reductions) are hand-written kernels with fixed-order reductions.
//
// All matrices are row-major; a symmetric row-major matrix is handed to the column-major libraries
// unchanged, "lower" here == CUBLAS_FILL_MODE_UPPER there.
#include "common.cuh"
#include <cstdint>
#include <algorithm>
#include <cusolverDn.h>
#include <cublas_v2.h>

namespace {

// library handles are per device (a process may drive several GPUs, e.g. after torch.cuda.set_device in a notebook)
constexpr int MAX_DEV = 64;
cusolverDnHandle_t g_solver_dev[MAX_DEV] = {};
cublasHandle_t g_blas_dev[MAX_DEV] = {};
cusolverDnParams_t g_params_dev[MAX_DEV] = {};
thread_local cusolverDnHandle_t g_solver = nullptr;     // handles of the current device, set by handles()
thread_local cublasHandle_t g_blas = nullptr;
thread_local cusolverDnParams_t g_params = nullptr;

int handles(cudaStream_t st) {
    { int rc0 = gprb_pool_init(); if (rc0) return rc0; }
    int dev = 0;
    GPRB_CUDA(cudaGetDevice(&dev));
    GPRB_REQUIRE(dev >= 0 && dev < MAX_DEV, "device index %d out of range", dev);
    if (!g_solver_dev[dev]) {
        if (cusolverDnCreate(&g_solver_dev[dev]) != CUSOLVER_STATUS_SUCCESS) { gprb_set_error("cusolverDnCreate failed"); return GPRB_ERR_CUDA; }
    }
    if (!g_blas_dev[dev]) {
        if (cublasCreate(&g_blas_dev[dev]) != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasCreate failed"); return GPRB_ERR_CUDA; }
    }
    if (!g_params_dev[dev]) {
        if (cusolverDnCreateParams(&g_params_dev[dev]) != CUSOLVER_STATUS_SUCCESS) { gprb_set_error("cusolverDnCreateParams failed"); return GPRB_ERR_CUDA; }
    }
    g_solver = g_solver_dev[dev]; g_blas = g_blas_dev[dev]; g_params = g_params_dev[dev];
    if (cusolverDnSetStream(g_solver, st) != CUSOLVER_STATUS_SUCCESS || cublasSetStream(g_blas, st) != CUBLAS_STATUS_SUCCESS) {
        gprb_set_error("setting the library stream failed");
        return GPRB_ERR_CUDA;
    }
    return GPRB_OK;
}

// Stream-ordered temporaries that are returned to the pool on every exit path of an entry point.
struct Scratch {
    cudaStream_t st;
    std::vector<void *> ptrs;
    explicit Scratch(cudaStream_t s) : st(s) {}
    Scratch(const Scratch &) = delete;
    void *get(size_t bytes) {
        void *p = nullptr;
        cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 8, st);
        if (e != cudaSuccess) { gprb_set_error("cudaMallocAsync of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); return nullptr; }
        ptrs.push_back(p);
        return p;
    }
    ~Scratch() { for (void *p : ptrs) gprb_pool_free(p, st); }
};

// The Cholesky factor L lives in the row-major lower triangle == CUBLAS_FILL_MODE_UPPER of the column-major view the
// libraries see (K = U^T U, U = L^T); every consumer below (potrs, trsm) reads that triangle.  gprb_chol_factor
// itself runs cuSOLVER's potrf in the OTHER fill mode, which is 20 % faster on B200 (357 vs 446 ms at N = 32 980,
// profiles/r02_potrf_modes.txt), and mirrors the factor into the lower triangle afterwards (3 ms), so the trsm-heavy
// consumers keep the mode in which cuBLAS trsm is faster (inverse rows: 990 vs 1 043 ms).
constexpr cublasFillMode_t FACTOR_UPLO = CUBLAS_FILL_MODE_UPPER;
// the two triangular solves of (U^T U) X = B, first and second
constexpr cublasOperation_t solve_op(int step) { return step == 0 ? CUBLAS_OP_T : CUBLAS_OP_N; }

__global__ void add_noise_kernel(double *K, long long ld, int N, int NE, double ne2, double nf2) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) K[(long long)i * ld + i] += (i < NE) ? ne2 : nf2;
}

// A[i][j] = A[j][i] for i > j (fill the lower triangle from the upper one)
__global__ void mirror_upper_kernel(double *A, long long ld, int N) {
    __shared__ double t[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;       // source block (bi, bj) with bj >= bi
    if (bj < bi) return;
    const int i = bi * 32 + threadIdx.y, j = bj * 32 + threadIdx.x;
    if (i < N && j < N) t[threadIdx.y][threadIdx.x] = A[(long long)i * ld + j];
    __syncthreads();
    const int ti = bj * 32 + threadIdx.y, tj = bi * 32 + threadIdx.x;   // destination (transposed block)
    if (ti < N && tj < N && ti > tj) A[(long long)ti * ld + tj] = t[threadIdx.x][threadIdx.y];
}

__device__ __forceinline__ double block_sum(double v, double *sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x == 0) for (int i = 0; i < nw; i++) r += sh[i];
    return r;   // valid in thread 0
}

__global__ void lml_terms_kernel(const double *L, long long ld, int N, const double *y, const double *alpha, double *out) {
    __shared__ double sh[32];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        a += log(L[(long long)i * ld + i]);
        b += y[i] * alpha[i];
    }
    a = block_sum(a, sh);
    b = block_sum(b, sh);
    if (threadIdx.x == 0) { out[0] = a; out[1] = b; }
}

// partial[3 b + 0] = sum over the block's rows of sum_j (alpha_i alpha_j - Kinv_ij) * dK_ij
// partial[3 b + 1] = sum over rows of (alpha_i^2 - Kinv_ii) * w_i          (w = we / wf for energy / force rows)
// partial[3 b + 2] = the same with the second weight pair (we2 / wf2)
// dK holds the rows of the row-sharded build: energy rows (i < NE) K_ee only, force rows K_fe and the J >= I blocks of
// K_ff, so tr = EE (j in [i, NE), doubled off the diagonal) + 2 FE + FF (j >= i, doubled).  Kinv has to be valid for
// j >= i only: the columns j < NE of a force row come from the energy rows of the inverse, Kinv[i, j] = KinvE[j * ldE + i].
__global__ void __launch_bounds__(256) trace_kernel(int N, int r0, int r1, const double *__restrict__ alpha,
                                                    const double *__restrict__ Kinv, long long ldi,
                                                    const double *__restrict__ dK, long long lddk,
                                                    int NE, double we, double wf, double we2, double wf2, double *partial,
                                                    const double *__restrict__ KinvE, long long ldE) {
    __shared__ double sh[32];
    double acc = 0.0, acc2 = 0.0, acc3 = 0.0;
    for (int i = r0 + blockIdx.x; i < r1; i += gridDim.x) {
        const double ai = alpha[i];
        const double *ki = Kinv + (long long)i * ldi;
        if (dK) {
            const double *di = dK + (long long)(i - r0) * lddk;
            const int jend = i < NE ? NE : N;
            for (int j = i + threadIdx.x; j < jend; j += blockDim.x) {
                const double t = fma(ai, alpha[j], -ki[j]) * di[j];
                acc += (j == i) ? t : 2.0 * t;
            }
            if (i >= NE)
                for (int j = threadIdx.x; j < NE; j += blockDim.x) acc += 2.0 * fma(ai, alpha[j], -KinvE[(long long)j * ldE + i]) * di[j];
        }
        if (threadIdx.x == 0) {
            const double wii = ai * ai - ki[i];
            acc2 += wii * (i < NE ? we : wf);
            acc3 += wii * (i < NE ? we2 : wf2);
        }
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) { partial[3 * blockIdx.x] = acc; partial[3 * blockIdx.x + 1] = acc2; partial[3 * blockIdx.x + 2] = acc3; }
}

__global__ void block_sum_kernel(int N, int r0, int r1, int c0, int c1, const double *__restrict__ alpha,
                                 const double *__restrict__ Kinv, long long ldi, double *partial) {
    __shared__ double sh[32];
    double acc = 0.0;
    for (int i = r0 + blockIdx.x; i < r1; i += gridDim.x) {
        const double ai = alpha[i];
        const double *ki = Kinv + (long long)i * ldi;
        for (int j = c0 + threadIdx.x; j < c1; j += blockDim.x) acc += fma(ai, alpha[j], -ki[j]);
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) { partial[3 * blockIdx.x] = acc; partial[3 * blockIdx.x + 1] = 0.0; partial[3 * blockIdx.x + 2] = 0.0; }
}

// out[k] += 0.5 * sum_b partial[3 b + k]: one warp, lane-strided partial sums combined in a fixed order (deterministic)
__global__ void final_sum_kernel(const double *partial, int n, double *out) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = threadIdx.x; i < n; i += 32) { a += partial[3 * i]; b += partial[3 * i + 1]; c += partial[3 * i + 2]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if (threadIdx.x == 0) { out[0] += 0.5 * a; out[1] += 0.5 * b; out[2] += 0.5 * c; }
}

// one CTA per test row: mean = Ks[i,:].alpha
__global__ void __launch_bounds__(256) predict_rows_kernel(int N, const double *__restrict__ Ks, long long ldks,
                                                           const double *__restrict__ alpha, double *mean) {
    __shared__ double sh[32];
    const int i = blockIdx.x;
    const double *k = Ks + (long long)i * ldks;
    double m = 0.0;
    for (int j = threadIdx.x; j < N; j += blockDim.x) m = fma(k[j], alpha[j], m);
    m = block_sum(m, sh);
    if (threadIdx.x == 0) mean[i] = m;
}

__global__ void unit_columns_kernel(double *B, long long ldb, int n_rows, int col0) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_rows) B[(long long)k * ldb + col0 + k] = 1.0;
}

// ---- enqueue-only building blocks (no host synchronisation) of gprb_chol_factor, gprb_chol_inverse_rows and gprb_lml_eval ----

// potrf in cuSOLVER's faster fill mode + mirror of the factor into the row-major lower triangle; *info_dev = potrf status
int factor_enqueue(double *K, long long ldk, int N, int *info_dev, Scratch &scratch, cudaStream_t st) {
    size_t wdev = 0, whost = 0;
    if (cusolverDnXpotrf_bufferSize(g_solver, g_params, CUBLAS_FILL_MODE_LOWER, (int64_t)N, CUDA_R_64F, K, (int64_t)ldk,
                                    CUDA_R_64F, &wdev, &whost) != CUSOLVER_STATUS_SUCCESS) {
        gprb_set_error("Xpotrf_bufferSize failed"); return GPRB_ERR_CUDA;
    }
    void *dwork = scratch.get(wdev);
    if (!dwork) return GPRB_ERR_CUDA;
    std::vector<unsigned char> hwork(whost);
    cusolverStatus_t cs = cusolverDnXpotrf(g_solver, g_params, CUBLAS_FILL_MODE_LOWER, (int64_t)N, CUDA_R_64F, K, (int64_t)ldk,
                                           CUDA_R_64F, dwork, wdev, whost ? hwork.data() : nullptr, whost, info_dev);
    if (cs != CUSOLVER_STATUS_SUCCESS) { gprb_set_error("cusolver potrf status %d", (int)cs); return GPRB_ERR_CUDA; }
    dim3 grid((N + 31) / 32, (N + 31) / 32), block(32, 32);
    mirror_upper_kernel<<<grid, block, 0, st>>>(K, ldk, N);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

int solve_vec_enqueue(const double *L, long long ldl, int N, double *b, int *info_dev) {
    cusolverStatus_t cs = cusolverDnDpotrs(g_solver, FACTOR_UPLO, N, 1, L, (int)ldl, b, N, info_dev);
    if (cs != CUSOLVER_STATUS_SUCCESS) { gprb_set_error("cusolverDnDpotrs status %d", (int)cs); return GPRB_ERR_CUDA; }
    return GPRB_OK;
}

// K^-1[T, T] = (L_TT L_TT^T)^-1 for the trailing index set T = [c0, N) (L^-1 is triangular), so rows [r0, r1) of the
// inverse, restricted to the columns >= c0, are the solution of the trailing system with the unit vectors of those
// rows as right-hand sides (symmetric: row = column).
int inverse_rows_enqueue(const double *L, long long ldl, int N, int r0, int r1, int c0, double *out, long long ldo, cudaStream_t st) {
    const int n = N - c0, nrhs = r1 - r0;
    GPRB_CUDA(cudaMemset2DAsync(out, ldo * sizeof(double), 0, (size_t)n * sizeof(double), nrhs, st));
    unit_columns_kernel<<<(nrhs + 255) / 256, 256, 0, st>>>(out, ldo, nrhs, r0 - c0);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    // what potrs does, through the 64-bit cuBLAS interface (N^2 may exceed 2^31, e.g. the S4 configuration):
    // column-major view, K_T = U^T U with U in the upper triangle of the factor's buffer;  U^T Y = E, then U X = Y
    const double one = 1.0;
    const double *U = L + (long long)c0 * ldl + c0;
    cublasStatus_t b1 = cublasDtrsm_64(g_blas, CUBLAS_SIDE_LEFT, FACTOR_UPLO, solve_op(0), CUBLAS_DIAG_NON_UNIT,
                                       (int64_t)n, (int64_t)nrhs, &one, U, (int64_t)ldl, out, (int64_t)ldo);
    cublasStatus_t b2 = cublasDtrsm_64(g_blas, CUBLAS_SIDE_LEFT, FACTOR_UPLO, solve_op(1), CUBLAS_DIAG_NON_UNIT,
                                       (int64_t)n, (int64_t)nrhs, &one, U, (int64_t)ldl, out, (int64_t)ldo);
    if (b1 != CUBLAS_STATUS_SUCCESS || b2 != CUBLAS_STATUS_SUCCESS) {
        gprb_set_error("cublasDtrsm_64 (inverse rows) status %d / %d", (int)b1, (int)b2); return GPRB_ERR_CUDA;
    }
    return GPRB_OK;
}

int trace_blocks(int rows) { return rows < 1184 ? rows : 1184; }     // 8 x 148

// dev_out[0..2] += {1/2 tr-term, 1/2 sum W_ii w_i, 1/2 sum W_ii w2_i} of the rows [r0, r1)
int trace_enqueue(int N, int r0, int r1, const double *alpha, const double *Kinv_virt, long long ldi, const double *dK_rows,
                  long long lddk, int NE, double we, double wf, double we2, double wf2,
                  const double *KinvE, long long ldE, double *dev_out, Scratch &scratch, cudaStream_t st) {
    const int blocks = trace_blocks(r1 - r0);
    double *d = (double *)scratch.get((size_t)3 * blocks * sizeof(double));
    if (!d) return GPRB_ERR_CUDA;
    trace_kernel<<<blocks, 256, 0, st>>>(N, r0, r1, alpha, Kinv_virt, ldi, dK_rows, lddk, NE, we, wf, we2, wf2, d, KinvE, ldE);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    final_sum_kernel<<<1, 32, 0, st>>>(d, blocks, dev_out);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

int block_sum_enqueue(int N, int r0, int r1, int c0, int c1, const double *alpha, const double *Kinv, long long ldi,
                      double *dev_out, Scratch &scratch, cudaStream_t st) {
    const int blocks = trace_blocks(r1 - r0);
    double *d = (double *)scratch.get((size_t)3 * blocks * sizeof(double));
    if (!d) return GPRB_ERR_CUDA;
    block_sum_kernel<<<blocks, 256, 0, st>>>(N, r0, r1, c0, c1, alpha, Kinv, ldi, d);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    final_sum_kernel<<<1, 32, 0, st>>>(d, blocks, dev_out);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

// the kernels index Kinv[i * ld + j] with global (i, j): shift the base so that (r0, c0) is element 0 of a slab
const double *virtual_base(const double *rows, long long ldr, int r0, int c0) {
    return reinterpret_cast<const double *>(reinterpret_cast<uintptr_t>(rows) -
                                            (uintptr_t)(((long long)r0 * ldr + c0) * (long long)sizeof(double)));
}

}  // namespace

extern "C" int gprb_add_noise(double *K, long long ldk, int N, int NE, double noise_e, double noise_f, void *stream) {
    GPRB_REQUIRE(K && N >= 0, "gprb_add_noise: bad argument");
    if (N == 0) return GPRB_OK;
    add_noise_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(K, ldk, N, NE, noise_e * noise_e, noise_f * noise_f);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

extern "C" int gprb_chol_factor(double *K, long long ldk, int N, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(K && N > 0, "gprb_chol_factor: bad argument");
    int rc = handles(st);
    if (rc) return rc;
    Scratch scratch(st);
    int *info = (int *)scratch.get(sizeof(int));
    if (!info) return GPRB_ERR_CUDA;
    if ((rc = factor_enqueue(K, ldk, N, info, scratch, st))) return rc;
    int hinfo = -1;
    GPRB_CUDA(cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    if (hinfo != 0) { gprb_set_error("matrix not positive definite (potrf info = %d)", hinfo); return GPRB_ERR_LINALG; }
    return GPRB_OK;
}

extern "C" int gprb_chol_inverse_rows(const double *L, long long ldl, int N, int r0, int r1, int c0,
                                      double *out, long long ldo, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(L && out && N > 0 && 0 <= c0 && c0 <= r0 && r0 <= r1 && r1 <= N && ldo >= N - c0,
                 "gprb_chol_inverse_rows: bad argument");
    if (r0 == r1) return GPRB_OK;
    int rc = handles(st);
    if (rc) return rc;
    return inverse_rows_enqueue(L, ldl, N, r0, r1, c0, out, ldo, st);
}

// One likelihood evaluation after the covariance build, enqueued back to back with ONE host synchronisation at the end
// (GP.log_marginal_likelihood, gaussianprocess.py:160-198): K += noise, Cholesky in place, alpha = K^-1 y, log-det and
// y.alpha, and -- want_grad -- the traces of W = alpha alpha^T - K^-1 against the rows of dK/dl this rank holds, with
// K^-1 taken block of rows by block of rows from trailing-block triangular solves (no explicit inverse).
//   ranges_host: n_ranges (r0, r1) row ranges of the assembled matrix whose rows of dK are stacked in dK_rows (NULL: no
//   dK term, e.g. the Dot kernel); rows < NE hold the K_ee part, force rows K_fe and the J >= I blocks of K_ff.
//   out_host[8]: 0 log-det term sum(log L_ii), 1 y.alpha, 2 1/2 tr(W dK) over the held rows, 3 1/2 sum W_ii noise_i^2,
//   4 1/2 sum W_ii 2 noise_i, 5 1/2 sum of W over the held energy rows x all energy columns (want_s0, Dot sigma0 term).
extern "C" int gprb_lml_eval(double *K, long long ldk, int N, int NE, const double *y, double noise_e, double noise_f,
                             const double *dK_rows, long long lddk, int n_ranges, const int *ranges_host,
                             int want_grad, int want_s0, int parts, int prefactored, double *alpha, double *work,
                             long long work_doubles, double *out_host, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(K && y && alpha && out_host && N > 0 && NE >= 0 && NE <= N && ldk >= N, "gprb_lml_eval: bad argument");
    GPRB_REQUIRE(n_ranges >= 0 && (n_ranges == 0 || ranges_host), "gprb_lml_eval: bad row ranges");
    int rc = handles(st);
    if (rc) return rc;
    for (int k = 0; k < 8; k++) out_host[k] = 0.0;
    Scratch scratch(st);
    int *info = (int *)scratch.get(2 * sizeof(int));
    double *acc = (double *)scratch.get(9 * sizeof(double));      // [0..1] lml terms, [2..4] traces, [5..7] sigma0 block sum
    if (!info || !acc) return GPRB_ERR_CUDA;
    GPRB_CUDA(cudaMemsetAsync(acc, 0, 9 * sizeof(double), st));
    GPRB_CUDA(cudaMemsetAsync(info, 0, 2 * sizeof(int), st));
    // device time of the two phases (factor + alpha, gradient solves + traces): out_host[6], out_host[7] in ms
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    struct EvGuard { cudaEvent_t *e; ~EvGuard() { for (int k = 0; k < 3; k++) if (e[k]) cudaEventDestroy(e[k]); } } ev_guard{ev};
    for (int k = 0; k < 3; k++) GPRB_CUDA(cudaEventCreate(&ev[k]));
    GPRB_CUDA(cudaEventRecord(ev[0], st));
    if (!prefactored) {      // prefactored: K already holds the factor of K + noise in its row-major lower triangle (multi-GPU Cholesky)
        add_noise_kernel<<<(N + 255) / 256, 256, 0, st>>>(K, ldk, N, NE, noise_e * noise_e, noise_f * noise_f);
        GPRB_LAUNCHED();
        if ((rc = factor_enqueue(K, ldk, N, info, scratch, st))) return rc;
    }
    GPRB_CUDA(cudaMemcpyAsync(alpha, y, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if ((rc = solve_vec_enqueue(K, ldk, N, alpha, info + 1))) return rc;
    lml_terms_kernel<<<1, 1024, 0, st>>>(K, ldk, N, y, alpha, acc);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    GPRB_CUDA(cudaEventRecord(ev[1], st));
    if (want_grad) {
        if (parts < 1) parts = 16;
        const double we = noise_e * noise_e, wf = noise_f * noise_f, we2 = 2.0 * noise_e, wf2 = 2.0 * noise_f;
        const int blk = std::max(512, (N + parts - 1) / parts);
        // the K^-1 slabs live in the caller's workspace ([NE + blk, N] doubles, gprb_lml_eval_work): large buffers that come and go
        // fragment the stream-ordered pool the packs are allocated from (measured: occasional 1-2 s stalls of the next pack creation)
        GPRB_REQUIRE(work && work_doubles >= (long long)(NE + std::min(blk, N)) * N, "gprb_lml_eval: workspace of %lld doubles needed",
                     (long long)(NE + std::min(blk, N)) * N);
        double *Einv = nullptr;
        double *slab_buf = work + (size_t)NE * N;
        if (NE) {
            Einv = work;
            if ((rc = inverse_rows_enqueue(K, ldk, N, 0, NE, 0, Einv, N, st))) return rc;
        }
        long long off = 0;                                   // first row of the range inside dK_rows
        for (int q = 0; q < n_ranges; q++) {
            const int R0 = ranges_host[2 * q], R1 = ranges_host[2 * q + 1];
            GPRB_REQUIRE(0 <= R0 && R0 <= R1 && R1 <= N, "gprb_lml_eval: bad row range [%d, %d)", R0, R1);
            int a = R0;
            while (a < R1) {
                int b;
                const double *rows; long long ldr; int c0;
                if (a < NE) {                                 // energy rows: a slice of K^-1[0:NE, :]
                    b = std::min(R1, NE);
                    rows = Einv + (size_t)a * N; ldr = N; c0 = 0;
                } else {                                      // stream order: the previous block's trace has read the slab
                    b = std::min(R1, a + blk);
                    c0 = a; ldr = N - c0;
                    if ((rc = inverse_rows_enqueue(K, ldk, N, a, b, c0, slab_buf, ldr, st))) return rc;
                    rows = slab_buf;
                }
                const double *dptr = dK_rows ? dK_rows + (off + (a - R0)) * lddk : nullptr;
                rc = trace_enqueue(N, a, b, alpha, virtual_base(rows, ldr, a, c0), ldr, dptr, lddk, NE, we, wf, we2, wf2,
                                   Einv, N, acc + 2, scratch, st);
                if (!rc && want_s0 && b <= NE)
                    rc = block_sum_enqueue(N, a, b, 0, NE, alpha, Einv, N, acc + 5, scratch, st);
                if (rc) return rc;
                a = b;
            }
            off += R1 - R0;
        }
    }
    GPRB_CUDA(cudaEventRecord(ev[2], st));
    double hacc[9];
    int hinfo[2] = {-1, -1};
    GPRB_CUDA(cudaMemcpyAsync(hacc, acc, sizeof hacc, cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaMemcpyAsync(hinfo, info, sizeof hinfo, cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    if (hinfo[0] != 0) { gprb_set_error("matrix not positive definite (potrf info = %d)", hinfo[0]); return GPRB_ERR_LINALG; }
    out_host[0] = hacc[0]; out_host[1] = hacc[1]; out_host[2] = hacc[2]; out_host[3] = hacc[3]; out_host[4] = hacc[4];
    out_host[5] = hacc[5];
    float ms01 = 0.f, ms12 = 0.f;
    cudaEventElapsedTime(&ms01, ev[0], ev[1]);
    cudaEventElapsedTime(&ms12, ev[1], ev[2]);
    out_host[6] = ms01; out_host[7] = ms12;
    return GPRB_OK;
}

extern "C" long long gprb_lml_eval_work(int N, int NE, int want_grad, int parts) {
    if (!want_grad || N <= 0) return 0;
    if (parts < 1) parts = 16;
    const int blk = std::max(512, (N + parts - 1) / parts);
    return (long long)(NE + std::min(blk, N)) * N;
}

// one CTA per test row, half-product variant: W = Ks . triu(Kinv) (trmm), k^T Kinv k = sum_j k_j (2 W_j - Kinv_jj k_j)
__global__ void __launch_bounds__(256) predict_rows_sym_kernel(int N, const double *__restrict__ Ks, long long ldks,
                                                               const double *__restrict__ alpha, const double *__restrict__ W,
                                                               const double *__restrict__ kdiag, const double *__restrict__ diag,
                                                               double *mean, double *var) {
    __shared__ double sh[32];
    const int i = blockIdx.x;
    const double *k = Ks + (long long)i * ldks;
    const double *w = W + (long long)i * N;
    double m = 0.0, v = 0.0;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const double kj = k[j];
        m = fma(kj, alpha[j], m);
        v = fma(kj, fma(2.0, w[j], -kdiag[j] * kj), v);
    }
    m = block_sum(m, sh);
    v = block_sum(v, sh);
    if (threadIdx.x == 0) {
        mean[i] = m;
        const double r = diag[i] - v;
        var[i] = r < 0.0 ? 0.0 : r;                  // gaussianprocess.py:906-907
    }
}

__global__ void extract_diag_kernel(const double *A, long long ld, int N, double *d) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) d[i] = A[(long long)i * ld + i];
}

extern "C" int gprb_predict(int m, int N, const double *Ks, long long ldks, const double *alpha,
                            const double *Kinv, long long ldi, const double *diag,
                            double *mean, double *var, double *work, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(Ks && alpha && mean && m >= 0 && N > 0, "gprb_predict: bad argument");
    if (m == 0) return GPRB_OK;
    if (!var) {
        predict_rows_kernel<<<m, 256, 0, st>>>(N, Ks, ldks, alpha, mean);
        GPRB_LAUNCHED();
        GPRB_CUDA(cudaGetLastError());
        return GPRB_OK;
    }
    GPRB_REQUIRE(Kinv && diag && work, "gprb_predict: variance needs Kinv, diag and work");
    int rc = handles(st);
    if (rc) return rc;
    // K^-1 is symmetric: work = Ks . tri(Kinv) is half the flops of the full product (cuBLAS trmm, m N^2 instead of the
    // 2 m N^2 of a gemm: 104 vs 189 ms for m = 3 104 rows at N = 32 980, profiles/r02_predict_variance_routes.txt), and
    // k^T Kinv k = sum_j k_j (2 work_j - Kinv_jj k_j).  Column-major view: work^T (N x m) = tril_cm(Kinv) . Ks^T
    const double one = 1.0;
    Scratch scratch(st);
    double *kd = (double *)scratch.get((size_t)N * sizeof(double));
    if (!kd) return GPRB_ERR_CUDA;
    extract_diag_kernel<<<(N + 255) / 256, 256, 0, st>>>(Kinv, ldi, N, kd);
    GPRB_LAUNCHED();
    cublasStatus_t bs = cublasDtrmm(g_blas, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, CUBLAS_DIAG_NON_UNIT,
                                    N, m, &one, Kinv, (int)ldi, Ks, (int)ldks, work, N);
    if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDtrmm status %d", (int)bs); return GPRB_ERR_CUDA; }
    predict_rows_sym_kernel<<<m, 256, 0, st>>>(N, Ks, ldks, alpha, work, kd, diag, mean, var);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

// one CTA per test row: mean = Ks[i,:].alpha ; var = max(diag - |Y[i,:]|^2, 0) with Y = (L^-1 Ks^T)^T
__global__ void __launch_bounds__(256) predict_rows_chol_kernel(int N, const double *__restrict__ Ks, long long ldks,
                                                                const double *__restrict__ alpha, const double *__restrict__ Y,
                                                                const double *__restrict__ diag, double *mean, double *var) {
    __shared__ double sh[32];
    const int i = blockIdx.x;
    const double *k = Ks + (long long)i * ldks;
    const double *y = Y + (long long)i * N;
    double m = 0.0, v = 0.0;
    for (int j = threadIdx.x; j < N; j += blockDim.x) { m = fma(k[j], alpha[j], m); const double t = y[j]; v = fma(t, t, v); }
    m = block_sum(m, sh);
    v = block_sum(v, sh);
    if (threadIdx.x == 0) {
        mean[i] = m;
        const double r = diag[i] - v;
        var[i] = r < 0.0 ? 0.0 : r;
    }
}

extern "C" int gprb_predict_chol(int m, int N, const double *Ks, long long ldks, const double *alpha,
                                 const double *L, long long ldl, const double *diag,
                                 double *mean, double *var, double *work, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(Ks && alpha && mean && var && L && diag && work && m >= 0 && N > 0, "gprb_predict_chol: bad argument");
    if (m == 0) return GPRB_OK;
    int rc = handles(st);
    if (rc) return rc;
    // k*^T K^-1 k* = |L^-1 k*|^2: one triangular solve with m right-hand sides (m N^2 flops) instead of the
    // product with the explicit inverse (2 m N^2).  Column-major view: work (N x m) = Ks^T, U^T Y = Ks^T.
    GPRB_CUDA(cudaMemcpy2DAsync(work, (size_t)N * sizeof(double), Ks, (size_t)ldks * sizeof(double), (size_t)N * sizeof(double), m,
                                cudaMemcpyDeviceToDevice, st));
    const double one = 1.0;
    cublasStatus_t bs = cublasDtrsm_64(g_blas, CUBLAS_SIDE_LEFT, FACTOR_UPLO, solve_op(0), CUBLAS_DIAG_NON_UNIT,
                                       (int64_t)N, (int64_t)m, &one, L, (int64_t)ldl, work, (int64_t)N);
    if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDtrsm_64 (predict) status %d", (int)bs); return GPRB_ERR_CUDA; }
    predict_rows_chol_kernel<<<m, 256, 0, st>>>(N, Ks, ldks, alpha, work, diag, mean, var);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

namespace {
// *acc = first failing global row (1-based, potrf convention) over a sequence of panel factorisations
__global__ void accumulate_info_kernel(const int *info, int k0, int *acc) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && *info != 0 && *acc == 0) *acc = *info > 0 ? k0 + *info : *info;
}
}  // namespace

// ---- building blocks of the multi-GPU right-looking Cholesky (GP._distributed_cholesky, dist.py) -------------------
// K is the row-major symmetric matrix (every rank holds a full copy); the factor L (K = L L^T) ends in the row-major lower
// triangle, panel by panel.  gprb_chol_panel (owner of block column k): L_kk = chol(A_kk) (cuSOLVER potrf on the nb x nb block),
// then the rows below, L_ik = A_ik L_kk^-T (one cuBLAS trsm).  info_dev accumulates the first failing row (0 = ok); no host
// synchronisation.  gprb_chol_trailing (owner of block column j > k): A[j0:N, j0:j0+nbj] -= L[j0:N, k0:k0+nbk] L[j0:j0+nbj, k0:k0+nbk]^T.
extern "C" int gprb_chol_panel(double *K, long long ldk, int N, int k0, int nbk, int *info_dev, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(K && info_dev && N > 0 && 0 <= k0 && nbk > 0 && k0 + nbk <= N, "gprb_chol_panel: bad argument");
    int rc = handles(st);
    if (rc) return rc;
    double *Akk = K + (long long)k0 * ldk + k0;
    Scratch scratch(st);
    int lwork = 0;
    if (cusolverDnDpotrf_bufferSize(g_solver, FACTOR_UPLO, nbk, Akk, (int)ldk, &lwork) != CUSOLVER_STATUS_SUCCESS) {
        gprb_set_error("potrf_bufferSize failed"); return GPRB_ERR_CUDA;
    }
    double *work = (double *)scratch.get((size_t)(lwork > 0 ? lwork : 1) * sizeof(double));
    int *info = (int *)scratch.get(sizeof(int));
    if (!work || !info) return GPRB_ERR_CUDA;
    if (cusolverDnDpotrf(g_solver, FACTOR_UPLO, nbk, Akk, (int)ldk, work, lwork, info) != CUSOLVER_STATUS_SUCCESS) {
        gprb_set_error("cusolverDnDpotrf (panel) failed"); return GPRB_ERR_CUDA;
    }
    accumulate_info_kernel<<<1, 32, 0, st>>>(info, k0, info_dev);
    GPRB_LAUNCHED();
    const int m = N - (k0 + nbk);
    if (m > 0) {
        // column-major view: X^T (nbk x m) = (U^T)^-1 A_ik^T with U = L_kk^T in the upper triangle of the block
        const double one = 1.0;
        cublasStatus_t bs = cublasDtrsm_64(g_blas, CUBLAS_SIDE_LEFT, FACTOR_UPLO, CUBLAS_OP_T, CUBLAS_DIAG_NON_UNIT, (int64_t)nbk, (int64_t)m,
                                           &one, Akk, (int64_t)ldk, K + (long long)(k0 + nbk) * ldk + k0, (int64_t)ldk);
        if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDtrsm_64 (panel) status %d", (int)bs); return GPRB_ERR_CUDA; }
    }
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

extern "C" int gprb_chol_trailing(double *K, long long ldk, int N, int k0, int nbk, int j0, int nbj, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(K && N > 0 && 0 <= k0 && nbk > 0 && k0 + nbk <= j0 && nbj > 0 && j0 + nbj <= N, "gprb_chol_trailing: bad argument");
    int rc = handles(st);
    if (rc) return rc;
    // row-major C [m x nbj] -= A [m x nbk] B^T, B = the first nbj rows of A; column-major view: C^T (nbj x m) -= B_cm^T A_cm
    const double minus = -1.0, one = 1.0;
    const long long m = N - j0;
    const double *A = K + (long long)j0 * ldk + k0;
    cublasStatus_t bs = cublasDgemm_64(g_blas, CUBLAS_OP_T, CUBLAS_OP_N, (int64_t)nbj, (int64_t)m, (int64_t)nbk, &minus, A, (int64_t)ldk, A,
                                       (int64_t)ldk, &one, K + (long long)j0 * ldk + j0, (int64_t)ldk);
    if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDgemm_64 (trailing update) status %d", (int)bs); return GPRB_ERR_CUDA; }
    return GPRB_OK;
}

// y_cov = Kxx - K* K^-1 K*^T through the factor, the way gaussianprocess.py:363-366 does it (cho_solve):
// Y = L^-1 K*^T (one trsm with m right-hand sides), cov -= Y^T Y.  cov_dev holds k(X, X) on entry.
extern "C" int gprb_predict_cov(int m, int N, const double *Ks, long long ldks, const double *L, long long ldl,
                                double *cov, long long ldc, double *work, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(Ks && L && cov && work && m >= 0 && N > 0 && ldc >= m, "gprb_predict_cov: bad argument");
    if (m == 0) return GPRB_OK;
    int rc = handles(st);
    if (rc) return rc;
    GPRB_CUDA(cudaMemcpy2DAsync(work, (size_t)N * sizeof(double), Ks, (size_t)ldks * sizeof(double), (size_t)N * sizeof(double), m,
                                cudaMemcpyDeviceToDevice, st));
    const double one = 1.0, minus = -1.0;
    cublasStatus_t bs = cublasDtrsm_64(g_blas, CUBLAS_SIDE_LEFT, FACTOR_UPLO, solve_op(0), CUBLAS_DIAG_NON_UNIT,
                                       (int64_t)N, (int64_t)m, &one, L, (int64_t)ldl, work, (int64_t)N);
    if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDtrsm_64 (predict_cov) status %d", (int)bs); return GPRB_ERR_CUDA; }
    // column-major view: work is Y (N x m); cov (m x m, symmetric) -= Y^T Y
    bs = cublasDgemm(g_blas, CUBLAS_OP_T, CUBLAS_OP_N, m, m, N, &minus, work, N, work, N, &one, cov, (int)ldc);
    if (bs != CUBLAS_STATUS_SUCCESS) { gprb_set_error("cublasDgemm (predict_cov) status %d", (int)bs); return GPRB_ERR_CUDA; }
    return GPRB_OK;
}

namespace {
// omega[i] = sum over the first n_low eigenvectors (rows of V, ascending eigenvalues) of V[k][i]^2
__global__ void leverage_kernel(const double *V, long long ld, int n, int n_low, double *omega) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc = 0.0;
    for (int k = 0; k < n_low; k++) { const double v = V[(long long)k * ld + i]; acc = fma(v, v, acc); }
    omega[i] = acc;
}
}  // namespace

// CUR leverage scores (gaussianprocess.py:1165-1182): eigen-decomposition of the symmetric block A (cuSOLVER syevd, in
// place: on return row k of A is the eigenvector of the k-th smallest eigenvalue), eigenvalues to w_host[n],
// omega_dev[i] = sum_{k: w_k < l_tol} U[i, k]^2; *n_low_host = number of eigenvalues below l_tol.
extern "C" int gprb_cur_scores(double *A, long long lda, int n, double l_tol, double *w_host, double *omega, int *n_low_host,
                               void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(A && w_host && omega && n_low_host && n > 0 && lda >= n, "gprb_cur_scores: bad argument");
    int rc = handles(st);
    if (rc) return rc;
    Scratch scratch(st);
    double *w = (double *)scratch.get((size_t)n * sizeof(double));
    int *info = (int *)scratch.get(sizeof(int));
    if (!w || !info) return GPRB_ERR_CUDA;
    int lwork = 0;
    if (cusolverDnDsyevd_bufferSize(g_solver, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, A, (int)lda, w, &lwork) !=
        CUSOLVER_STATUS_SUCCESS) { gprb_set_error("syevd_bufferSize failed"); return GPRB_ERR_CUDA; }
    double *work = (double *)scratch.get((size_t)(lwork > 0 ? lwork : 1) * sizeof(double));
    if (!work) return GPRB_ERR_CUDA;
    cusolverStatus_t cs = cusolverDnDsyevd(g_solver, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, A, (int)lda, w, work, lwork, info);
    if (cs != CUSOLVER_STATUS_SUCCESS) { gprb_set_error("cusolverDnDsyevd status %d", (int)cs); return GPRB_ERR_CUDA; }
    int hinfo = -1;
    GPRB_CUDA(cudaMemcpyAsync(w_host, w, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    GPRB_CUDA(cudaStreamSynchronize(st));
    if (hinfo != 0) { gprb_set_error("syevd did not converge (info = %d)", hinfo); return GPRB_ERR_LINALG; }
    int n_low = 0;
    while (n_low < n && w_host[n_low] < l_tol) n_low++;        // eigenvalues are ascending
    *n_low_host = n_low;
    leverage_kernel<<<(n + 255) / 256, 256, 0, st>>>(A, lda, n, n_low, omega);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

// dst[j][i] = src[i][j] for a rows x cols block (32 x 32 tiles through shared memory)
__global__ void transpose_copy_kernel(double *dst, long long ldd, const double *src, long long lds, int rows, int cols) {
    __shared__ double t[32][33];
    const int i = blockIdx.y * 32 + threadIdx.y, j = blockIdx.x * 32 + threadIdx.x;
    if (i < rows && j < cols) t[threadIdx.y][threadIdx.x] = src[(long long)i * lds + j];
    __syncthreads();
    const int tj = blockIdx.x * 32 + threadIdx.y, ti = blockIdx.y * 32 + threadIdx.x;   // dst row = src col
    if (tj < cols && ti < rows) dst[(long long)tj * ldd + ti] = t[threadIdx.x][threadIdx.y];
}

extern "C" int gprb_transpose_copy(double *dst, long long ldd, const double *src, long long lds, int rows, int cols, void *stream) {
    GPRB_REQUIRE(dst && src && rows >= 0 && cols >= 0, "gprb_transpose_copy: bad argument");
    if (rows == 0 || cols == 0) return GPRB_OK;
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 32);
    transpose_copy_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(dst, ldd, src, lds, rows, cols);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

extern "C" int gprb_symmetrize(double *A, long long ld, int n, void *stream) {
    GPRB_REQUIRE(A && n >= 0, "gprb_symmetrize: bad argument");
    if (n == 0) return GPRB_OK;
    dim3 grid((n + 31) / 32, (n + 31) / 32), block(32, 32);
    mirror_upper_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(A, ld, n);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}

namespace {
__global__ void dmma_peak_kernel(double *out, int iters) {
    double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
    double c[16][2];
#pragma unroll
    for (int i = 0; i < 16; i++) { c[i][0] = 0.0; c[i][1] = 0.0; }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += c[i][0] + c[i][1];
    if (s == 123.456) out[threadIdx.x] = s;
}
}  // namespace

extern "C" int gprb_fp64_dmma_peak(double *tflops_host, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(tflops_host, "gprb_fp64_dmma_peak: NULL output");
    int dev = 0, sms = 0;
    GPRB_CUDA(cudaGetDevice(&dev));
    GPRB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    double *d = nullptr;
    GPRB_CUDA(cudaMalloc((void **)&d, 1024 * sizeof(double)));
    cudaEvent_t e0, e1;
    GPRB_CUDA(cudaEventCreate(&e0));
    GPRB_CUDA(cudaEventCreate(&e1));
    const int iters = 20000, warps = 8;
    dmma_peak_kernel<<<sms, warps * 32, 0, st>>>(d, iters / 10);
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        GPRB_CUDA(cudaEventRecord(e0, st));
        dmma_peak_kernel<<<sms, warps * 32, 0, st>>>(d, iters);
        GPRB_CUDA(cudaEventRecord(e1, st));
        GPRB_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        GPRB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops_host = (double)sms * warps * iters * 16.0 * 512.0 / (best * 1e-3) * 1e-12;
    return GPRB_OK;
}
