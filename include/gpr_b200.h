/*
 * gpr_b200.h — C ABI of libgpr_b200.so, the B200 (sm_100a) implementation of the covariance hot
 * path of MaterSim/GPR_calculator.
 *
 * This header is the drop-in boundary.  The reference binds 13 scalar CPU loops through cffi
 * (gpr_calc/kernels/rbf_kernel.h:4-38, dot_kernel.h:4-27, loaded by rbf_kernel.py:4 and
 * dot_kernel.py:4).  Each entry point below names the reference symbol(s) it replaces.
 *
 * Differences from the reference ABI, all deliberate (SURVEY.md §8b):
 *   - inputs are packed ONCE into a device-resident `gprb_pack` (pre-normalised rows in the DMMA
 *     tile layout) instead of being re-marshalled for every call (rbf_kernel.py:40-45);
 *   - groups are described by a host array of rows-per-group (the reference's `indices` list),
 *     not by per-row group ids;
 *   - outputs are OVERWRITTEN (the reference accumulates into caller-zeroed buffers), already
 *     carry the wrapper normalisations (1/n_I, 1/(n_I n_J), sigma^2 zeta ...) and can be written
 *     straight into a sub-block of a larger row-major matrix through a leading dimension;
 *   - every call takes a cudaStream_t (as void*) and returns an int status
 *     (0 = ok; see gprb_last_error()); nothing falls back to the CPU;
 *   - a group window [grp_begin, grp_end) on side 1 selects the row block a rank owns
 *     (replaces the mpi4py row split of RBF_mb.py:471-481).
 *
 * Pointer conventions: `*_host` = host memory, `*_dev` = device memory, `*_any` = either (UVA).
 * All matrices are row-major float64.  Threading: calls on different streams may be issued
 * from different host threads; a pack must not be destroyed while a call using it is in flight.
 */
#ifndef GPR_B200_H
#define GPR_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gprb_pack gprb_pack;

enum { GPRB_OK = 0, GPRB_ERR_ARG = 1, GPRB_ERR_CUDA = 2, GPRB_ERR_UNSUPPORTED = 3, GPRB_ERR_LINALG = 4 };
enum { GPRB_KERNEL_RBF = 0, GPRB_KERNEL_DOT = 1 };
/* mode of the force-force builder */
enum { GPRB_FF_FULL = 0,      /* every (I,J) block of the window                                  */
       GPRB_FF_SYMMETRIC = 1, /* side1 is side2: evaluate J >= I only and mirror the block         */
       GPRB_FF_DIAG = 2,      /* only the diagonal entries of the (I,I) blocks -> vector [3*G]     */
       GPRB_FF_UPPER = 3 };   /* side1 is side2, any window: evaluate J >= I only, no mirroring; the
                                 blocks left of the diagonal are NOT written (see gprb_symmetrize)   */

int gprb_version(void);
const char *gprb_last_error(void);   /* thread-local message of the last failing call */
int gprb_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* number of CUDA kernels this library has launched in the process so far (bench.py's gpu_launches) */
long long gprb_launch_count(void);

/* ---- packing -------------------------------------------------------------------------------
 * Replaces utilities.list_to_tuple (utilities.py:340-390) + the per-call cffi marshalling and the
 * per-pair norm recomputation (rbf_kernel.cpp:364-381).
 *   ncols = 0 : energy rows (x only)          -> tiles of [x^]
 *   ncols = 3 : force rows (x, dxdr[.,d,3])   -> tiles of [x^; A~_x; A~_y; A~_z]
 * with x^ = x/|x| and A~ = (I - x^ x^T) dxdr / |x|.  Rows with |x| <= 1e-8 are dropped as in
 * rbf_kernel.cpp:26,37.  group_rows_host[g] = number of rows of group g (the `indices` list).
 * x_any/dxdr_any/ele_any may be host or device pointers.
 * The descriptor length d must be at most 64 (the longest the covariance kernels take); a longer one
 * returns GPRB_ERR_UNSUPPORTED before any CUDA call, with *out = NULL.
 * norm_eps = 0 is the covariance convention.  norm_eps > 0 replaces |x| by |x| + norm_eps everywhere
 * and drops nothing: the convention of the numpy K_ff that Dot_mb.diag alone uses (Dot_mb.py:204-221). */
int gprb_pack_create(gprb_pack **out, int n_groups, const int *group_rows_host, int d, int ncols,
                     const double *x_any, const double *dxdr_any, const int *ele_any, double norm_eps,
                     void *stream);
void gprb_pack_destroy(gprb_pack *p);
int gprb_pack_info(const gprb_pack *p, int *n_groups, int *n_rows, int *d, int *ncols, int *n_tiles);
/* number of same-species, non-dropped row pairs between groups [g0,g1) of a and all groups of b
 * (the unit of work of SURVEY.md §8d); computed on the host from cached per-group species counts */
long long gprb_pack_pair_count(const gprb_pack *a, int g0, int g1, const gprb_pack *b);

/* ---- atom plan of a force pack (host part; no device needed) -----------------------------------
 * gprb_kff and gprb_kef with dK/dl (RBF) over a whole force pack use the factored build when the pack's rows are
 * copies of a few atoms' descriptors (one row per neighbour atom of every force centre of a structure).
 * gprb_atom_plan_host cuts the groups into clusters of consecutive groups whose distinct rows, keyed by
 * (hash, code), number at most a_max (and at most max_groups groups); a new cluster also starts when a
 * group shares no key with the current one.  Rows with unique[r] != 0 (may be NULL) always get a slot
 * of their own.  Outputs: cluster_grp [n_groups + 1] first group of each cluster (and the end),
 * cluster_slots [n_groups] slots per cluster, row_slot [n_rows] slot of each row inside its cluster,
 * slot_rep [n_rows] the first row of every slot, cluster after cluster.  Returns GPRB_ERR_UNSUPPORTED
 * with *n_clusters = 0 when one group alone has more than a_max distinct rows.
 * gprb_atom_plan_cost: the DMMA instructions the pairwise kernel and the factored build execute for
 * such a plan (upper != 0: the J >= I group blocks of GPRB_FF_UPPER / SYMMETRIC, else every block);
 * gprb_kff takes the factored build when pairwise >= 2 x factored.
 * gprb_atom_plan_cost_kef: the same for gprb_kef with dK/dl of such a force pack (n_rows rows) against an
 * energy pack of n_energy_rows rows in n_energy_groups groups; gprb_kef takes the factored build on the
 * same rule. */
int gprb_atom_plan_host(int n_groups, const int *row_ptr, const unsigned long long *hash, const int *code,
                        const unsigned char *unique, int a_max, int max_groups,
                        int *n_clusters, int *cluster_grp, int *cluster_slots, int *row_slot, int *slot_rep);
int gprb_atom_plan_cost(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows, int upper,
                        double *pairwise_dmma, double *factored_dmma);
int gprb_atom_plan_cost_kef(int n_clusters, const int *cluster_grp, const int *cluster_slots, int n_rows,
                            int n_energy_rows, int n_energy_groups, double *pairwise_dmma, double *factored_dmma);

/* ---- covariance blocks ------------------------------------------------------------------------
 * kernel = GPRB_KERNEL_RBF: p0 = sigma, p1 = l.   GPRB_KERNEL_DOT: p0 = sigma, p1 = sigma0.
 * dK_dev may be NULL (no hyper-parameter gradient).  For RBF dK is dK/dl; dK/dsigma = 2K/sigma is
 * never materialised.  For DOT the gradient blocks are closed-form constants and are not produced.
 *
 * gprb_kff : force-force block.  Replaces rbf_kff_many (rbf_kernel.cpp:341-473, use_tol=1),
 *            rbf_kff_many_with_grad (:475-640, use_tol=0, dK_dev != NULL), dot_kff_many
 *            (dot_kernel.cpp:217-336) and their wrappers kff_C (rbf_kernel.py:191-337,
 *            dot_kernel.py:162-270).
 *            K[(3(I-grp_begin)+c)*ldk + 3J+e]; in GPRB_FF_SYMMETRIC mode side 1 must be side 2,
 *            the window must be the whole set and the mirrored entries are written too;
 *            in GPRB_FF_DIAG mode K is a vector [3*(grp_end-grp_begin)]. */
int gprb_kff(int kernel, const gprb_pack *f1, const gprb_pack *f2, double p0, double p1, double zeta,
             int use_tol, double tol, int mode, int grp_begin, int grp_end,
             double *K_dev, long long ldk, double *dK_dev, long long lddk, void *stream);

/* gprb_kef : energy-force block K_ef[I, 3J+c] (I = energy group of `e`, J = force group of `f`),
 *            window over the FORCE groups.  Replaces rbf_kef_many / _with_grad
 *            (rbf_kernel.cpp:101-253), dot_kef_many (dot_kernel.cpp:58-130), kef_C.
 *            Kef_dev[I*ld_ef + 3(J-grp_begin)+c] and/or its transpose
 *            Kfe_dev[(3(J-grp_begin)+c)*ld_fe + I]; either may be NULL. */
int gprb_kef(int kernel, const gprb_pack *e, const gprb_pack *f, double p0, double p1, double zeta,
             int grp_begin, int grp_end,
             double *Kef_dev, long long ld_ef, double *Kfe_dev, long long ld_fe,
             double *dKef_dev, long long ld_def, double *dKfe_dev, long long ld_dfe, void *stream);

/* ---- row-sharded build with the all-gather fused into the epilogue ------------------------------
 * The reference gathers the row slabs of every MPI rank as pickles on rank 0, vstacks them and
 * broadcasts the result (RBF_mb.py:471-521, gaussianprocess.py:246-247, 305-306).  Here the GPU that
 * owns a row block stores every finished value straight into the same slab of ALL copies of K:
 * K_dst_host[0] is the slab in this GPU's matrix, K_dst_host[1..n_dst) the same slab in the peers'
 * matrices (device pointers mapped with gprb_peer_open; NVLink peer stores / fp64 reductions issued by
 * the kernel epilogue, overlapped with the DMMAs of the following column groups).  dK stays local.
 * Unlike gprb_kff / gprb_kef the K destinations are NOT zeroed by the call (a GPU cannot order a memset
 * of a peer's matrix against that peer's other writers): every GPU zeroes its own matrix, the ranks
 * synchronise, then build; they synchronise again before anyone reads K.
 * gprb_kff_multi: mode GPRB_FF_FULL or GPRB_FF_UPPER.  gprb_kfe_multi: the K_fe rows of the force
 * window (K_fe[(3(J-grp_begin)+c)*ld_fe + I]). */
#define GPRB_MAX_DST 8
int gprb_kff_multi(int kernel, const gprb_pack *f1, const gprb_pack *f2, double p0, double p1, double zeta,
                   int use_tol, double tol, int mode, int grp_begin, int grp_end,
                   int n_dst, double *const *K_dst_host, long long ldk, double *dK_dev, long long lddk, void *stream);
int gprb_kfe_multi(int kernel, const gprb_pack *e, const gprb_pack *f, double p0, double p1, double zeta,
                   int grp_begin, int grp_end, int n_dst, double *const *Kfe_dst_host, long long ld_fe,
                   double *dKfe_dev, long long ld_dfe, void *stream);

/* Peer-visible device memory for the fused gather (one process per GPU on one NVLink / NVSwitch node).
 * gprb_peer_alloc: cudaMalloc on the current device.  gprb_peer_export: 64-byte CUDA IPC handle to hand to
 * the other processes (any transport; dist.py uses torch.distributed).  gprb_peer_open: map another
 * process's allocation into this one with peer access enabled; the pointer is valid for kernels on the
 * current device.  gprb_peer_close / gprb_peer_free undo them. */
int gprb_peer_alloc(void **ptr_dev, unsigned long long bytes);
int gprb_peer_free(void *ptr_dev);
int gprb_peer_export(void *ptr_dev, unsigned char *handle64_host);
int gprb_peer_open(const unsigned char *handle64_host, void **ptr_dev);
int gprb_peer_close(void *ptr_dev);

/* gprb_kee : energy-energy block K[(I-grp_begin)*ldk + J].  Replaces rbf_kee_many / _with_grad
 *            (rbf_kernel.cpp:5-98), dot_kee_many (dot_kernel.cpp:5-56), kee_C. */
int gprb_kee(int kernel, const gprb_pack *e1, const gprb_pack *e2, double p0, double p1, double zeta,
             int grp_begin, int grp_end, double *K_dev, long long ldk, double *dK_dev, long long lddk,
             void *stream);

/* gprb_kee_diag : prior variance of energy rows with the eps-regularised numpy formula the
 *            reference uses only in diag() (kernels/base.py:107-130 K_ee_RBF, Dot_mb.py:177-202). */
int gprb_kee_diag(int kernel, const gprb_pack *e, double p0, double p1, double zeta,
                  double *out_dev, void *stream);

/* ---- GP algebra on device (gaussianprocess.py:128-202, 286-317, 319-379, 880-908) ------------ */
/* K[i,i] += (i < NE ? noise_e^2 : noise_f^2)                       (gaussianprocess.py:165-173) */
int gprb_add_noise(double *K_dev, long long ldk, int N, int NE, double noise_e, double noise_f, void *stream);
/* In-place Cholesky K = L L^T (cuSOLVER potrf).  Returns GPRB_ERR_LINALG if not positive definite
 * (the reference maps that to LML = -inf, gaussianprocess.py:174-177). */
int gprb_chol_factor(double *K_dev, long long ldk, int N, void *stream);
/* A[i][j] = A[j][i] for all i > j of the n x n block at A (fills the lower triangle from the upper
 * one after an all-gather of GPRB_FF_UPPER row blocks). */
int gprb_symmetrize(double *A_dev, long long ld, int n, void *stream);
/* dst[j*ldd + i] = src[i*lds + j] for a rows x cols block (K_ef = K_fe^T after a row-sharded build). */
int gprb_transpose_copy(double *dst_dev, long long ldd, const double *src_dev, long long lds, int rows, int cols, void *stream);
/* Rows of the inverse without forming it (row-sharded likelihood gradient: a rank that holds the rows
 * [r0, r1) of dK with valid entries right of the diagonal only needs Kinv[r0:r1, c0:N] with c0 <= r0):
 *   out[k*ldo + t] = Kinv[r0 + k, c0 + t],  k < r1 - r0,  t < N - c0,
 * from the TRAILING block of the factor, K^-1[T,T] = (L_TT L_TT^T)^-1 for T = [c0, N) (two cuBLAS trsm, i.e. potrs, with
 * r1 - r0 unit right-hand sides on the (N - c0)-dimensional trailing system: 2 (N-c0)^2 (r1-r0) flops
 * instead of forming the whole inverse on every rank).  c0 = 0 gives full rows (the energy rows). */
int gprb_chol_inverse_rows(const double *L_dev, long long ldl, int N, int r0, int r1, int c0,
                           double *out_dev, long long ldo, void *stream);
/* Live FP64 tensor-pipe roofline denominator: DMMA.8x8x4 issue-rate micro-benchmark (all SMs,
 * 16 independent accumulators per warp).  MEASURED_PEAKS.json carries no fp64 entry. */
int gprb_fp64_dmma_peak(double *tflops_host, void *stream);
/* One likelihood evaluation after the covariance build, enqueued back to back with a single host synchronisation
 * (GP.log_marginal_likelihood, gaussianprocess.py:160-198; the scipy cholesky / cho_solve / einsum steps of :174-198):
 * K += noise on the diagonal, in-place Cholesky, alpha = K^-1 y, and -- want_grad -- the traces of
 * W = alpha alpha^T - K^-1 against the rows of dK/dl this rank holds, K^-1 taken block of rows by block of rows
 * (N / parts rows, >= 512) from trailing-block triangular solves as in gprb_chol_inverse_rows (no explicit inverse).
 *   ranges_host[2 n_ranges]: row ranges (r0, r1) of the assembled matrix whose rows of dK are stacked in
 *     dK_rows_dev (leading dimension lddk; NULL = no dK term).  Only the entries of the row-sharded build are read:
 *     an energy row i < NE reads the K_ee columns j in [i, NE), a force row i >= NE the K_fe columns j < NE and the
 *     columns j >= i (J >= I blocks of K_ff); W and dK are symmetric, so off-diagonal terms count twice.  A full dK
 *     satisfies this layout.
 *   alpha_dev[N] receives alpha; K_dev holds the factor on return.
 *   out_host[8]: [0] sum_i log L_ii, [1] y.alpha, [2] 1/2 tr(W dK) over the held rows, [3] 1/2 sum W_ii noise_i^2,
 *     [4] 1/2 sum W_ii 2 noise_i, [5] 1/2 sum of W over (held energy rows) x (all energy columns) when want_s0
 *     (the Dot kernel's d/dsigma0 term, dot_kernel.py:58).  Sharded callers all-reduce [2..5].  [6], [7]: device milliseconds
 *     of the factor + alpha phase and of the gradient phase (solves + traces) of this call.
 * Returns GPRB_ERR_LINALG when K is not positive definite (gaussianprocess.py:174-177).
 *   prefactored != 0: K_dev already holds the factor of K + noise in its row-major lower triangle (the multi-GPU Cholesky below);
 *     noise and potrf are skipped.
 *   work_dev: caller-owned workspace of gprb_lml_eval_work(N, NE, want_grad, parts) doubles (the K^-1 slabs of one block of rows
 *     and of the energy rows; may be NULL when want_grad = 0). */
int gprb_lml_eval(double *K_dev, long long ldk, int N, int NE, const double *y_dev, double noise_e, double noise_f,
                  const double *dK_rows_dev, long long lddk, int n_ranges, const int *ranges_host,
                  int want_grad, int want_s0, int parts, int prefactored, double *alpha_dev, double *work_dev,
                  long long work_doubles, double *out_host, void *stream);
long long gprb_lml_eval_work(int N, int NE, int want_grad, int parts);
/* Building blocks of the multi-GPU right-looking Cholesky (every rank holds a full row-major copy of K + noise; block column k
 * of the lower triangle is owned by rank k mod G; dist.distributed_cholesky broadcasts each finished panel to all ranks):
 *   gprb_chol_panel    (owner of k): L_kk = chol(A_kk) (cuSOLVER potrf, nbk x nbk), then L_ik = A_ik L_kk^-T for the rows below
 *                      (one cuBLAS trsm); *info_dev keeps the first failing row (0 = positive definite so far); no host sync.
 *   gprb_chol_trailing (owner of j > k): A[j0:N, j0:j0+nbj] -= L[j0:N, k0:k0+nbk] L[j0:j0+nbj, k0:k0+nbk]^T (one cuBLAS gemm).
 * Replaces the replicated scipy cholesky of gaussianprocess.py:174 on every MPI rank. */
int gprb_chol_panel(double *K_dev, long long ldk, int N, int k0, int nbk, int *info_dev, void *stream);
int gprb_chol_trailing(double *K_dev, long long ldk, int N, int k0, int nbk, int j0, int nbj, void *stream);

/* mean[i] = Ks[i,:].alpha ;  if var_dev: var[i] = max(diag[i] - Ks[i,:] Kinv Ks[i,:]^T, 0)
 * (cuBLAS DGEMM + fused row reduction; gaussianprocess.py:880, 904-908).  work_dev: [m, N] scratch. */
int gprb_predict(int m, int N, const double *Ks_dev, long long ldks, const double *alpha_dev,
                 const double *Kinv_dev, long long ldi, const double *diag_dev,
                 double *mean_dev, double *var_dev, double *work_dev, void *stream);

/* Same outputs from the Cholesky factor instead of the explicit inverse: var[i] = max(diag[i] - |L^-1 Ks[i,:]^T|^2, 0)
 * (one cuBLAS trsm with m right-hand sides, m N^2 flops instead of 2 m N^2, no N x N inverse to form after a fit).
 * Used for batches of test rows; work_dev: [m, N] scratch. */
int gprb_predict_chol(int m, int N, const double *Ks_dev, long long ldks, const double *alpha_dev,
                      const double *L_dev, long long ldl, const double *diag_dev,
                      double *mean_dev, double *var_dev, double *work_dev, void *stream);

/* cov_dev (m x m, holds k(X, X) on entry) -= K* K^-1 K*^T through the factor, as GP.predict(return_cov=True) does with
 * cho_solve (gaussianprocess.py:363-366): one cuBLAS trsm with m right-hand sides + one m x m x N gemm.  work_dev: [m, N]. */
int gprb_predict_cov(int m, int N, const double *Ks_dev, long long ldks, const double *L_dev, long long ldl,
                     double *cov_dev, long long ldc, double *work_dev, void *stream);

/* CUR leverage scores of a symmetric block (CUR(), gaussianprocess.py:1165-1182; Jinnouchi et al. PRB 100, 014105 App. D):
 * cuSOLVER syevd in place (A_dev is destroyed: row k = eigenvector of the k-th smallest eigenvalue), eigenvalues to
 * w_host[n], omega_dev[i] = sum_{k: w_k < l_tol} U[i,k]^2, *n_low_host = #{w_k < l_tol}. */
int gprb_cur_scores(double *A_dev, long long lda, int n, double l_tol, double *w_host, double *omega_dev, int *n_low_host,
                    void *stream);

/* ---- SO(3) power-spectrum descriptor (gpr_calc/SO3.py:186-727), batched over structures --------
 * Atoms of all structures are concatenated; atom_ptr[S+1] gives the first atom of each structure,
 * struct_of[n_atoms] the structure of each atom.  All pointers are device pointers.
 *
 * gprb_so3_neighbors : replaces SO3.build_neighbor_list (SO3.py:348-407) and the un-vendored
 *   ase.neighborlist.NeighborList it calls (:357-363): all (i, j, S) with |r_j + S.cell - r_i| < rcut
 *   except (i, i, 0); nimg[S,3] = images searched per axis (0 on non-periodic axes).
 *   mode 0 counts: nnb[i] neighbours and nuniq[i] = |{j} U {i}| rows of `seq`;
 *   mode 1 fills nb_j / nb_rvec at nb_ptr[i] (exclusive scan of nnb), sorted by (j, S).
 * gprb_so3_radial    : radial integrals of compute_dcs (SO3.py:619-652) per neighbour,
 *   rad[w] = { I[nmax][lmax+1], dI/dr[nmax][lmax+1] }; rho[nq], G[nmax,nq] are the quadrature
 *   nodes and the combined weights g_n(rho) rho^2 e^{-a rho^2} sqrt(1-t^2) w (SO3.py:633,646-647).
 * gprb_so3_power     : c_nlm, power spectrum x[n_atoms,d], dxdr[n_seq,d,3] and seq[n_seq,2] (int64,
 *   atom indices local to the structure) (SO3.py:243-273, 655-727); seq_ptr = exclusive scan of nuniq.
 *   derivative: bit 0 = also dxdr / seq; bit 1 = weight_on (SO3.py:381-385: a neighbour whose species differs
 *   from the centre's enters with weight -Z_j instead of Z_j).
 *   rdxdr != NULL (stress, SO3.py:253-273, 304-306): also rdxdr[n_seq,d,3,3] = -pstress / volume with
 *   pos[n_atoms,3] the atom positions and inv_vol[S] = 1 / cell volume of each structure. */
int gprb_so3_neighbors(int n_struct, int n_atoms, const int *atom_ptr, const int *struct_of,
                       const double *pos, const double *cell, const int *nimg, double rcut,
                       int mode, int *nnb, int *nuniq, const int *nb_ptr, int *nb_j, double *nb_rvec,
                       void *stream);
int gprb_so3_radial(int n_nb, const double *nb_rvec, int nmax, int lmax, int nq, double alpha, double rcut,
                    const double *rho, const double *G, double *rad, void *stream);
int gprb_so3_power(int n_atoms, const int *nb_ptr, const int *nb_j, const double *nb_rvec, const double *rad,
                   const int *numbers, const int *atom_ptr, const int *struct_of, const int *seq_ptr,
                   int nmax, int lmax, double alpha, double rcut, const double *norm_l, int derivative,
                   double *x, double *dxdr, long long *seq,
                   const double *pos, const double *inv_vol, double *rdxdr, void *stream);

/* gprb_virial_rows : strain derivative of every atom's descriptor, the row of that atom in its structure's
 *   total-stress group:  out[a, k, v] = sum_{q in [seq_ptr[a], seq_ptr[a+1])} rdxdr[q, k, voigt(v)]
 *   with v = xx, yy, zz, xy, xz, yz; seq_ptr[n_atoms + 1] and rdxdr[n_seq, d, 3, 3] as gprb_so3_power writes them,
 *   out [n_atoms, d, 6].  Each entry is summed by one thread in increasing q (bitwise reproducible).
 *   GPRB_ERR_ARG for n_atoms < 0, d outside [1, 64] or a NULL pointer (n_atoms > 0). */
int gprb_virial_rows(int n_atoms, int d, const int *seq_ptr_dev, const double *rdxdr_dev, double *out_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GPR_B200_H */
