// Shared declarations for libgpr_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdarg>
#include <vector>
#include <map>
#include <cstdint>
#include "../../include/gpr_b200.h"

#define GPRB_TILE_ROWS 8           // rows of one DMMA operand tile (M or N of mma.m8n8k4)
#define GPRB_MAX_KS 8              // k-steps of 4 held in registers (d <= 32) by the MMA kernels
#define GPRB_EPS_NORM 1e-8         // rbf_kernel.cpp:10,26

void gprb_set_error(const char *fmt, ...);
int gprb_pool_init();            // stream-ordered pool of the current device, memory kept across synchronisations (pack.cu)
void gprb_pool_free(void *ptr, cudaStream_t st);  // cudaFreeAsync ordered on st (NULL pointer is fine)

struct gprb_pack;
int gprb_check_device(const gprb_pack *p, const char *who);   // GPRB_ERR_ARG unless the pack lives on the current device (pack.cu)

// kernels launched by this library so far (gprb_launch_count); bumped next to every <<< >>>
#include <atomic>
extern std::atomic<long long> g_gprb_launches;
#define GPRB_LAUNCHED() (g_gprb_launches.fetch_add(1, std::memory_order_relaxed))

#define GPRB_CUDA(call)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (call);                                                                \
        if (_e != cudaSuccess) {                                                                \
            gprb_set_error("%s:%d CUDA error %s (%s)", __FILE__, __LINE__, cudaGetErrorName(_e), \
                           cudaGetErrorString(_e));                                             \
            return GPRB_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)

#define GPRB_REQUIRE(cond, ...)                                                                 \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            gprb_set_error(__VA_ARGS__);                                                        \
            return GPRB_ERR_ARG;                                                                \
        }                                                                                       \
    } while (0)

// Device-resident packed side of a covariance block.
//
// Flat tile layout (the unit every kernel consumes): the rows of all groups are concatenated in
// group order WITHOUT per-group padding and cut into tiles of 8 consecutive rows, so a tile may hold
// the last rows of one group and the first rows of the next (only the tail of the pack is padded, to
// a multiple of GPRB_CHUNK_TILES tiles).  One tile stores, for each component c (0 = x^, 1..3 = A~
// columns), the 8 x (4*ks) operand slab in k-step-major order
//        P[((tile*ncomp + c)*ks + kstep)*32 + row*4 + kk]      (k = 4*kstep + kk, zero padded)
// so that the m8n8k4 fragment of (c, kstep) is the 32 consecutive doubles read by lane = row*4+kk:
// one fully coalesced 256-byte access from global memory and a conflict-free one from shared
// memory after a verbatim bulk copy.
//
// Tile record (GPRB_REC_INTS ints per tile, travels with the tile through the TMA ring):
//   [0..7]  species of the 8 rows (-1 padding, -(z+2) dropped because |x| <= eps)
//   [8]     number of group segments in the tile
//   [10+2s] group id of segment s ; [11+2s] = row mask (bits 0..7) | 0x100 if the group ends in this tile
#define GPRB_CHUNK_TILES 4         // tiles per column chunk (one TMA stage)
#define GPRB_REC_INTS 28           // 112 bytes: a multiple of 16 for cp.async.bulk

struct gprb_atom_plan;               // atom plan of a force pack (cov_factored.cu)
void gprb_atom_plan_free(gprb_atom_plan *plan, cudaStream_t st);
// K_ff + dK/dl (RBF) of a force pack against itself, full window, one pre-zeroed destination, over the atoms its rows share
// (cov_factored.cu); *done = false when the pairwise kernel is to run instead
int gprb_kff_factored(gprb_pack *f, double p0, double p1, double zeta, int mode, double *K, long long ldk, double *dK,
                      long long lddk, cudaStream_t st, bool *done);

struct gprb_pack {
    int n_groups = 0, n_rows = 0, d = 0, ncols = 0, ncomp = 0, ks = 0, n_tiles = 0;
    int device = 0;
    cudaStream_t stream = nullptr; // creation stream: the pack's buffers are returned to the pool in its order
    std::vector<int> group_rows;   // host, [G]
    std::vector<int> row_ptr;      // host, [G+1]  first flat row of each group
    // per-group species histogram (non-dropped rows) for pair counting
    std::vector<std::map<int, long long>> species;
    bool species_ready = false;
    // device buffers
    double *P = nullptr;           // [n_tiles][ncomp][ks][32]
    double *norm = nullptr;        // [n_tiles*8]  |x| of each row (0 for padding)
    int *elep = nullptr;           // [n_tiles*8]  species; -1 padding; -(z+2) dropped (|x|<=eps)
    int *row_group = nullptr;      // [n_tiles*8]  group of each flat row (-1 padding)
    int *tile_rec = nullptr;       // [n_tiles][GPRB_REC_INTS]
    int *d_row_ptr = nullptr;      // [G+1]
    int *d_group_rows = nullptr;   // [G]
    uint64_t *row_hash = nullptr;  // [n_tiles*8]  hash of the raw x bits and the species code of each row (0 for padding)
    // atom plan of the factored K_ff path (cov_factored.cu): built on the first call that can use it
    gprb_atom_plan *plan = nullptr;
    bool plan_tried = false;
    // cached row-side schedule for the last window used (see cov_mma.cu)
    int sched_g0 = -1, sched_g1 = -1, sched_n = 0;
    int4 *sched = nullptr;         // device [sched_n] {tile0, ntiles, entry_begin, n_entries}
    int4 *sched_ent = nullptr;     // device entries {group, row0, row1 (block-local rows), shared}
    std::vector<int4> sched_host, sched_ent_host;
};
