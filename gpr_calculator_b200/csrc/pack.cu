// pack.cu — device-resident packed operands (`gprb_pack`) and the row-preparation kernel.
//
// Replaces, for the whole life of a training set, what the reference redoes on every kernel call:
// list_to_tuple (utilities.py:340-390), the ravel().tolist() marshalling (rbf_kernel.py:40-45,
// 246-252) and the per-pair norm / projection arithmetic (rbf_kernel.cpp:364-399).
#include "common.cuh"
#include <cstring>
#include <string>

static thread_local std::string g_err;

void gprb_set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
}

extern "C" const char *gprb_last_error(void) { return g_err.c_str(); }
extern "C" int gprb_version(void) { return 101; }

std::atomic<long long> g_gprb_launches{0};
extern "C" long long gprb_launch_count(void) { return g_gprb_launches.load(); }

extern "C" int gprb_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    GPRB_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    GPRB_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return GPRB_OK;
}

// splitmix64 finaliser
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// One warp per row of the flat tile layout (rows >= n_rows are tail padding).
// HBM-bound: reads 8*d*(1+ncols) bytes and writes 8*4ks*(1+ncols) per row.
__global__ void prep_rows_kernel(int n_padded, int n_rows, int d, int ncols, int ks, double norm_eps,
                                 const double *__restrict__ x, const double *__restrict__ dxdr,
                                 const int *__restrict__ ele,
                                 double *__restrict__ P, double *__restrict__ norm_out,
                                 int *__restrict__ elep, int *__restrict__ tile_rec, uint64_t *__restrict__ row_hash) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= n_padded) return;
    const int ncomp = 1 + ncols;
    const int tile = warp >> 3, r = warp & 7;
    const int kp = 4 * ks;
    const int src = warp < n_rows ? warp : -1;
    double *Pt = P + (size_t)tile * ncomp * ks * 32;
    if (src < 0) {   // padding row
        for (int c = 0; c < ncomp; c++)
            for (int k = lane; k < kp; k += 32) Pt[((size_t)c * ks + (k >> 2)) * 32 + r * 4 + (k & 3)] = 0.0;
        if (lane == 0) { norm_out[warp] = 0.0; elep[warp] = -1; tile_rec[(size_t)tile * GPRB_REC_INTS + r] = -1; row_hash[warp] = 0; }
        return;
    }
    const double *xr = x + (size_t)src * d;
    double ss = 0.0;
    uint64_t h = 0;                 // sum over k of mix(bits(x_k), k): equal rows hash equally (the atom plan's merge key)
    for (int k = lane; k < d; k += 32) {
        double v = xr[k];
        ss += v * v;
        h += mix64((uint64_t)__double_as_longlong(v) + (uint64_t)k * 0x9e3779b97f4a7c15ull);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, (unsigned long long)h, o);
    const double n = sqrt(ss) + norm_eps;
    const bool dropped = (norm_eps == 0.0) && !(n > GPRB_EPS_NORM);
    const double inv = dropped ? 0.0 : 1.0 / n;
    // t_c = x^ . A[:,c]
    double t[9];
    const double *Ar = ncols ? dxdr + (size_t)src * d * ncols : nullptr;
    for (int c = 0; c < ncols; c++) {
        double acc = 0.0;
        for (int k = lane; k < d; k += 32) acc += (xr[k] * inv) * Ar[(size_t)k * ncols + c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        t[c] = acc;
    }
    for (int k = lane; k < kp; k += 32) {
        const size_t off = (size_t)(k >> 2) * 32 + r * 4 + (k & 3);
        const double xh = (k < d) ? xr[k] * inv : 0.0;
        Pt[off] = xh;
        for (int c = 0; c < ncols; c++) {
            double v = 0.0;
            if (k < d && !dropped) v = (Ar[(size_t)k * ncols + c] - xh * t[c]) * inv;
            Pt[(size_t)(c + 1) * ks * 32 + off] = v;
        }
    }
    if (lane == 0) {
        norm_out[warp] = n - norm_eps;
        const int z = ele[src];
        const int code = dropped ? -(z + 2) : z;
        elep[warp] = code;
        tile_rec[(size_t)tile * GPRB_REC_INTS + r] = code;
        row_hash[warp] = mix64(h ^ ((uint64_t)(uint32_t)code * 0xc2b2ae3d27d4eb4full));
    }
}

static bool is_device_ptr(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

template <typename T>
static int stage_input(const T *any, size_t count, const T **dev, T **owned, cudaStream_t st) {
    *owned = nullptr;
    if (count == 0 || any == nullptr) { *dev = nullptr; return GPRB_OK; }
    if (is_device_ptr(any)) { *dev = any; return GPRB_OK; }
    GPRB_CUDA(cudaMallocAsync((void **)owned, count * sizeof(T), st));
    GPRB_CUDA(cudaMemcpyAsync(*owned, any, count * sizeof(T), cudaMemcpyHostToDevice, st));
    *dev = *owned;
    return GPRB_OK;
}

// All device memory of the library comes from the stream-ordered pool of the device with the release
// threshold raised to "never": packs are created and destroyed on every training-set change and once per
// predicted structure, and cudaMalloc / cudaFree (and a pool that hands its memory back to the OS at every
// synchronisation) showed up as random 0.1 - 1 s host stalls in the end-to-end likelihood step.
int gprb_pool_init() {
    static bool done[64] = {};
    int dev = 0;
    GPRB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || done[dev]) return GPRB_OK;
    cudaMemPool_t pool;
    GPRB_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    unsigned long long never = ~0ULL;
    GPRB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &never));
    done[dev] = true;
    return GPRB_OK;
}

// Frees are ordered on the stream the pack was created on (the stream its consumers normally run on; the header
// requires that no call using a pack is in flight when it is destroyed).  If that stream no longer exists the
// synchronous cudaFree is the safe fallback.
void gprb_pool_free(void *ptr, cudaStream_t st) {
    if (!ptr) return;
    if (cudaFreeAsync(ptr, st) != cudaSuccess) { cudaGetLastError(); cudaFree(ptr); }
}

int gprb_check_device(const gprb_pack *p, const char *who) {
    int dev = -1;
    GPRB_CUDA(cudaGetDevice(&dev));
    GPRB_REQUIRE(p == nullptr || p->device == dev, "%s: the pack was created on device %d but the current device is %d", who,
                 p ? p->device : -1, dev);
    return GPRB_OK;
}

extern "C" void gprb_pack_destroy(gprb_pack *p) {
    if (!p) return;
    cudaStream_t st = p->stream;
    gprb_pool_free(p->P, st); gprb_pool_free(p->norm, st); gprb_pool_free(p->elep, st); gprb_pool_free(p->row_group, st);
    gprb_pool_free(p->tile_rec, st); gprb_pool_free(p->d_row_ptr, st); gprb_pool_free(p->d_group_rows, st);
    gprb_pool_free(p->sched, st); gprb_pool_free(p->sched_ent, st); gprb_pool_free(p->row_hash, st);
    gprb_atom_plan_free(p->plan, st);
    delete p;
}

extern "C" int gprb_pack_create(gprb_pack **out, int n_groups, const int *group_rows_host, int d, int ncols,
                                const double *x_any, const double *dxdr_any, const int *ele_any, double norm_eps,
                                void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GPRB_REQUIRE(out != nullptr, "gprb_pack_create: out is NULL");
    *out = nullptr;
    GPRB_REQUIRE(n_groups >= 0 && d > 0, "gprb_pack_create: bad sizes n_groups=%d d=%d", n_groups, d);
    GPRB_REQUIRE(ncols == 0 || ncols == 3, "gprb_pack_create: ncols must be 0 (energy) or 3 (force), got %d", ncols);
    GPRB_REQUIRE(norm_eps >= 0.0, "gprb_pack_create: norm_eps must be >= 0");
    GPRB_REQUIRE(ncols == 0 || dxdr_any != nullptr || n_groups == 0, "gprb_pack_create: dxdr is NULL for a force pack");
    // the covariance kernels hold at most 2 * GPRB_MAX_KS k-steps of 4 (cov_mma.cu): refuse a pack none of them can use
    if (d > 8 * GPRB_MAX_KS) {
        gprb_set_error("gprb_pack_create: descriptor length %d > %d is not supported by the DMMA kernels", d, 8 * GPRB_MAX_KS);
        return GPRB_ERR_UNSUPPORTED;
    }
    { int rc0 = gprb_pool_init(); if (rc0) return rc0; }
    gprb_pack *p = new gprb_pack();
    p->stream = st;
    GPRB_CUDA(cudaGetDevice(&p->device));
    p->n_groups = n_groups; p->d = d; p->ncols = ncols; p->ncomp = 1 + ncols; p->ks = (d + 3) / 4;
    p->group_rows.assign(group_rows_host, group_rows_host + n_groups);
    p->row_ptr.resize(n_groups + 1);
    long long rows = 0;
    for (int g = 0; g < n_groups; g++) {
        int ng = p->group_rows[g];
        if (ng < 0) { delete p; GPRB_REQUIRE(false, "gprb_pack_create: negative group size"); }
        p->row_ptr[g] = (int)rows;
        rows += ng;
    }
    if (rows > 2000000000LL) { delete p; GPRB_REQUIRE(false, "gprb_pack_create: too many rows"); }
    p->row_ptr[n_groups] = (int)rows;
    int tiles = (int)((rows + GPRB_TILE_ROWS - 1) / GPRB_TILE_ROWS);
    tiles = (tiles + GPRB_CHUNK_TILES - 1) / GPRB_CHUNK_TILES * GPRB_CHUNK_TILES;
    p->n_tiles = tiles; p->n_rows = (int)rows;
    if (rows > 0 && (x_any == nullptr || ele_any == nullptr)) { delete p; GPRB_REQUIRE(false, "gprb_pack_create: x/ele NULL"); }

    const int n_padded = tiles * GPRB_TILE_ROWS;
    // per-row group ids and per-tile segment records (species slots are filled by the prep kernel)
    std::vector<int> rgroup(n_padded, -1), rec((size_t)tiles * GPRB_REC_INTS, 0);
    for (int g = 0; g < n_groups; g++)
        for (int r = p->row_ptr[g]; r < p->row_ptr[g + 1]; r++) rgroup[r] = g;
    for (int t = 0; t < tiles; t++) {
        int *R = rec.data() + (size_t)t * GPRB_REC_INTS;
        int nseg = 0;
        for (int r = 0; r < GPRB_TILE_ROWS; r++) {
            const int g = rgroup[t * GPRB_TILE_ROWS + r];
            if (g < 0) break;                                   // tail padding
            if (nseg == 0 || R[10 + 2 * (nseg - 1)] != g) { R[10 + 2 * nseg] = g; R[11 + 2 * nseg] = 0; nseg++; }
            R[11 + 2 * (nseg - 1)] |= 1 << r;
            if (t * GPRB_TILE_ROWS + r == p->row_ptr[g + 1] - 1) R[11 + 2 * (nseg - 1)] |= 0x100;
        }
        R[8] = nseg;
    }
    if (tiles == 0) { *out = p; return GPRB_OK; }

    const size_t pbytes = (size_t)tiles * p->ncomp * p->ks * 32 * sizeof(double);
#define PK_CUDA(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { gprb_set_error("%s:%d CUDA error %s", __FILE__, __LINE__, cudaGetErrorString(_e)); gprb_pack_destroy(p); return GPRB_ERR_CUDA; } } while (0)
    PK_CUDA(cudaMallocAsync((void **)&p->P, pbytes, st));
    PK_CUDA(cudaMallocAsync((void **)&p->norm, (size_t)n_padded * sizeof(double), st));
    PK_CUDA(cudaMallocAsync((void **)&p->elep, (size_t)n_padded * sizeof(int), st));
    PK_CUDA(cudaMallocAsync((void **)&p->row_group, (size_t)n_padded * sizeof(int), st));
    PK_CUDA(cudaMallocAsync((void **)&p->row_hash, (size_t)n_padded * sizeof(uint64_t), st));
    PK_CUDA(cudaMallocAsync((void **)&p->tile_rec, rec.size() * sizeof(int), st));
    PK_CUDA(cudaMallocAsync((void **)&p->d_row_ptr, (size_t)(n_groups + 1) * sizeof(int), st));
    PK_CUDA(cudaMallocAsync((void **)&p->d_group_rows, (size_t)(n_groups > 0 ? n_groups : 1) * sizeof(int), st));
    PK_CUDA(cudaMemcpyAsync(p->row_group, rgroup.data(), (size_t)n_padded * sizeof(int), cudaMemcpyHostToDevice, st));
    PK_CUDA(cudaMemcpyAsync(p->tile_rec, rec.data(), rec.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    PK_CUDA(cudaMemcpyAsync(p->d_row_ptr, p->row_ptr.data(), (size_t)(n_groups + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
    if (n_groups > 0)
        PK_CUDA(cudaMemcpyAsync(p->d_group_rows, p->group_rows.data(), (size_t)n_groups * sizeof(int), cudaMemcpyHostToDevice, st));

    const double *dx = nullptr, *ddx = nullptr; const int *de = nullptr;
    double *ox = nullptr, *odx = nullptr; int *oe = nullptr;
    int rc;
    if ((rc = stage_input(x_any, (size_t)rows * d, &dx, &ox, st)) ||
        (rc = stage_input(dxdr_any, ncols ? (size_t)rows * d * ncols : 0, &ddx, &odx, st)) ||
        (rc = stage_input(ele_any, (size_t)rows, &de, &oe, st))) { gprb_pack_destroy(p); return rc; }
    {
        const int threads = 256, wpb = threads / 32;
        const int blocks = (n_padded + wpb - 1) / wpb;
        prep_rows_kernel<<<blocks, threads, 0, st>>>(n_padded, p->n_rows, d, ncols, p->ks, norm_eps, dx, ddx, de,
                                                     p->P, p->norm, p->elep, p->tile_rec, p->row_hash);
        GPRB_LAUNCHED();
        PK_CUDA(cudaGetLastError());
    }
    if (ox) PK_CUDA(cudaFreeAsync(ox, st));
    if (odx) PK_CUDA(cudaFreeAsync(odx, st));
    if (oe) PK_CUDA(cudaFreeAsync(oe, st));
    // the host vectors (rgroup, rec) die at return: pageable H2D copies have been staged by then,
    // but make that explicit and surface asynchronous faults of the prep kernel here.
    PK_CUDA(cudaStreamSynchronize(st));
#undef PK_CUDA
    *out = p;
    return GPRB_OK;
}

extern "C" int gprb_pack_info(const gprb_pack *p, int *n_groups, int *n_rows, int *d, int *ncols, int *n_tiles) {
    GPRB_REQUIRE(p != nullptr, "gprb_pack_info: NULL pack");
    if (n_groups) *n_groups = p->n_groups;
    if (n_rows) *n_rows = p->n_rows;
    if (d) *d = p->d;
    if (ncols) *ncols = p->ncols;
    if (n_tiles) *n_tiles = p->n_tiles;
    return GPRB_OK;
}

static int ensure_species(gprb_pack *p) {
    if (p->species_ready) return GPRB_OK;
    std::vector<int> e((size_t)p->n_tiles * GPRB_TILE_ROWS);
    if (!e.empty()) GPRB_CUDA(cudaMemcpy(e.data(), p->elep, e.size() * sizeof(int), cudaMemcpyDeviceToHost));
    p->species.assign(p->n_groups, {});
    for (int g = 0; g < p->n_groups; g++)
        for (int r = p->row_ptr[g]; r < p->row_ptr[g + 1]; r++)
            if (e[r] >= 0) p->species[g][e[r]]++;
    p->species_ready = true;
    return GPRB_OK;
}

extern "C" long long gprb_pack_pair_count(const gprb_pack *a_, int g0, int g1, const gprb_pack *b_) {
    gprb_pack *a = const_cast<gprb_pack *>(a_), *b = const_cast<gprb_pack *>(b_);
    if (!a || !b || ensure_species(a) || ensure_species(b)) return -1;
    std::map<int, long long> tot;
    for (auto &m : b->species) for (auto &kv : m) tot[kv.first] += kv.second;
    long long pairs = 0;
    if (g0 < 0) g0 = 0;
    if (g1 > a->n_groups) g1 = a->n_groups;
    for (int g = g0; g < g1; g++)
        for (auto &kv : a->species[g]) { auto it = tot.find(kv.first); if (it != tot.end()) pairs += kv.second * it->second; }
    return pairs;
}
