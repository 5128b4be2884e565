// virial.cu — strain derivative of each atom's descriptor, the rows of a structure's total-stress group.
//
// The stress rows of predict_structure(stress=True) hold r (x) dx_c/dr_j for every (centre c, neighbour j) row of `seq`.
// The K_fe / K_ff contractions are linear in the dxdr columns of a row once x^ is fixed, and the pair cut depends on x^
// alone, so the rows of one centre may be summed before the contraction: sum_j r_cj (x) dx_c/dr_j = dx_c/d(strain).
// This kernel forms that sum; the total stress of a structure is then one force-like group with one row per atom.
//
//   out[a, k, v] = sum_{q in [seq_ptr[a], seq_ptr[a+1])} rdxdr[q, k, voigt(v)],   voigt = {xx, yy, zz, xy, xz, yz}
//
// One CTA per atom, one thread per (k, v); each thread sums its entry in increasing q, so the result does not depend on
// the launch and two calls are bitwise equal.  HBM bound: 8 * 9 * d bytes read per seq row (DESIGN.md §4).
#include "common.cuh"

namespace {

__constant__ int c_voigt[6] = {0, 4, 8, 1, 2, 5};   // flat index of (xx, yy, zz, xy, xz, yz) in a row-major 3 x 3

__global__ void __launch_bounds__(384) virial_rows_kernel(int d, const int *__restrict__ seq_ptr,
                                                          const double *__restrict__ rdxdr, double *__restrict__ out) {
    const int a = blockIdx.x;
    const int t = threadIdx.x;
    if (t >= 6 * d) return;
    const int k = t / 6, v = t - 6 * k;
    const long long q0 = seq_ptr[a], q1 = seq_ptr[a + 1];
    const double *src = rdxdr + (size_t)k * 9 + c_voigt[v];
    double acc = 0.0;
    for (long long q = q0; q < q1; q++) acc += src[(size_t)q * 9 * d];
    out[(size_t)a * 6 * d + t] = acc;
}

}  // namespace

extern "C" int gprb_virial_rows(int n_atoms, int d, const int *seq_ptr, const double *rdxdr, double *out, void *stream) {
    GPRB_REQUIRE(n_atoms >= 0, "gprb_virial_rows: n_atoms = %d < 0", n_atoms);
    GPRB_REQUIRE(d >= 1 && d <= 64, "gprb_virial_rows: descriptor length %d outside [1, 64]", d);
    if (n_atoms == 0) return GPRB_OK;
    GPRB_REQUIRE(seq_ptr && rdxdr && out, "gprb_virial_rows: NULL argument");
    virial_rows_kernel<<<n_atoms, 32 * ((6 * d + 31) / 32), 0, (cudaStream_t)stream>>>(d, seq_ptr, rdxdr, out);
    GPRB_LAUNCHED();
    GPRB_CUDA(cudaGetLastError());
    return GPRB_OK;
}
