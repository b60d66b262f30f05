/*
 * CPU oracle of the float Hamming distance of real-valued codes (TEST INFRASTRUCTURE — see oracle/__init__.py).
 * Never linked into, or called from, the product library.
 *
 *  oracle_real_hamming_dist <- /root/reference/main/engine/accuracy_calculator.py:183-186
 *                              (calc_hamming_dist = 0.5 * (B - q @ r.T) in float32) for codes that are not +-1
 *                              (raw logits, sign(0) = 0, +-inf, NaN), in the summation order of the device scorer
 *                              (b200_real_hamming_dist): s = one fmaf chain over d = 0 .. D-1 from +0.0f, then
 *                              out = 0.5f * ((float)nbits - s).
 *
 * Build: oracle/real_codes.py (gcc -O3 -march=x86-64-v3 -ffp-contract=off -fopenmp -shared -fPIC): with contraction
 * off nothing but the explicit fmaf is fused, and fmaf is the correctly rounded instruction.
 */
#include <math.h>
#include <stddef.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* q [Q,D], r [N,D] float32 -> out [Q,N] float32. */
int oracle_real_hamming_dist(const float *q, const float *r, int Q, long N, int D, int nbits, float *out, int nthreads) {
    if (Q < 0 || N < 0 || D < 1 || nbits < 1) return -1;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(dynamic, 4)
    for (int i = 0; i < Q; ++i) {
        const float *qi = q + (size_t)i * D;
        for (long j = 0; j < N; ++j) {
            const float *rj = r + (size_t)j * D;
            float s = 0.f;
            for (int d = 0; d < D; ++d) s = fmaf(qi[d], rj[d], s);
            out[(size_t)i * N + j] = 0.5f * ((float)nbits - s);
        }
    }
    return 0;
}
