/*
 * TEST INFRASTRUCTURE ONLY: CPU restatement of the dense x SoA kernels, libxsmm_create_rm_ac_soa / libxsmm_create_rm_bc_soa
 * (reference src/libxsmm_main.c:2477,2500).  tests/test_rm_soa.py compiles it with -ffp-contract=off into a temporary directory:
 * every fused multiply-add here is an explicit fma() / fmaf().
 *
 * form 0 (ac): A [M][lda][soa], b K x N with pitch ldb, C [M][ldc][soa]:  C[m][n][s] = chain over k ascending of acc = fma(A[m][k][s], b[k][n], acc).
 * form 1 (bc): a M x K with pitch lda, B [K][ldb][soa]:                    C[m][n][s] = chain over k ascending of acc = fma(a[m][k], B[k][n][s], acc).
 * acc starts from C (beta = 1) or +0 (beta = 0, C not read); zeros are not skipped; only columns 0 .. N-1 are written.  The
 * generator source is not restated here: this is the arithmetic of a dense register-blocked kernel that zeroes or loads its
 * accumulators and issues one fused multiply-add per k.  n_elem elements, element strides in scalars (0: shared operand).
 */
#include <math.h>
#include <stddef.h>

void orc_rm_soa_execute(int dbl, int form, int M, int N, int K, int lda, int ldb, int ldc, int soa, double beta,
                        const void* a, const void* b, void* c, long n_elem, long stride_a, long stride_b, long stride_c)
{
  long e; int m, n, s, k;
  for (e = 0; e < n_elem; ++e) for (m = 0; m < M; ++m) for (n = 0; n < N; ++n) for (s = 0; s < soa; ++s) {
    const size_t cat = (size_t)e * stride_c + ((size_t)m * ldc + n) * soa + s;
    const size_t ea = (size_t)e * stride_a, eb = (size_t)e * stride_b;
    if (dbl) {
      const double* A = (const double*)a; const double* B = (const double*)b;
      double acc = (0.0 == beta) ? 0.0 : ((double*)c)[cat];
      for (k = 0; k < K; ++k) {
        if (0 == form) acc = fma(A[ea + ((size_t)m * lda + k) * soa + s], B[eb + (size_t)k * ldb + n], acc);
        else acc = fma(A[ea + (size_t)m * lda + k], B[eb + ((size_t)k * ldb + n) * soa + s], acc);
      }
      ((double*)c)[cat] = acc;
    }
    else {
      const float* A = (const float*)a; const float* B = (const float*)b;
      float acc = (0.0 == beta) ? 0.f : ((float*)c)[cat];
      for (k = 0; k < K; ++k) {
        if (0 == form) acc = fmaf(A[ea + ((size_t)m * lda + k) * soa + s], B[eb + (size_t)k * ldb + n], acc);
        else acc = fmaf(A[ea + (size_t)m * lda + k], B[eb + ((size_t)k * ldb + n) * soa + s], acc);
      }
      ((float*)c)[cat] = acc;
    }
  }
}
