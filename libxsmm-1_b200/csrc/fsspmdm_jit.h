// Baking a fixed sparse operator into a specialised sm_100a kernel at create time -- the GPU
// counterpart of the reference's x86 JIT (src/generator_spgemm_csr_asparse_reg.c:196-300): A's
// values become immediates, A's column indices become register names, B's rows live in registers.
#pragma once
#include <cuda_runtime.h>

namespace xb {
struct FsJit;
// returns NULL when the operator is outside what the baked kernel supports (the caller then uses the
// generic kernel) or when NVRTC is not available (reported through set_error).
FsJit* fs_jit_build(int is_double, int vec2, int M, int K, int beta_one, int skip_empty_rows,
                    const int* rowptr, const int* col, const double* val, int batched = 0, int variant = 0);
// number of emitter variants worth timing at create (1: only variant 0, the plain form)
int fs_jit_variants(int is_double, int vec2, int M, int K, const int* rowptr, const int* col);
// batched form: thread n -> item n / cols_per_item (element item / items_per_elem, item-in-element item % items_per_elem), column
// n % cols_per_item; B / C of an item start at slot * stride + item-in-element * item stride, the slot being the element or, for a
// non-NULL index (DEVICE array), index[element]; an element with a slot at or past its slot count is skipped
bool fs_jit_launch_batched(const FsJit* j, const void* dB, void* dC, long long n_elem, long long items_per_elem, long long cols_per_item, long long ldb, long long ldc,
                           long long stride_b, long long stride_c, long long item_b, long long item_c,
                           const unsigned int* b_index, long long b_slots, const unsigned int* c_index, long long c_slots, cudaStream_t stream);
bool fs_jit_launch(const FsJit* j, const void* dB, void* dC, long long ncols, long long ldb, long long ldc, cudaStream_t stream);
void fs_jit_destroy(FsJit* j);
// 0: outside what can be baked (generic kernel), 1: B rows in registers, 2: B strip staged in shared memory by TMA
int fs_jit_form(int is_double, int vec2, int M, int K, const int* rowptr, const int* col);
// the CUDA source that would be compiled (for tests / inspection); caller frees with free()
char* fs_jit_source(int is_double, int vec2, int M, int K, int beta_one, int skip_empty_rows,
                    const int* rowptr, const int* col, const double* val);
}  // namespace xb
