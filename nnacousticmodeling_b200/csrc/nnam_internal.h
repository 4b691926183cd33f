// Internal helpers shared by the .cu translation units (error state, TMA descriptor encoding).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include "../../include/nnam_b200.h"

namespace nnam {

int set_error(int code, const char* fmt, ...);
int set_cuda_error(cudaError_t e, const char* what);
int check_launch(const char* kernel_name);
int sm_count();

// 2-D bf16 tensor map, SWIZZLE_128B, zero OOB fill.  inner = contiguous extent (elements), box_inner*2 B <= 128.
int encode_tmap_bf16_2d(CUtensorMap* m, const void* ptr, unsigned long long inner, unsigned long long rows,
                        unsigned long long ld_elems, unsigned box_inner, unsigned box_rows);

// Same for bf16 or fp32 elements (box_inner * element size must be <= 128 B).
int encode_tmap_2d(CUtensorMap* m, const void* ptr, bool f32, unsigned long long inner, unsigned long long rows,
                   unsigned long long ld_elems, unsigned box_inner, unsigned box_rows);

int gemm_bias_act(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                  long long ldw, const float* bias, void* out_hi, void* out_lo, long long ldo, int M, int N, int K,
                  int act, int out_kind, int nsplit, int elem, cudaStream_t stream);

int linear_logsoftmax(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                      long long ldw, const float* bias, const float* prior, float prior_scale, float* out,
                      long long ld_out, void* out16, long long ld16, float* row_ref, const int* out_row_map,
                      const int* targets, float* nll, int* pred, int M, int N, int K, int nsplit, int elem,
                      cudaStream_t stream);

}  // namespace nnam
