// C ABI (include/nnam_b200.h): argument plumbing, error state, TMA descriptor encoding.
#include <stdarg.h>
#include <stdio.h>

#include <cudaTypedefs.h>

#include "nnam_internal.h"

namespace nnam {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int set_cuda_error(cudaError_t e, const char* what) {
  return set_error(NNAM_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}

int check_launch(const char* kernel_name) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, kernel_name);
  return NNAM_OK;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 1;
  if (dev >= 0 && dev < 64 && cached[dev] > 0) return cached[dev];
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 1;
  if (dev >= 0 && dev < 64) cached[dev] = n;
  return n;
}

// cuTensorMapEncodeTiled is a driver-API symbol; resolve it through the runtime so that the library
// has no link-time dependency on libcuda.so (the build container has no driver).
static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || p == nullptr) return nullptr;
  fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  return fn;
}

int encode_tmap_2d(CUtensorMap* m, const void* ptr, bool f32, unsigned long long inner, unsigned long long rows,
                   unsigned long long ld_elems, unsigned box_inner, unsigned box_rows) {
  auto fn = get_encode_fn();
  if (!fn) return set_error(NNAM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {ld_elems * (f32 ? 4ull : 2ull)};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(NNAM_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) inner=%llu rows=%llu ld=%llu box=%ux%u",
                     static_cast<int>(r), inner, rows, ld_elems, box_inner, box_rows);
  return NNAM_OK;
}

int encode_tmap_bf16_2d(CUtensorMap* m, const void* ptr, unsigned long long inner, unsigned long long rows,
                        unsigned long long ld_elems, unsigned box_inner, unsigned box_rows) {
  return encode_tmap_2d(m, ptr, false, inner, rows, ld_elems, box_inner, box_rows);
}

int splice_transform(const float* x, long long x_row0, long long x_rows, long long n_total, int dim, int splice,
                     const float* add_shift, const float* rescale, const float* ivec, int ivec_dim, long long f0,
                     long long f1, void* out_hi, void* out_lo, long long ldo, int out_kind, cudaStream_t stream);
int convert_f32(const float* src, long long rows, int cols, long long lds, void* dst_hi, void* dst_lo, long long ldd,
                int out_kind, cudaStream_t stream);
int head(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in, int pre_normalize,
         const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior, float prior_scale,
         int final_normalize, float* out, long long ld_out, long long rows, int n_classes, const int* out_row_map,
         void* out16, long long ld16, float* row_ref, const int* targets, float* nll, int* pred, cudaStream_t stream);
int gather_transform(const float* x, long long n_src, int dim, const float* add_shift, const float* rescale,
                     const float* ivec, int ivec_dim, const int* row_map, long long n_rows, void* out_hi, void* out_lo,
                     long long ldo, int out_kind, cudaStream_t stream);
int peephole_cell(int phase, const float* gx, long long gx_ld, const float* g1, long long g1_ld, const float* p2,
                  long long p2_ld, const float* c_prev, float* c_new, void* out_hi, void* out_lo, long long out_ld, int n,
                  int H, int fast, int elem, cudaStream_t stream);
int rnn_seq(const NnamRnnDesc* d, cudaStream_t stream);
int rnn_solo_step_cycles(int cell, int hidden, int batch, int nsplit, int* cycles);
int rnn_plan(int cell, int hidden, int batch, int nsplit, int* group_ctas, int* max_groups, int* step_cycles,
             int* streams);

}  // namespace nnam

extern "C" {

int nnam_abi_version(void) { return NNAM_ABI_VERSION; }
const char* nnam_last_error(void) { return nnam::g_err; }
int nnam_sm_count(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return nnam::set_cuda_error(e, "nnam_sm_count");
  return nnam::sm_count();
}

int nnam_splice_transform(const float* x, long long x_row0, long long x_rows, long long n_total, int dim, int splice,
                          const float* add_shift, const float* rescale, const float* ivec, int ivec_dim,
                          long long f0, long long f1, void* out_hi, void* out_lo, long long ldo, int out_kind,
                          void* stream) {
  return nnam::splice_transform(x, x_row0, x_rows, n_total, dim, splice, add_shift, rescale, ivec, ivec_dim, f0, f1,
                                out_hi, out_lo, ldo, out_kind, static_cast<cudaStream_t>(stream));
}

int nnam_convert_f32(const float* src, long long rows, int cols, long long lds, void* dst_hi, void* dst_lo,
                     long long ldd, int out_kind, void* stream) {
  return nnam::convert_f32(src, rows, cols, lds, dst_hi, dst_lo, ldd, out_kind, static_cast<cudaStream_t>(stream));
}

int nnam_linear_bias_act(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                         long long ldw, const float* bias, void* out_hi, void* out_lo, long long ldo, int M, int N,
                         int K, int act, int out_kind, int nsplit, int elem, void* stream) {
  return nnam::gemm_bias_act(a_hi, a_lo, lda, w_hi, w_lo, ldw, bias, out_hi, out_lo, ldo, M, N, K, act, out_kind,
                             nsplit, elem, static_cast<cudaStream_t>(stream));
}

int nnam_linear_logsoftmax(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                           long long ldw, const float* bias, const float* prior, float prior_scale, float* out,
                           long long ld_out, void* out16, long long ld16, float* row_ref, const int* out_row_map,
                           int M, int N, int K, int nsplit, int elem, void* stream) {
  return nnam::linear_logsoftmax(a_hi, a_lo, lda, w_hi, w_lo, ldw, bias, prior, prior_scale, out, ld_out, out16, ld16,
                                 row_ref, out_row_map, nullptr, nullptr, nullptr, M, N, K, nsplit, elem,
                                 static_cast<cudaStream_t>(stream));
}

int nnam_linear_logsoftmax_score(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                                 long long ldw, const float* bias, const float* prior, float prior_scale,
                                 const int* targets, float* nll, int* pred, const int* out_row_map, int M, int N, int K,
                                 int nsplit, int elem, void* stream) {
  if (nll == nullptr) return nnam::set_error(NNAM_ERR_ARG, "linear_logsoftmax_score: nll is NULL");
  return nnam::linear_logsoftmax(a_hi, a_lo, lda, w_hi, w_lo, ldw, bias, prior, prior_scale, nullptr, 0, nullptr, 0,
                                 nullptr, out_row_map, targets, nll, pred, M, N, K, nsplit, elem,
                                 static_cast<cudaStream_t>(stream));
}

int nnam_head(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
              int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
              float prior_scale, int final_normalize, float* out, long long ld_out, long long rows, int n_classes,
              void* stream) {
  return nnam::head(logits_host, weights_host, n_inputs, ld_in, pre_normalize, rpl_w, rpl_b, rpl_lb, prior,
                    prior_scale, final_normalize, out, ld_out, rows, n_classes, nullptr, nullptr, 0, nullptr, nullptr,
                    nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int nnam_head_scatter(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                      int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb,
                      const float* prior, float prior_scale, int final_normalize, float* out, long long ld_out,
                      long long rows, int n_classes, const int* out_row_map, void* stream) {
  return nnam::head(logits_host, weights_host, n_inputs, ld_in, pre_normalize, rpl_w, rpl_b, rpl_lb, prior,
                    prior_scale, final_normalize, out, ld_out, rows, n_classes, out_row_map, nullptr, 0, nullptr, nullptr,
                    nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int nnam_head_f16(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                  int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
                  float prior_scale, int final_normalize, void* out16, long long ld16, float* row_ref, long long rows,
                  int n_classes, const int* out_row_map, void* stream) {
  if (out16 == nullptr) return nnam::set_error(NNAM_ERR_ARG, "head_f16: out16 is NULL");
  return nnam::head(logits_host, weights_host, n_inputs, ld_in, pre_normalize, rpl_w, rpl_b, rpl_lb, prior,
                    prior_scale, final_normalize, nullptr, 0, rows, n_classes, out_row_map, out16, ld16, row_ref, nullptr,
                    nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int nnam_head_score(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                    int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
                    float prior_scale, int final_normalize, const int* targets, float* nll, int* pred, long long rows,
                    int n_classes, const int* out_row_map, void* stream) {
  if (nll == nullptr) return nnam::set_error(NNAM_ERR_ARG, "head_score: nll is NULL");
  return nnam::head(logits_host, weights_host, n_inputs, ld_in, pre_normalize, rpl_w, rpl_b, rpl_lb, prior,
                    prior_scale, final_normalize, nullptr, 0, rows, n_classes, out_row_map, nullptr, 0, nullptr,
                    targets, nll, pred, static_cast<cudaStream_t>(stream));
}

int nnam_gather_transform(const float* x, long long n_src, int dim, const float* add_shift, const float* rescale,
                          const float* ivec, int ivec_dim, const int* row_map, long long n_rows, void* out_hi,
                          void* out_lo, long long ldo, int out_kind, void* stream) {
  return nnam::gather_transform(x, n_src, dim, add_shift, rescale, ivec, ivec_dim, row_map, n_rows, out_hi, out_lo,
                                ldo, out_kind, static_cast<cudaStream_t>(stream));
}

int nnam_peephole_cell(int phase, const float* gx, long long gx_ld, const float* g1, long long g1_ld, const float* p2,
                       long long p2_ld, const float* c_prev, float* c_new, void* out_hi, void* out_lo,
                       long long out_ld, int n, int hidden, int fast_tanh, int elem, void* stream) {
  return nnam::peephole_cell(phase, gx, gx_ld, g1, g1_ld, p2, p2_ld, c_prev, c_new, out_hi, out_lo, out_ld, n, hidden,
                             fast_tanh, elem, static_cast<cudaStream_t>(stream));
}

int nnam_rnn_seq(const NnamRnnDesc* desc, void* stream) {
  return nnam::rnn_seq(desc, static_cast<cudaStream_t>(stream));
}

int nnam_rnn_desc_size(void) { return static_cast<int>(sizeof(NnamRnnDesc)); }

int nnam_rnn_plan(int cell, int hidden, int batch, int nsplit, int* group_ctas, int* max_groups, int* step_cycles,
                  int* streams) {
  if (!group_ctas || !max_groups) return nnam::set_error(NNAM_ERR_ARG, "rnn_plan: NULL output");
  return nnam::rnn_plan(cell, hidden, batch, nsplit, group_ctas, max_groups, step_cycles, streams);
}

int nnam_rnn_solo_step_cycles(int cell, int hidden, int batch, int nsplit, int* cycles) {
  if (!cycles) return nnam::set_error(NNAM_ERR_ARG, "rnn_solo_step_cycles: NULL output");
  return nnam::rnn_solo_step_cycles(cell, hidden, batch, nsplit, cycles);
}

}  // extern "C"
