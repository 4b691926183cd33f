// K4 -- fused output head: (ensemble mean ->) (RPL4 ->) minus log-prior -> log-softmax.
//
// Reference semantics:
//   y - logsum(y, axis=1)                       predict_folds.py:57,88 with kw_utils.py:38-43
//   y = y - ap ; y = y - logsum(y, axis=1)      evaluateModelForTest.py:75-77,110-112 (ap = ap_coef * log_ap)
//   NNWithRPL.__call__ logit averaging          evaluate.py:35-51
//   RPL4.__call__                               RPL.py:68-74
//   dev-mode mean of fold log-softmax outputs   predict_folds.py:199-219
//
// HBM-bound: one warp owns one row, the whole row lives in registers (C <= 2048), reductions are warp
// shuffles, so every logit is read once and every output written once: (n_inputs + 1) * C * 4 B per frame.
#include <math_constants.h>

#include "ptx.cuh"
#include "nnam_internal.h"

namespace nnam {

constexpr int HEAD_MAX_INPUTS = 16;
constexpr int HEAD_THREADS = 256;

struct HeadParams {
  const float* in[HEAD_MAX_INPUTS];
  float w[HEAD_MAX_INPUTS];
  int n_inputs;
  long long ld_in;
  int pre_normalize;
  const float* rpl_w;
  const float* rpl_b;
  const float* rpl_lb;
  const float* prior;
  float prior_scale;
  int final_normalize;
  float* out;
  long long ld_out;
  long long rows;
  int n_classes;
  const int* out_row_map;  // optional scatter: logits row r -> out row map[r] (negative: drop)
  // compact transfer format (nnam_head_f16): out16[r][c] = fp16(y[r][c] - row_ref[r]) with row_ref[r] = max_c y[r][c];
  // `out` is unused then.  The largest entries of a row -- the ones a decoder compares -- keep ~fp32 resolution (their
  // offsets from the maximum are tiny), the far tail keeps 11 significant bits of its distance from the maximum.
  uint16_t* out16;
  long long ld16;
  float* row_ref;
  // scoring output (nnam_head_score): per output row q, nll[q] = -y[q][targets[q]] (0 when targets[q] < 0) and
  // pred[q] = argmax_c y[q][c] (lowest column on ties); a zero-fill entry -2 - q gives nll[q] = 0, pred[q] = -1.
  // `out` and `out16` are unused then: a row costs 8 B of output instead of 4 * C.
  const int* targets;
  float* nll;
  int* pred;
};

__device__ __forceinline__ uint32_t head_pack_f16x2(float lo, float hi) { return pack_f16x2(lo, hi); }

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// (value, column) of the row maximum, lowest column on ties, across the warp; every lane gets the result
__device__ __forceinline__ void warp_argmax(float& best, int& col) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oc = __shfl_xor_sync(0xffffffffu, col, o);
    if (ov > best || (ov == best && oc < col)) {
      best = ov;
      col = oc;
    }
  }
}

// Scoring epilogue of one row (one warp): `best` / `col` are this lane's running maximum over its columns (visited in
// increasing order, strict > so the lowest column wins), `vt` the written value of column t if this lane holds it
// (lane t_lane does).
__device__ __forceinline__ void score_row(const HeadParams& p, long long q, bool zero, int t, int t_lane, float best,
                                          int col, float vt, int lane) {
  warp_argmax(best, col);
  vt = __shfl_sync(0xffffffffu, vt, t_lane & 31);
  if (lane == 0) {
    p.nll[q] = (zero || t < 0) ? 0.0f : -vt;
    p.pred[q] = zero ? -1 : col;
  }
}

// log(sum(exp(v))) over the row held as v[i] <-> column lane + 32*i (invalid columns are skipped)
template <int NV>
__device__ __forceinline__ float row_logsumexp(const float (&v)[NV], int lane, int n_classes) {
  float mx = -CUDART_INF_F;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (lane + 32 * i < n_classes) mx = fmaxf(mx, v[i]);
  mx = warp_max(mx);
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (lane + 32 * i < n_classes) s += expf(v[i] - mx);
  s = warp_sum(s);
  return mx + logf(s);
}

template <int NV, bool MULTI, bool SCORE>
__global__ void __launch_bounds__(HEAD_THREADS, (MULTI || NV < 64) ? 1 : 2) head_kernel(const HeadParams p) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = (static_cast<long long>(blockIdx.x) * HEAD_THREADS + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * HEAD_THREADS) >> 5;
  const int C = p.n_classes;
  for (long long row = warp_global; row < p.rows; row += n_warps) {
    float h[NV];
    if (!MULTI) {  // one input, no per-input normalisation: the common predict()/evaluate path
      const float* src = p.in[0] + row * p.ld_in;
      const float w0 = p.w[0];
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        h[i] = c < C ? __ldg(src + c) * w0 : 0.0f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) h[i] = 0.0f;
      for (int k = 0; k < p.n_inputs; ++k) {
        const float* src = p.in[k] + row * p.ld_in;
        float t[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = lane + 32 * i;
          t[i] = c < C ? __ldg(src + c) : 0.0f;
        }
        const float lse = p.pre_normalize ? row_logsumexp<NV>(t, lane, C) : 0.0f;
        const float wk = p.w[k];
#pragma unroll
        for (int i = 0; i < NV; ++i) h[i] += wk * (t[i] - lse);
      }
    }
    if (p.rpl_w != nullptr) {
      const float lse = row_logsumexp<NV>(h, lane, C);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < C) {
          const float x = h[i] - lse;
          const float g = x + x * __ldg(p.rpl_w + c) + __ldg(p.rpl_b + c);
          const float lb = __ldg(p.rpl_lb + c);
          const float mx = fmaxf(g, lb), mn = fminf(g, lb);
          h[i] = mx + logf(1.0f + expf(mn - mx));
        }
      }
    }
    if (p.prior != nullptr) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < C) h[i] -= p.prior_scale * __ldg(p.prior + c);
      }
    }
    const float lse = p.final_normalize ? row_logsumexp<NV>(h, lane, C) : 0.0f;
    long long out_row = row;
    bool zero = false;
    if (p.out_row_map != nullptr) {
      out_row = __ldg(p.out_row_map + row);
      if (out_row == -1) continue;  // warp-uniform: one row per warp
      if (out_row < 0) {            // -2 - r: fill output row r with zeros (quirk Q4 rows the reference never writes)
        out_row = -2 - out_row;
        zero = true;
      }
    }
    if constexpr (SCORE) {
      // the values the float32 path below writes, h[i] - lse
      const int t = zero ? -1 : __ldg(p.targets + out_row);
      float best = -CUDART_INF_F, vt = 0.0f;
      int col = 0x7fffffff;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < C) {
          const float y = h[i] - lse;
          if (y > best || col == 0x7fffffff) {
            best = y;
            col = c;
          }
          if (c == t) vt = y;
        }
      }
      score_row(p, out_row, zero, t, t, best, col, vt, lane);
      continue;
    }
    if (p.out16 != nullptr) {
      float mx = -CUDART_INF_F;
#pragma unroll
      for (int i = 0; i < NV; ++i)
        if (lane + 32 * i < C) mx = fmaxf(mx, h[i]);
      mx = zero ? 0.0f : warp_max(mx);
      uint16_t* d16 = p.out16 + out_row * p.ld16;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < C) d16[c] = static_cast<uint16_t>(head_pack_f16x2(zero ? 0.0f : h[i] - mx, 0.0f) & 0xffffu);
      }
      if (lane == 0) p.row_ref[out_row] = zero ? 0.0f : mx - lse;
      continue;
    }
    float* dst = p.out + out_row * p.ld_out;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < C) dst[c] = zero ? 0.0f : h[i] - lse;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Fast path for the common case: ONE input, optional prior, optional scatter map (predict() and the evaluate path of a
// single net).  The first ncu pass of the generic kernel (profiles/r01_cfg2_gemm_before.md) showed ~2100 warp
// instructions per row -- per-element predicates, 4-byte loads and stores -- i.e. issue-bound at 40 % of the DRAM
// roofline.  Here a lane owns whole 16-byte chunks: chunk k = lane + 32 i holds columns 4k .. 4k+3.
//   * loads are 128-bit and unpredicated for every chunk that lies inside the row (only the last i is checked);
//   * exp is ex2.approx of a pre-scaled argument (one FFMA + one MUFU per element);
//   * the output matrix is (rows, C) with C = 1909: a row starts at an address that is only 4-byte aligned, so the
//     lanes RE-ALIGN the row with shuffles (each takes the last `a` elements of its left neighbour's chunk, where
//     a = (row start / 4) mod 4) and store 16-byte aligned chunks; only the row's ragged ends are scalar stores.
constexpr int HEAD_FAST_THREADS = 128;

template <int NV4, bool SCORE>
__global__ void __launch_bounds__(HEAD_FAST_THREADS, 4) head_fast_kernel(const HeadParams p) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = (static_cast<long long>(blockIdx.x) * HEAD_FAST_THREADS + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * HEAD_FAST_THREADS) >> 5;
  const int C = p.n_classes;
  const int n_full = C >> 7;  // iterations whose 32 chunks all lie inside the row
  const float w0 = p.w[0];
  constexpr float LOG2E = 1.4426950408889634f;
  for (long long row = warp_global; row < p.rows; row += n_warps) {
    const float4* src = reinterpret_cast<const float4*>(p.in[0] + row * p.ld_in);
    float4 v[NV4];
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int k = lane + 32 * i;
      if (i < n_full) {
        v[i] = __ldcs(src + k);
      } else {
        // ragged end of the row: the buffer is only guaranteed to hold ld_in >= C floats per row
        const float* s1 = reinterpret_cast<const float*>(src) + 4 * k;
        v[i].x = 4 * k < C ? __ldcs(s1) : 0.0f;
        v[i].y = 4 * k + 1 < C ? __ldcs(s1 + 1) : 0.0f;
        v[i].z = 4 * k + 2 < C ? __ldcs(s1 + 2) : 0.0f;
        v[i].w = 4 * k + 3 < C ? __ldcs(s1 + 3) : 0.0f;
      }
    }
    if (w0 != 1.0f) {
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        v[i].x *= w0; v[i].y *= w0; v[i].z *= w0; v[i].w *= w0;
      }
    }
    if (p.prior != nullptr) {
      const float ps = p.prior_scale;
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int k = lane + 32 * i;
        if (i < n_full) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(p.prior) + k);
          v[i].x -= ps * a.x; v[i].y -= ps * a.y; v[i].z -= ps * a.z; v[i].w -= ps * a.w;
        } else {
          if (4 * k < C) v[i].x -= ps * __ldg(p.prior + 4 * k);
          if (4 * k + 1 < C) v[i].y -= ps * __ldg(p.prior + 4 * k + 1);
          if (4 * k + 2 < C) v[i].z -= ps * __ldg(p.prior + 4 * k + 2);
          if (4 * k + 3 < C) v[i].w -= ps * __ldg(p.prior + 4 * k + 3);
        }
      }
    }
    float lse = 0.0f, mx = 0.0f;
    if (p.final_normalize || p.out16 != nullptr) {
      // columns past the end of the row become -inf: neutral for the max, and exp2 maps them to 0
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        if (i < n_full) continue;
        const int k = lane + 32 * i;
        if (4 * k >= C) v[i].x = -CUDART_INF_F;
        if (4 * k + 1 >= C) v[i].y = -CUDART_INF_F;
        if (4 * k + 2 >= C) v[i].z = -CUDART_INF_F;
        if (4 * k + 3 >= C) v[i].w = -CUDART_INF_F;
      }
      mx = -CUDART_INF_F;
#pragma unroll
      for (int i = 0; i < NV4; ++i) mx = fmaxf(fmaxf(mx, fmaxf(v[i].x, v[i].y)), fmaxf(v[i].z, v[i].w));
      mx = warp_max(mx);
    }
    if (p.final_normalize) {
      const float mxs = mx * LOG2E;
      float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        s0 += exp2f(fmaf(v[i].x, LOG2E, -mxs)) + exp2f(fmaf(v[i].y, LOG2E, -mxs));
        s1 += exp2f(fmaf(v[i].z, LOG2E, -mxs)) + exp2f(fmaf(v[i].w, LOG2E, -mxs));
      }
      lse = mx + logf(warp_sum(s0 + s1));
    }
    long long out_row = row;
    bool zero = false;
    if (p.out_row_map != nullptr) {
      out_row = __ldg(p.out_row_map + row);
      if (out_row == -1) continue;  // warp-uniform: one row per warp
      if (out_row < 0) {            // -2 - r: fill output row r with zeros (quirk Q4 rows the reference never writes)
        out_row = -2 - out_row;
        zero = true;
        lse = 0.0f;
        mx = 0.0f;
#pragma unroll
        for (int i = 0; i < NV4; ++i) v[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      }
    }
    if constexpr (SCORE) {
      // the values the float32 path below writes, v - lse; a lane's columns 4k .. 4k+3 (k = lane + 32 i) increase with i
      const int t = zero ? -1 : __ldg(p.targets + out_row);
      float best = -CUDART_INF_F, vt = 0.0f;
      int col = 0x7fffffff;
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int c0 = 4 * (lane + 32 * i);
        const float y[4] = {v[i].x - lse, v[i].y - lse, v[i].z - lse, v[i].w - lse};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (c0 + e < C) {
            if (y[e] > best || col == 0x7fffffff) {
              best = y[e];
              col = c0 + e;
            }
            if (c0 + e == t) vt = y[e];
          }
        }
      }
      score_row(p, out_row, zero, t, t >> 2, best, col, vt, lane);  // column t sits in lane (t / 4) % 32
      continue;
    }
    if (p.out16 != nullptr) {
      // rows of the fp16 matrix are 16-byte aligned (ld16 % 8 == 0): a lane's chunk k is one 8-byte store
      uint2* d2 = reinterpret_cast<uint2*>(p.out16 + out_row * p.ld16);
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int k = lane + 32 * i;
        if (4 * k < p.ld16)  // columns in [C, ld16) are written as fp16(-inf - mx) or 0; the host never reads them
          __stcs(d2 + k, make_uint2(head_pack_f16x2(v[i].x - mx, v[i].y - mx), head_pack_f16x2(v[i].z - mx, v[i].w - mx)));
      }
      if (lane == 0) p.row_ref[out_row] = mx - lse;
      continue;
    }
    float* dst = p.out + out_row * p.ld_out;
    const int a = static_cast<int>((reinterpret_cast<uintptr_t>(dst) >> 2) & 3);  // row start modulo 16 bytes, in floats
    float4* dst4 = reinterpret_cast<float4*>(dst - a);                              // aligned chunk 0 of the row
    float c1 = 0.0f, c2 = 0.0f, c3 = 0.0f;  // last elements of lane 31's previous chunk (for lane 0)
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int k = lane + 32 * i;
      float4 x = v[i];
      x.x -= lse; x.y -= lse; x.z -= lse; x.w -= lse;
      // y = aligned chunk k of the output row = columns 4k-a .. 4k-a+3
      float p1 = __shfl_up_sync(0xffffffffu, x.y, 1), p2 = __shfl_up_sync(0xffffffffu, x.z, 1),
            p3 = __shfl_up_sync(0xffffffffu, x.w, 1);
      if (lane == 0) { p1 = c1; p2 = c2; p3 = c3; }
      c1 = __shfl_sync(0xffffffffu, x.y, 31);
      c2 = __shfl_sync(0xffffffffu, x.z, 31);
      c3 = __shfl_sync(0xffffffffu, x.w, 31);
      float4 y;
      if (a == 0) y = x;
      else if (a == 1) y = make_float4(p3, x.x, x.y, x.z);
      else if (a == 2) y = make_float4(p2, p3, x.x, x.y);
      else y = make_float4(p1, p2, p3, x.x);
      const int col0 = 4 * k - a;
      if (col0 >= 0 && col0 + 3 < C) {
        __stcs(dst4 + k, y);
      } else {  // ragged ends of the row
        if (col0 >= 0 && col0 < C) __stcs(dst + col0, y.x);
        if (col0 + 1 >= 0 && col0 + 1 < C) __stcs(dst + col0 + 1, y.y);
        if (col0 + 2 >= 0 && col0 + 2 < C) __stcs(dst + col0 + 2, y.z);
        if (col0 + 3 >= 0 && col0 + 3 < C) __stcs(dst + col0 + 3, y.w);
      }
    }
    // the last `a` elements of chunk 32*NV4-1 would belong to aligned chunk 32*NV4: they exist only when C > 128*NV4 - a,
    // which the host excludes by choosing NV4 with 128*NV4 >= C + 3
  }
}

int head(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in, int pre_normalize,
         const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior, float prior_scale,
         int final_normalize, float* out, long long ld_out, long long rows, int n_classes, const int* out_row_map,
         void* out16, long long ld16, float* row_ref, const int* targets, float* nll, int* pred, cudaStream_t stream) {
  const bool score = nll != nullptr;
  if (n_inputs < 1 || n_inputs > HEAD_MAX_INPUTS)
    return set_error(NNAM_ERR_ARG, "head: n_inputs must be in [1, %d]", HEAD_MAX_INPUTS);
  if (n_classes < 1 || n_classes > 2048) return set_error(NNAM_ERR_UNSUPPORTED, "head: n_classes must be in [1, 2048]");
  if (ld_in < n_classes || (out16 == nullptr && !score && ld_out < n_classes))
    return set_error(NNAM_ERR_ARG, "head: leading dimension < n_classes");
  if (out16 != nullptr && (row_ref == nullptr || ld16 < n_classes || ld16 % 8 || (reinterpret_cast<uintptr_t>(out16) & 15)))
    return set_error(NNAM_ERR_ARG, "head: the fp16 output needs row_ref, ld16 >= n_classes, ld16 %% 8 == 0 and a "
                     "16-byte aligned buffer");
  if (score && (targets == nullptr || pred == nullptr || out != nullptr || out16 != nullptr))
    return set_error(NNAM_ERR_ARG, "head: scoring needs targets, nll and pred, and no row output");
  if (out16 == nullptr && out == nullptr && !score) return set_error(NNAM_ERR_ARG, "head: no output buffer");
  if (rows < 0) return set_error(NNAM_ERR_ARG, "head: negative row count");
  if (rows == 0) return NNAM_OK;
  if ((rpl_w != nullptr) != (rpl_b != nullptr) || (rpl_w != nullptr) != (rpl_lb != nullptr))
    return set_error(NNAM_ERR_ARG, "head: RPL4 needs W, b and lb together");
  HeadParams p;
  for (int k = 0; k < n_inputs; ++k) {
    if (logits_host[k] == nullptr) return set_error(NNAM_ERR_ARG, "head: logits[%d] is NULL", k);
    p.in[k] = logits_host[k];
    p.w[k] = weights_host ? weights_host[k] : 1.0f / n_inputs;
  }
  p.n_inputs = n_inputs;
  p.ld_in = ld_in;
  p.pre_normalize = pre_normalize;
  p.rpl_w = rpl_w;
  p.rpl_b = rpl_b;
  p.rpl_lb = rpl_lb;
  p.prior = prior;
  p.prior_scale = prior_scale;
  p.final_normalize = final_normalize;
  p.out = out;
  p.ld_out = ld_out;
  p.rows = rows;
  p.n_classes = n_classes;
  p.out_row_map = out_row_map;
  p.out16 = static_cast<uint16_t*>(out16);
  p.ld16 = ld16;
  p.row_ref = row_ref;
  p.targets = targets;
  p.nll = nll;
  p.pred = pred;
  // fast path: one input, no RPL4 / per-input normalisation, 16-byte aligned input rows
  const bool fast_ok = n_inputs == 1 && !pre_normalize && rpl_w == nullptr && ld_in % 4 == 0 &&
                       (reinterpret_cast<uintptr_t>(logits_host[0]) & 15) == 0 &&
                       (prior == nullptr || (reinterpret_cast<uintptr_t>(prior) & 15) == 0) &&
                       (reinterpret_cast<uintptr_t>(out) & 3) == 0 && n_classes + 3 <= 2048 &&
                       (out16 == nullptr || ld16 <= 2048);
  if (fast_ok) {
    const int wpb = HEAD_FAST_THREADS / 32;
    long long fb = (rows + wpb - 1) / wpb;
    const long long fcap = static_cast<long long>(sm_count()) * 16;
    if (fb > fcap) fb = fcap;
    const unsigned fg = static_cast<unsigned>(fb);
    const int need = n_classes + 3;  // see the kernel's closing comment
#define NNAM_HEAD_FAST_LAUNCH(NV4)                                        \
  do {                                                                    \
    if (score)                                                            \
      head_fast_kernel<NV4, true><<<fg, HEAD_FAST_THREADS, 0, stream>>>(p);  \
    else                                                                  \
      head_fast_kernel<NV4, false><<<fg, HEAD_FAST_THREADS, 0, stream>>>(p); \
  } while (0)
    if (need <= 128) NNAM_HEAD_FAST_LAUNCH(1);
    else if (need <= 512) NNAM_HEAD_FAST_LAUNCH(4);
    else if (need <= 1024) NNAM_HEAD_FAST_LAUNCH(8);
    else if (need <= 1920) NNAM_HEAD_FAST_LAUNCH(15);
    else NNAM_HEAD_FAST_LAUNCH(16);
#undef NNAM_HEAD_FAST_LAUNCH
    return check_launch("head_fast_kernel");
  }
  const int warps_per_block = HEAD_THREADS / 32;
  long long blocks = (rows + warps_per_block - 1) / warps_per_block;
  const long long cap = static_cast<long long>(sm_count()) * 8;  // grid-stride beyond 8 resident blocks per SM
  if (blocks > cap) blocks = cap;
  const bool multi = n_inputs > 1 || pre_normalize;
  const unsigned g = static_cast<unsigned>(blocks);
#define NNAM_HEAD_LAUNCH(NV)                                              \
  do {                                                                    \
    if (score && multi)                                                   \
      head_kernel<NV, true, true><<<g, HEAD_THREADS, 0, stream>>>(p);     \
    else if (score)                                                       \
      head_kernel<NV, false, true><<<g, HEAD_THREADS, 0, stream>>>(p);    \
    else if (multi)                                                       \
      head_kernel<NV, true, false><<<g, HEAD_THREADS, 0, stream>>>(p);    \
    else                                                                  \
      head_kernel<NV, false, false><<<g, HEAD_THREADS, 0, stream>>>(p);   \
  } while (0)
  if (n_classes <= 128)
    NNAM_HEAD_LAUNCH(4);
  else if (n_classes <= 1024)
    NNAM_HEAD_LAUNCH(32);
  else
    NNAM_HEAD_LAUNCH(64);
#undef NNAM_HEAD_LAUNCH
  return check_launch("head_kernel");
}

}  // namespace nnam
