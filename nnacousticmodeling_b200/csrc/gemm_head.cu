// K2+K4 -- the output layer fused with the head of a single net:
//
//   out[r, :] = log_softmax( A[r, :] . W^T + bias - prior_scale * prior )          (float32 rows or compact format)
//
// Replaces, for one model without RPL, the pair  L.Linear (chainer_networks.py:21-22, 61-62 ...)  +
// `y - logsum(y, axis=1)` (predict_folds.py:57,88; kw_utils.py:38-43) / `y = y - ap; y - logsum(y)`
// (evaluateModelForTest.py:75-77,110-112).  The unfused path writes the float32 logits (7.6 KB per frame at 1909
// classes), reads them back in the head kernel and writes the result: 15 KB per frame of HBM traffic that exists only
// because the row-wise log-sum-exp spans eight 256-column GEMM tiles.  Here the CTAs that hold the column tiles of one
// 128-row block form a THREAD-BLOCK CLUSTER (one CTA per tile, <= 8):
//
//   pass 1   eight epilogue warps, two per TMEM lane quarter: a thread owns one row (a TMEM lane) of one 128-column half
//            of its CTA's accumulator tile: running max m and s = sum exp(v - m) over the half's valid columns
//   exchange (m, s) of every row goes into the shared memory of ALL CTAs of the cluster with st.async, which completes
//            transaction bytes on the receiving CTA's mbarrier -- 16 partials per row, no fences
//   pass 2   lse = M + log(sum_r s_r exp(m_r - M)); the accumulator is read from TMEM a second time, v - lse goes through
//            a swizzled shared-memory box and leaves as 128-byte row segments (the (N, 1909) float32 rows are only
//            4-byte aligned, so no TMA store), through the optional row map of the recurrent path
//
// A third instance scores the rows against targets instead of storing them (nnam_linear_logsoftmax_score): pass 2
// computes the same values but stages and stores none; each thread keeps the (max, lowest column) of its half and the
// value at the target column, the thread holding the target writes nll = -v_t, and a second st.async exchange -- on the
// staging boxes, which this instance leaves unused, and a barrier of its own -- brings every half's (max, column) of a
// row to cluster rank 0, which writes pred.  8 B per row leave the kernel instead of 4 * N.
//
// Accumulators are double-buffered in TMEM (2 x 256 columns), so the epilogue of block i -- including the exchange
// latency -- overlaps the MMAs of block i+1.  Main loop as in gemm.cu's single-CTA kernel (TMA producer warp, one
// elected MMA thread, SWIZZLE_128B operand ring).
#include <math_constants.h>

#include "ptx.cuh"
#include "nnam_internal.h"

namespace nnam {
namespace fused {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int UK = 16;
constexpr int ST = 3;
constexpr int HALF = 128;                   // columns of a tile one epilogue warp handles
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KiB
constexpr int B_STAGE_BYTES = BN * BK * 2;  // 32 KiB
constexpr int THREADS = 384;                // 4 control warps + 8 epilogue warps
constexpr int BOX_BYTES = 32 * 128;         // one epilogue warp's staging box: 32 rows x 128 B
constexpr int MAX_CLUSTER = 8;
constexpr int XCHG_BYTES = 2 * 2 * MAX_CLUSTER * BM * 8;  // [accumulator parity][source rank, half][row] (m, s)
constexpr int ROWPTR_BYTES = 8 * 32 * 8;               // per epilogue warp: output address of each of its 32 rows
constexpr int SMEM_BYTES = ST * (A_STAGE_BYTES + B_STAGE_BYTES) + 8 * BOX_BYTES + BN * 4 + XCHG_BYTES + ROWPTR_BYTES + 256;
static_assert(SMEM_BYTES <= 227 * 1024, "fused output kernel: shared memory over budget");
static_assert(XCHG_BYTES <= 8 * BOX_BYTES, "scoring instance: the argmax exchange lives in the staging boxes");
// what pass 2 produces: float32 rows, the compact transfer format, or (nll, pred) against targets
constexpr int OUT_ROWS = 0, OUT_COMPACT = 1, OUT_SCORE = 2;
constexpr int TMEM_COLS = 512;
constexpr float NEG_BIG = -3.0e38f;  // finite stand-in for -inf as the running maximum's start value
constexpr float LOG2E = 1.4426950408889634f;

struct Params {
  int M, N, K;
  int tiles_m, k_blocks, nsplit, passes, f16;
  int cluster;  // CTAs per cluster = 256-column tiles covering N
  const float* bias;
  const float* prior;
  float prior_scale;
  // The scoring instance stores no rows: its outputs and targets (indexed by output row) share the row outputs' slots,
  // which keeps the kernel parameters -- and the register allocation of the other two instances -- as they were.
  union {
    float* out;  // float32 rows
    float* nll;
  };
  long long ld_out;
  union {
    uint16_t* out16;  // compact format (nnam_head_f16): fp16 offsets from the row maximum + row_ref
    int* pred;
  };
  long long ld16;
  union {
    float* row_ref;
    const int* targets;
  };
  const int* out_row_map;
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 8-byte store into a peer CTA's shared memory that completes 8 transaction bytes on an mbarrier of THAT CTA when it
// lands: data and signal travel together, so the sender needs no release fence.  (A fence.acq_rel.cluster or an
// mbarrier.arrive.release.cluster here compiles to MEMBAR.ALL.GPU + ERRBAR, which also waits for the thread's
// outstanding global output stores of the previous block: the first version of this kernel lost ~40 k clocks per tile
// to it.)
__device__ __forceinline__ void st_async_f32x2(uint32_t cluster_addr, float a, float b, uint32_t cluster_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(cluster_addr),
               "f"(a), "f"(b), "r"(cluster_bar)
               : "memory");
}
// the row addresses come out of shared memory as integers: say that they are global (a plain C++ store through the
// reinterpreted pointer compiles to the generic ST, which resolves the address space per access)
__device__ __forceinline__ void st_global_f32(unsigned long long addr, float v) {
  asm volatile("st.global.f32 [%0], %1;" ::"l"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_global_v4(unsigned long long addr, const uint4& v) {
  asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void named_bar_sync_epi() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// running (max, sum exp) over one 32-column chunk held as raw accumulator bits + the staged bias slice
__device__ __forceinline__ void online_chunk(const uint32_t (&r)[32], const float* bias_s, float& m, float& s) {
  float v[32];
  const float4* b4 = reinterpret_cast<const float4*>(bias_s);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = b4[j];
    v[4 * j] = __uint_as_float(r[4 * j]) + b.x;
    v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b.y;
    v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b.z;
    v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b.w;
  }
  float cm = v[0];
#pragma unroll
  for (int j = 1; j < 32; ++j) cm = fmaxf(cm, v[j]);
  const float mn = fmaxf(m, cm);
  const float off = mn * LOG2E;
  float a = 0.0f;
#pragma unroll
  for (int j = 0; j < 32; ++j) a += ex2_approx(fmaf(v[j], LOG2E, -off));  // columns >= N carry bias -inf: exp = 0
  s = fmaf(s, ex2_approx((m - mn) * LOG2E), a);
  m = mn;
}

template <int MODE>
__global__ void __maxnreg__(168)
    gemm_logsoftmax_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                           const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
                           const Params p) {
  constexpr bool COMPACT = MODE == OUT_COMPACT;
  constexpr bool SCORE = MODE == OUT_SCORE;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + ST * A_STAGE_BYTES;
  uint8_t* smem_epi = smem_b + ST * B_STAGE_BYTES;
  float* bias_s = reinterpret_cast<float*>(smem_epi + 8 * BOX_BYTES);
  float2* xchg = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(bias_s) + BN * 4);
  unsigned long long* rowptr_s = reinterpret_cast<unsigned long long*>(reinterpret_cast<uint8_t*>(xchg) + XCHG_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(rowptr_s) + ROWPTR_BYTES);
  uint64_t* empty_bar = full_bar + ST;
  uint64_t* tfull_bar = empty_bar + ST;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* x_bar = tempty_bar + 2;
  uint64_t* x2_bar = x_bar + 2;  // scoring instance: argmax exchange into rank 0
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x2_bar + 2);
  float2* xchg2 = reinterpret_cast<float2*>(smem_epi);  // [accumulator parity][source rank, half][row] (max, column)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  const int rank = static_cast<int>(cluster_ctarank());  // = this CTA's column tile
  const int cl = p.cluster;
  const int cluster_id = blockIdx.x / cl;
  const int n_clusters = gridDim.x / cl;
  const int k_iters = p.k_blocks * p.passes;
  const int n0 = rank * BN;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a_hi);
    prefetch_tmap(&tm_w_hi);
    if (p.passes > 1) {
      prefetch_tmap(&tm_a_lo);
      prefetch_tmap(&tm_w_lo);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < ST; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 8);  // one arrive per epilogue warp
      mbar_init(&x_bar[a], 1);  // one arrive.expect_tx per block; the peers' st.async stores complete the bytes
      if (SCORE) mbar_init(&x2_bar[a], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  // every CTA's exchange barriers exist before a peer may arrive on them
  cluster_arrive_release();
  cluster_wait_acquire();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = static_cast<uint32_t>((BM + BN) * BK * 2);
    for (int mb = cluster_id; mb < p.tiles_m; mb += n_clusters) {
      for (int pass = 0; pass < p.passes; ++pass) {
        // pass 0: hi.hi;  NNAM_SPLIT_AW: 1 = A_hi.W_lo, 2 = A_lo.W_hi;  NNAM_SPLIT_A: 1 = A_lo.W_hi;  NNAM_SPLIT_W: 1 = A_hi.W_lo
        const CUtensorMap* ma = (pass == 2 || (pass == 1 && p.nsplit == NNAM_SPLIT_A)) ? &tm_a_lo : &tm_a_hi;
        const CUtensorMap* mw = (pass == 1 && p.nsplit != NNAM_SPLIT_A) ? &tm_w_lo : &tm_w_hi;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full_bar[stage], tx_bytes);
            tma_load_2d(smem_a + stage * A_STAGE_BYTES, ma, &full_bar[stage], kb * BK, mb * BM);
            tma_load_2d(smem_b + stage * B_STAGE_BYTES, mw, &full_bar[stage], kb * BK, n0);
          }
          __syncwarp();
          if (++stage == ST) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t idesc = make_idesc_e16_f32(BM, BN, p.f16);
    const uint64_t adesc0 = make_sw128_kmajor_desc(smem_u32(smem_a));
    const uint64_t bdesc0 = make_sw128_kmajor_desc(smem_u32(smem_b));
    for (int mb = cluster_id; mb < p.tiles_m; mb += n_clusters) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * BN);
      for (int it = 0; it < k_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t ad = adesc0 + static_cast<uint64_t>((stage * A_STAGE_BYTES) >> 4);
          const uint64_t bd = bdesc0 + static_cast<uint64_t>((stage * B_STAGE_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)
            umma_bf16(tmem_d, ad + static_cast<uint64_t>((k * UK * 2) >> 4), bd + static_cast<uint64_t>((k * UK * 2) >> 4),
                      idesc, (it | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (it == k_iters - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++stage == ST) {
          stage = 0;
          phase ^= 1;
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    // -------------------------------------------------------------- epilogue: 8 warps, two per TMEM lane quarter
    const int q = warp & 3;               // TMEM lane quarter of this warp
    const int hf = (warp - 4) >> 2;       // which 128-column half of the tile this warp handles
    const int trow = q * 32 + lane;       // row of the 128-row block = TMEM lane this thread owns
    const int h0 = hf * HALF;             // first column (within the tile) of this warp's half
    uint8_t* box = smem_epi + (warp - 4) * BOX_BYTES;
    unsigned long long* rowptr = rowptr_s + (warp - 4) * 32;  // this warp's copy of its rows' output addresses
    // the CTA's column tile never changes: stage bias - prior_scale * prior once; columns >= N get -inf, so they drop
    // out of max / sum-exp without predicates (their accumulators are 0: the TMA zero-fills W rows >= N)
    {
      const int c = threadIdx.x - 128;  // 256 epilogue threads, 256 columns
      const int gc = n0 + c;
      float b = -CUDART_INF_F;
      if (gc < p.N) {
        b = p.bias != nullptr ? __ldg(p.bias + gc) : 0.0f;
        if (p.prior != nullptr) b -= p.prior_scale * __ldg(p.prior + gc);
      }
      bias_s[c] = b;
    }
    named_bar_sync_epi();
    const int valid = max(0, min(HALF, p.N - n0 - h0));  // valid columns of this warp's half (0 for a ragged last tile)
    const int nch = (valid + 31) >> 5;                   // 32-column chunks with at least one valid column
    const float* bias_h = bias_s + h0;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t x_phase = 0;  // bit a: phase of x_bar[a]
    uint32_t x2_phase = 0;  // bit a: phase of x2_bar[a] (scoring instance, rank 0)
    for (int mb = cluster_id; mb < p.tiles_m; mb += n_clusters) {
      const long long grow = static_cast<long long>(mb) * BM + trow;
      long long orow = -1;
      bool zero = false;
      if (grow < p.M) {
        orow = p.out_row_map != nullptr ? static_cast<long long>(__ldg(p.out_row_map + grow)) : grow;
        if (orow <= -2) {  // -2 - r: fill output row r with zeros (quirk Q4 rows the reference never writes)
          orow = -2 - orow;
          zero = true;
        }
      }
      // address of this row's first element of the warp's half, staged for the store loops (0: row not written)
      if constexpr (!SCORE) {
        unsigned long long a = 0;
        if (orow >= 0)
          a = COMPACT ? reinterpret_cast<unsigned long long>(p.out16 + orow * p.ld16 + n0 + h0)
                      : reinterpret_cast<unsigned long long>(p.out + orow * p.ld_out + n0 + h0);
        rowptr[lane] = a;
      }
      __syncwarp();
      const uint32_t vmask = __ballot_sync(0xffffffffu, orow >= 0);
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr =
          tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * BN + h0);

      // ---- pass 1: running max / sum-exp over this half's columns; the load of chunk c+1 is in flight while chunk c
      // is reduced
      float m = NEG_BIG, s = 0.0f;
      if (nch > 0) {
        uint32_t ra[32], rb[32];
        tmem_ld32(taddr, ra);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < HALF / 32; c += 2) {
          if (c < nch) {
            if (c + 1 < nch) tmem_ld32(taddr + 32 * (c + 1), rb);
            online_chunk(ra, bias_h + 32 * c, m, s);
            tmem_ld_wait();
            if (c + 2 < nch) tmem_ld32(taddr + 32 * (c + 2), ra);
            if (c + 1 < nch) online_chunk(rb, bias_h + 32 * (c + 1), m, s);
            tmem_ld_wait();
          }
        }
      }

      // ---- exchange the row partials with every CTA of the cluster (this one included): 2 * cl partials per row
      {
        // this CTA's barrier expects (m, s) of 128 rows from both halves of each of the `cl` CTAs in the current phase
        if (warp == 4 && lane == 0) mbar_expect_tx(&x_bar[acc], static_cast<uint32_t>(cl * 2 * BM * 8));
        const uint32_t slot = smem_u32(xchg + (acc * 2 * MAX_CLUSTER + rank * 2 + hf) * BM + trow);
        const uint32_t bar = smem_u32(&x_bar[acc]);
        for (int r = 0; r < cl; ++r)
          st_async_f32x2(mapa_shared(slot, static_cast<uint32_t>(r)), m, s, mapa_shared(bar, static_cast<uint32_t>(r)));
        mbar_wait(&x_bar[acc], (x_phase >> acc) & 1u);
        x_phase ^= 1u << acc;
      }
      float mx = NEG_BIG;
      for (int r = 0; r < 2 * cl; ++r) mx = fmaxf(mx, xchg[(acc * 2 * MAX_CLUSTER + r) * BM + trow].x);
      float sum = 0.0f;
      for (int r = 0; r < 2 * cl; ++r) {
        const float2 t = xchg[(acc * 2 * MAX_CLUSTER + r) * BM + trow];
        sum = fmaf(t.y, ex2_approx((t.x - mx) * LOG2E), sum);
      }
      const float log_sum = logf(sum);
      // float32 rows: v - (mx + log_sum).  compact: fp16(v - mx) and row_ref = max_c y = -log_sum.
      const float sub = COMPACT ? mx : mx + log_sum;
      if (COMPACT && rank == 0 && hf == 0 && orow >= 0) p.row_ref[orow] = zero ? 0.0f : -log_sum;

      // ---- pass 2 (scoring): the values the float32 instance stores, reduced to this half's (max, lowest column) and
      // the value at the target column
      float best = -CUDART_INF_F;
      int bcol = valid > 0 ? n0 + h0 : 0x7fffffff;  // an all -inf half reports its first column
      if constexpr (SCORE) {
        const int t = (orow >= 0 && !zero) ? __ldg(p.targets + orow) : -1;
        const int t_half = t - (n0 + h0);  // target column within this half; here only if in [0, valid)
        float vt = 0.0f;
        for (int c0 = 0; c0 < valid; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(taddr + c0, r);
          tmem_ld_wait();
          const float4* b4 = reinterpret_cast<const float4*>(bias_h + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = b4[j];
            // columns >= N carry bias -inf: never above `best`
            const float v[4] = {__uint_as_float(r[4 * j]) + (b.x - sub), __uint_as_float(r[4 * j + 1]) + (b.y - sub),
                                __uint_as_float(r[4 * j + 2]) + (b.z - sub), __uint_as_float(r[4 * j + 3]) + (b.w - sub)};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (v[e] > best) {
                best = v[e];
                bcol = n0 + h0 + c0 + 4 * j + e;
              }
              if (c0 + 4 * j + e == t_half) vt = v[e];
            }
          }
        }
        if (t_half >= 0 && t_half < valid) p.nll[orow] = -vt;
        else if (rank == 0 && hf == 0 && orow >= 0 && t < 0) p.nll[orow] = 0.0f;  // ignore label or zero-fill row
      }

      // ---- pass 2: second read of the accumulator, normalise, stage, store row segments
      constexpr int CH2 = COMPACT ? 64 : 32;  // columns per staged box (128 B per row)
      for (int c0 = 0; c0 < (SCORE ? 0 : valid); c0 += CH2) {
        uint4 chunks[8];
        {
          uint32_t r[CH2 / 32][32];
#pragma unroll
          for (int j0 = 0; j0 < CH2 / 32; ++j0) tmem_ld32(taddr + c0 + 32 * j0, r[j0]);
          tmem_ld_wait();
          float v[CH2];
          const float4* b4 = reinterpret_cast<const float4*>(bias_h + c0);
#pragma unroll
          for (int j = 0; j < CH2 / 4; ++j) {
            const float4 b = b4[j];
            v[4 * j] = zero ? 0.0f : __uint_as_float(r[(4 * j) >> 5][(4 * j) & 31]) + (b.x - sub);
            v[4 * j + 1] = zero ? 0.0f : __uint_as_float(r[(4 * j + 1) >> 5][(4 * j + 1) & 31]) + (b.y - sub);
            v[4 * j + 2] = zero ? 0.0f : __uint_as_float(r[(4 * j + 2) >> 5][(4 * j + 2) & 31]) + (b.z - sub);
            v[4 * j + 3] = zero ? 0.0f : __uint_as_float(r[(4 * j + 3) >> 5][(4 * j + 3) & 31]) + (b.w - sub);
          }
          if (COMPACT) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_f16x2(v[8 * j], v[8 * j + 1]), pack_f16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_f16x2(v[8 * j + 4], v[8 * j + 5]), pack_f16x2(v[8 * j + 6], v[8 * j + 7]));
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]),
                                     __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
          }
        }
        // 16-byte chunk j of row `lane` at chunk position j ^ (lane & 7): conflict-free writes and reads
        {
          uint8_t* row = box + lane * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j) *reinterpret_cast<uint4*>(row + ((j ^ (lane & 7)) << 4)) = chunks[j];
        }
        __syncwarp();
        if (COMPACT) {
          // rows of out16 are 16-byte aligned (ld16 % 8 == 0): 8 lanes write one 128-byte row segment, 4 rows at a time
          const int sub_row = lane >> 3, ch = lane & 7;
          const int cw = c0 + ch * 8;          // first of this lane's 8 columns, within the half
          const int left = valid - cw;         // valid columns from there on
#pragma unroll
          for (int rr = 0; rr < 32; rr += 4) {
            const int r_ = rr + sub_row;
            const unsigned long long base = rowptr[r_];
            if (base != 0 && left > 0) {
              const uint4 val = *reinterpret_cast<const uint4*>(box + r_ * 128 + ((ch ^ (r_ & 7)) << 4));
              uint16_t* d = reinterpret_cast<uint16_t*>(base) + cw;
              if (left >= 8) {
                st_global_v4(base + static_cast<unsigned long long>(cw) * 2ull, val);
              } else {
                const uint32_t w[4] = {val.x, val.y, val.z, val.w};
                for (int e = 0; e < left; ++e) d[e] = static_cast<uint16_t>((w[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
              }
            }
          }
        } else {
          // (N, C) float32 rows are only 4-byte aligned: a warp writes one 128-byte row segment per instruction
          const bool col_ok = c0 + lane < valid;
          const unsigned long long lane_off = static_cast<unsigned long long>(c0 + lane) * 4ull;
#pragma unroll
          for (int rr = 0; rr < 32; ++rr) {
            if ((vmask >> rr) & 1u) {  // warp-uniform
              const unsigned long long base = rowptr[rr];  // broadcast
              const float val = *reinterpret_cast<const float*>(box + rr * 128 + (((lane >> 2) ^ (rr & 7)) << 4) + ((lane & 3) << 2));
              if (col_ok) st_global_f32(base + lane_off, val);
            }
          }
        }
        __syncwarp();  // the box is rewritten by the next chunk
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if constexpr (SCORE) {
        // every half's (max, column) of the row goes to rank 0, whose half-0 threads pick the lowest column among the
        // maxima (sources in column order) and write pred
        if (rank == 0 && warp == 4 && lane == 0) mbar_expect_tx(&x2_bar[acc], static_cast<uint32_t>(cl * 2 * BM * 8));
        const uint32_t slot = smem_u32(xchg2 + (acc * 2 * MAX_CLUSTER + rank * 2 + hf) * BM + trow);
        st_async_f32x2(mapa_shared(slot, 0u), best, __int_as_float(bcol), mapa_shared(smem_u32(&x2_bar[acc]), 0u));
        if (rank == 0 && hf == 0) {
          mbar_wait(&x2_bar[acc], (x2_phase >> acc) & 1u);
          x2_phase ^= 1u << acc;
          if (orow >= 0) {
            float bv = -CUDART_INF_F;
            int bc = 0x7fffffff;
            for (int r = 0; r < 2 * cl; ++r) {
              const float2 e = xchg2[(acc * 2 * MAX_CLUSTER + r) * BM + trow];
              const int c = __float_as_int(e.y);
              if (e.x > bv || (e.x == bv && c < bc)) {
                bv = e.x;
                bc = c;
              }
            }
            p.pred[orow] = zero ? -1 : bc;
          }
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  // no CTA leaves while a peer could still write into its exchange slots or arrive on its barriers
  cluster_arrive_release();
  cluster_wait_acquire();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int MODE>
static int launch(const CUtensorMap (&tm)[4], const Params& p, cudaStream_t stream) {
  auto kernel = gemm_logsoftmax_kernel<MODE>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  if (e != cudaSuccess) return set_cuda_error(e, "linear_logsoftmax: cudaFuncSetAttribute");
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(p.cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // how many clusters can be resident at once: the kernel is persistent over the 128-row blocks
  cfg.gridDim = dim3(static_cast<unsigned>(p.cluster * p.tiles_m));
  int max_clusters = 0;
  e = cudaOccupancyMaxActiveClusters(&max_clusters, kernel, &cfg);
  if (e != cudaSuccess) return set_cuda_error(e, "linear_logsoftmax: cudaOccupancyMaxActiveClusters");
  if (max_clusters < 1) return set_error(NNAM_ERR_UNSUPPORTED, "linear_logsoftmax: no cluster of %d CTAs fits the device", p.cluster);
  const int n_clusters = p.tiles_m < max_clusters ? p.tiles_m : max_clusters;
  cfg.gridDim = dim3(static_cast<unsigned>(p.cluster * n_clusters));
  e = cudaLaunchKernelEx(&cfg, kernel, tm[0], tm[1], tm[2], tm[3], p);
  if (e != cudaSuccess) return set_cuda_error(e, "linear_logsoftmax: launch");
  return check_launch("gemm_logsoftmax_kernel");
}

}  // namespace fused

int linear_logsoftmax(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                      long long ldw, const float* bias, const float* prior, float prior_scale, float* out,
                      long long ld_out, void* out16, long long ld16, float* row_ref, const int* out_row_map,
                      const int* targets, float* nll, int* pred, int M, int N, int K, int nsplit, int elem,
                      cudaStream_t stream) {
  using namespace fused;
  if (M <= 0 || N <= 0 || K <= 0) return set_error(NNAM_ERR_ARG, "linear_logsoftmax: empty problem");
  if (N > MAX_CLUSTER * BN)
    return set_error(NNAM_ERR_UNSUPPORTED, "linear_logsoftmax: at most %d classes (8 column tiles of 256)", MAX_CLUSTER * BN);
  if (nsplit < NNAM_SPLIT_NONE || nsplit > NNAM_SPLIT_W)
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: nsplit must be one of NNAM_SPLIT_* (1..4)");
  if (elem != NNAM_ELEM_BF16 && elem != NNAM_ELEM_F16)
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: unknown element type %d", elem);
  if (elem == NNAM_ELEM_F16 && nsplit != NNAM_SPLIT_NONE)
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: the hi/lo split passes are defined for bf16 operands only");
  const bool need_a_lo = nsplit == NNAM_SPLIT_A || nsplit == NNAM_SPLIT_AW;
  const bool need_w_lo = nsplit == NNAM_SPLIT_W || nsplit == NNAM_SPLIT_AW;
  if (lda % 8 || ldw % 8) return set_error(NNAM_ERR_ARG, "linear_logsoftmax: lda/ldw must be multiples of 8 elements (16 B)");
  if (lda < K || ldw < K) return set_error(NNAM_ERR_ARG, "linear_logsoftmax: leading dimension smaller than K");
  if ((need_a_lo && !a_lo) || (need_w_lo && !w_lo))
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: split passes need their lo operands");
  if ((out != nullptr) + (out16 != nullptr) + (nll != nullptr) != 1)
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: exactly one of out / out16 / nll must be given");
  if (nll != nullptr && (targets == nullptr || pred == nullptr))
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: scoring needs targets, nll and pred");
  if (out != nullptr && ld_out < N) return set_error(NNAM_ERR_ARG, "linear_logsoftmax: ld_out must be >= N");
  if (out16 != nullptr && (row_ref == nullptr || ld16 < N || ld16 % 8 || (reinterpret_cast<uintptr_t>(out16) & 15)))
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: compact output needs row_ref, ld16 >= N, ld16 %% 8 == 0, 16-byte alignment");
  if ((reinterpret_cast<uintptr_t>(a_hi) | reinterpret_cast<uintptr_t>(w_hi) | reinterpret_cast<uintptr_t>(a_lo) |
       reinterpret_cast<uintptr_t>(w_lo)) & 15)
    return set_error(NNAM_ERR_ARG, "linear_logsoftmax: operand pointers must be 16-byte aligned");

  Params p;
  p.M = M;
  p.N = N;
  p.K = K;
  p.tiles_m = (M + BM - 1) / BM;
  p.k_blocks = (K + BK - 1) / BK;
  p.nsplit = nsplit;
  p.passes = nsplit == NNAM_SPLIT_AW ? 3 : (nsplit == NNAM_SPLIT_NONE ? 1 : 2);
  p.f16 = elem == NNAM_ELEM_F16;
  p.cluster = (N + BN - 1) / BN;
  p.bias = bias;
  p.prior = prior;
  p.prior_scale = prior_scale;
  p.ld_out = ld_out;
  p.ld16 = ld16;
  p.out_row_map = out_row_map;
  if (nll != nullptr) {
    p.nll = nll;
    p.pred = pred;
    p.targets = targets;
  } else {
    p.out = out;
    p.out16 = static_cast<uint16_t*>(out16);
    p.row_ref = row_ref;
  }

  CUtensorMap tm[4];
  int rc;
  if ((rc = encode_tmap_bf16_2d(&tm[0], a_hi, K, M, lda, BK, BM))) return rc;
  if ((rc = encode_tmap_bf16_2d(&tm[2], w_hi, K, N, ldw, BK, BN))) return rc;
  tm[1] = tm[0];
  tm[3] = tm[2];
  if (need_a_lo && (rc = encode_tmap_bf16_2d(&tm[1], a_lo, K, M, lda, BK, BM))) return rc;
  if (need_w_lo && (rc = encode_tmap_bf16_2d(&tm[3], w_lo, K, N, ldw, BK, BN))) return rc;
  if (nll != nullptr) return launch<OUT_SCORE>(tm, p, stream);
  return out16 != nullptr ? launch<OUT_COMPACT>(tm, p, stream) : launch<OUT_ROWS>(tm, p, stream);
}

}  // namespace nnam
