// K2 -- Linear layer as a tcgen05/TMEM GEMM fed by TMA, bias + activation fused in the epilogue.
//
//   out[M, N] = act( A[M, K] . W[N, K]^T + bias[N] )
//
// Replaces every ``L.Linear`` call of the reference model specs (scripts/common/chainer_networks.py:16-22,
// 51-52, 61-62 ...; Chainer F.linear = x.dot(W.T) + b) and the batched input-to-hidden projections of the
// recurrent cells.  A and W are bf16, K-major (row-major with K contiguous), exactly the Chainer (out, in)
// weight layout, so no transposition is ever needed.
//
// Precision modes (nsplit = NNAM_SPLIT_*; elem = NNAM_ELEM_* picks bf16 or fp16 operands for the single-pass mode):
//   1  "bf16" / "fp16" : one pass, A_hi . W_hi
//   3  "bf16x3" : fp32-accurate.  A = A_hi + A_lo, W = W_hi + W_lo (each bf16); the kernel accumulates
//                 A_hi.W_hi + A_hi.W_lo + A_lo.W_hi into the same fp32 TMEM accumulator (the dropped
//                 A_lo.W_lo term is ~2^-18 relative).  Costs 3 bf16 passes = 1.5 TF32 passes but carries
//                 16 mantissa bits instead of TF32's 10.
//   2  A split only (A_hi.W_hi + A_lo.W_hi) and 4  W split only (A_hi.W_hi + A_hi.W_lo): two passes; per-layer
//                 choices for the bf16 parity study (which operand's rounding flips the frame argmax).
//
// Structure: persistent, warp-specialised, one CTA per SM.
//   warp 0 : TMA producer (one lane)          -- smem ring of STAGES x (A 128x64 + W bn x64) bf16, SWIZZLE_128B
//   warp 1 : tcgen05.mma issuer (one lane)    -- UMMA 128 x bn x 16, fp32 accumulators in TMEM, double-buffered
//   warp 2 : TMEM allocator
//   warps 4-7 : epilogue -- tcgen05.ld 32x32b, + bias, activation, (hi/lo split), vector stores
// Tile order is n-fastest so that CTAs running concurrently share the A tile in L2 while W stays L2-resident.
#include <stdlib.h>

#include "ptx.cuh"
#include "nnam_internal.h"

namespace nnam {

constexpr int BM = 128;
constexpr int BK = 64;  // bf16 elements per k-block = 128 B = one swizzle row
constexpr int UK = 16;  // K of one tcgen05.mma (kind::f16)
constexpr int MAX_BN = 256;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BM * BK * 2;      // 16 KiB
constexpr int B_STAGE_BYTES = MAX_BN * BK * 2;  // 32 KiB
constexpr int GEMM_THREADS = 256;
constexpr int EPI_BOX_BYTES = 32 * 128;         // one epilogue warp's store box: 32 rows x 128 B, SWIZZLE_128B
constexpr int EPI_BYTES = 4 * 2 * EPI_BOX_BYTES;  // 4 epilogue warps x 2 alternating boxes
constexpr int BIAS_BYTES = 2 * MAX_BN * 4;        // the tile's bias slice, double-buffered by tile parity
constexpr int GEMM_SMEM_BYTES = STAGES * (A_STAGE_BYTES + B_STAGE_BYTES) + EPI_BYTES + BIAS_BYTES + 256;
constexpr int TMEM_COLS = 512;

struct GemmParams {
  int M, N, K;
  int bn;         // tile width: a multiple of the store box width (64 bf16 / 32 fp32 columns), <= 256
  int tiles_m, tiles_n;
  int k_blocks;   // ceil(K / 64)
  int nsplit;     // NNAM_SPLIT_*
  int passes;     // tensor passes over K: 1, 2 or 3
  int f16;        // operands (and 16-bit outputs) are fp16 instead of bf16
  int act;        // NNAM_ACT_*
  const float* bias;
  void* out_hi;   // output planes and leading dimension, for the direct stores of a row's ragged last box
  void* out_lo;
  long long ldo;
};

// barrier among the four epilogue warps only (named barrier 1, 128 threads)
__device__ __forceinline__ void named_bar_sync_epi() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int ACT>
__device__ __forceinline__ float act_fn(float v) {
  if (ACT == NNAM_ACT_RELU) return fmaxf(v, 0.0f);
  if (ACT == NNAM_ACT_SIGMOID) return tanhf(v * 0.5f) * 0.5f + 0.5f;  // Chainer's sigmoid formulation
  if (ACT == NNAM_ACT_TANH) return tanhf(v);
  return v;
}

template <int NV>
__device__ __forceinline__ void apply_act(float (&v)[NV], int act) {  // warp-uniform switch hoisted out of the loop
  if (act == NNAM_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < NV; ++j) v[j] = act_fn<NNAM_ACT_RELU>(v[j]);
  } else if (act == NNAM_ACT_SIGMOID) {
#pragma unroll
    for (int j = 0; j < NV; ++j) v[j] = act_fn<NNAM_ACT_SIGMOID>(v[j]);
  } else if (act == NNAM_ACT_TANH) {
#pragma unroll
    for (int j = 0; j < NV; ++j) v[j] = act_fn<NNAM_ACT_TANH>(v[j]);
  }
}

// Output tile staging: the warp's 32 rows x 128 B go to shared memory in the SWIZZLE_128B pattern (16-byte chunk j of
// row r lives at chunk position j ^ (r & 7): conflict-free for 8 consecutive lanes), then ONE lane hands the box to
// the TMA store engine, which clips rows >= M and columns >= N (the latter only at 16-byte granularity: see
// box_crosses_ragged_end).  Replaces per-thread row-strided global stores, whose 32 separate lines per instruction
// had the L1/LSU pipe at ~73 % (profiles/r01_cfg2_gemm_before.md).
__device__ __forceinline__ void stage_row_128B(uint8_t* box, int lane, const uint4 (&chunks)[8]) {
  uint8_t* row = box + lane * 128;
#pragma unroll
  for (int j = 0; j < 8; ++j) *reinterpret_cast<uint4*>(row + ((j ^ (lane & 7)) << 4)) = chunks[j];
}

// The TMA store clips a box that crosses column N only at 16-byte granularity: the rest of the 16-byte segment holding
// column N - 1 would be written too.  When N does not end on a 16-byte boundary, the box that crosses N is therefore
// stored by each lane for its own row, element by element, and nothing past column N is touched.
template <int OUT_KIND>
__device__ __forceinline__ bool box_crosses_ragged_end(int col, int n) {
  constexpr int BOX_COLS = OUT_KIND == NNAM_OUT_F32 ? 32 : 64;
  constexpr int PER_16B = OUT_KIND == NNAM_OUT_F32 ? 4 : 8;
  return col + BOX_COLS > n && (n % PER_16B) != 0;
}
template <int OUT_KIND>
__device__ __forceinline__ void store_row_prefix(void* base, long long ldo, int row, int col, int valid,
                                                 const uint4 (&chunks)[8]) {
  if (OUT_KIND == NNAM_OUT_F32) {
    uint32_t* d = static_cast<uint32_t*>(base) + static_cast<long long>(row) * ldo + col;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t w[4] = {chunks[j].x, chunks[j].y, chunks[j].z, chunks[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (4 * j + e < valid) d[4 * j + e] = w[e];
    }
  } else {
    uint16_t* d = static_cast<uint16_t*>(base) + static_cast<long long>(row) * ldo + col;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t w[4] = {chunks[j].x, chunks[j].y, chunks[j].z, chunks[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (8 * j + 2 * e < valid) d[8 * j + 2 * e] = static_cast<uint16_t>(w[e] & 0xffffu);
        if (8 * j + 2 * e + 1 < valid) d[8 * j + 2 * e + 1] = static_cast<uint16_t>(w[e] >> 16);
      }
    }
  }
}

// Registers are capped (not via __launch_bounds__, which would let ptxas take 240) so that a 256-thread GEMM CTA leaves
// room on the SM for one 128-thread CTA of the HBM-bound head / splice kernels, which the engine runs on a second
// stream in the shadow of the GEMMs.
constexpr int GEMM_MAX_REGS = 184;

// ST: stages of the operand ring; NBOX: staging boxes per epilogue warp = TMA stores it keeps in flight.
template <int OUT_KIND, int ST, int NBOX>
__global__ void __maxnreg__(GEMM_MAX_REGS)
    gemm_bias_act_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                         const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
                         const __grid_constant__ CUtensorMap tm_o_hi, const __grid_constant__ CUtensorMap tm_o_lo,
                         const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];  // SWIZZLE_128B tiles need 1024 B alignment (checked below)
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + ST * A_STAGE_BYTES;
  uint8_t* smem_epi = smem_b + ST * B_STAGE_BYTES;
  float* smem_bias = reinterpret_cast<float*>(smem_epi + (4 * NBOX * EPI_BOX_BYTES));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_epi + (4 * NBOX * EPI_BOX_BYTES) + BIAS_BYTES);
  uint64_t* empty_bar = full_bar + ST;
  uint64_t* tfull_bar = empty_bar + ST;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.tiles_m * p.tiles_n;
  const int k_iters = p.k_blocks * p.passes;
  if ((smem_u32(smem) & 1023u) != 0) __trap();  // the dynamic shared window is 1024-byte aligned on sm_100

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a_hi);
    prefetch_tmap(&tm_w_hi);
    prefetch_tmap(&tm_o_hi);
    if (p.passes > 1) {
      prefetch_tmap(&tm_a_lo);
      prefetch_tmap(&tm_w_lo);
    }
    if (OUT_KIND == NNAM_OUT_BF16_SPLIT) prefetch_tmap(&tm_o_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < ST; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 4);  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // The producer and MMA warps run their loops with ALL lanes (warp-uniform control flow keeps addresses and
  // descriptors in uniform registers) and elect one lane only around the TMA / tcgen05 instructions.  The first version
  // ran the loops under `if (lane == 0)`: ptxas then wraps every uniform-datapath instruction in an ELECT waterfall
  // loop, and the MMA warp needed ~680 clocks to issue the 4 MMAs of a k-block that the tensor pipe retires in 512 --
  // the issue loop, not memory, capped the tensor pipe at 85 % (profiles/r01_cfg2_gemm_v2.md).
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = static_cast<uint32_t>((BM + p.bn) * BK * 2);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_blk = tile / p.tiles_n;
      const int n_blk = tile % p.tiles_n;
      for (int pass = 0; pass < p.passes; ++pass) {
        // pass 0: hi.hi;  NNAM_SPLIT_AW: 1 = A_hi.W_lo, 2 = A_lo.W_hi;  NNAM_SPLIT_A: 1 = A_lo.W_hi;  NNAM_SPLIT_W: 1 = A_hi.W_lo
        const CUtensorMap* ma = (pass == 2 || (pass == 1 && p.nsplit == NNAM_SPLIT_A)) ? &tm_a_lo : &tm_a_hi;
        const CUtensorMap* mw = (pass == 1 && p.nsplit != NNAM_SPLIT_A) ? &tm_w_lo : &tm_w_hi;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full_bar[stage], tx_bytes);
            tma_load_2d(smem_a + stage * A_STAGE_BYTES, ma, &full_bar[stage], kb * BK, m_blk * BM);
            tma_load_2d(smem_b + stage * B_STAGE_BYTES, mw, &full_bar[stage], kb * BK, n_blk * p.bn);
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
    const uint32_t idesc = make_idesc_e16_f32(BM, static_cast<uint32_t>(p.bn), p.f16);
    const uint64_t adesc0 = make_sw128_kmajor_desc(smem_u32(smem_a));
    const uint64_t bdesc0 = make_sw128_kmajor_desc(smem_u32(smem_b));
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * MAX_BN);
      for (int it = 0; it < k_iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          // the start-address field of the descriptor counts 16-byte units: stage and k offsets are plain adds
          const uint64_t ad = adesc0 + static_cast<uint64_t>((stage * A_STAGE_BYTES) >> 4);
          const uint64_t bd = bdesc0 + static_cast<uint64_t>((stage * B_STAGE_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < BK / UK; ++k)
            umma_bf16(tmem_d, ad + static_cast<uint64_t>((k * UK * 2) >> 4), bd + static_cast<uint64_t>((k * UK * 2) >> 4),
                      idesc, (it | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs have read it
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
    // -------------------------------------------------------------- epilogue
    // TMEM -> registers (tcgen05.ld 32x32b.x32) -> + bias, activation, (hi/lo split) -> swizzled smem box -> TMA store
    constexpr int BOX_COLS = OUT_KIND == NNAM_OUT_F32 ? 32 : 64;  // 128 B of output per row and box
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    uint8_t* boxes = smem_epi + q * NBOX * EPI_BOX_BYTES;
    int box_sel = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m_blk = tile / p.tiles_n;
      const int n_blk = tile % p.tiles_n;
      // the tile's bias slice goes to shared memory once (each thread of the four epilogue warps loads two values);
      // every thread needs every column's bias, and as broadcast shared loads that costs a fraction of the 256
      // 128-bit global loads per tile the first version issued (they alone held short-K layers ~25 us back)
      float* bias_s = smem_bias + acc * MAX_BN;
      if (p.bias != nullptr) {
        for (int c = q * 32 + lane; c < p.bn; c += 128) {
          const int gc = n_blk * p.bn + c;
          bias_s[c] = gc < p.N ? __ldg(p.bias + gc) : 0.0f;
        }
      }
      named_bar_sync_epi();
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * MAX_BN);
      const int row0 = m_blk * BM + q * 32;
      for (int c0 = 0; c0 < p.bn; c0 += BOX_COLS) {
        const int col = n_blk * p.bn + c0;
        if (col >= p.N || row0 >= p.M) break;  // warp-uniform; the TMA store clips partial boxes
        float v[BOX_COLS];
        {
          // both 32-column loads of a bf16 box are issued before the one wait (a single epilogue warp per scheduler
          // has nothing else to hide the TMEM latency behind)
          uint32_t r[BOX_COLS / 32][32];
#pragma unroll
          for (int j0 = 0; j0 < BOX_COLS / 32; ++j0) tmem_ld32(taddr + c0 + 32 * j0, r[j0]);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < BOX_COLS; ++j) v[j] = __uint_as_float(r[j >> 5][j & 31]);
        }
        if (p.bias != nullptr) {
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + c0);  // broadcast reads of the staged slice
#pragma unroll
          for (int j = 0; j < BOX_COLS / 4; ++j) {
            const float4 b = b4[j];
            v[4 * j] += b.x;
            v[4 * j + 1] += b.y;
            v[4 * j + 2] += b.z;
            v[4 * j + 3] += b.w;
          }
        }
        apply_act<BOX_COLS>(v, p.act);

        constexpr int N_OUT = OUT_KIND == NNAM_OUT_BF16_SPLIT ? 2 : 1;
#pragma unroll
        for (int o = 0; o < N_OUT; ++o) {
          uint4 chunks[8];
          if (OUT_KIND == NNAM_OUT_F32) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]),
                                     __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
          } else if (OUT_KIND == NNAM_OUT_F16) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_f16x2(v[8 * j], v[8 * j + 1]), pack_f16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_f16x2(v[8 * j + 4], v[8 * j + 5]), pack_f16x2(v[8 * j + 6], v[8 * j + 7]));
          } else if (o == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
          } else {
#pragma unroll
            for (int j = 0; j < BOX_COLS; ++j) v[j] -= bf16_round(v[j]);  // low half of the hi/lo split
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
          }
          if (box_crosses_ragged_end<OUT_KIND>(col, p.N)) {  // warp-uniform
            if (row0 + lane < p.M) store_row_prefix<OUT_KIND>(o == 0 ? p.out_hi : p.out_lo, p.ldo, row0 + lane, col,
                                                              p.N - col, chunks);
            continue;
          }
          uint8_t* box = boxes + box_sel * EPI_BOX_BYTES;
          if (lane == 0) tma_store_wait_read<NBOX - 1>();  // the store issued from this box NBOX boxes ago has read it
          __syncwarp();
          stage_row_128B(box, lane, chunks);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(o == 0 ? &tm_o_hi : &tm_o_lo, box, col, row0);
            tma_store_commit();
          }
          box_sel = box_sel + 1 == NBOX ? 0 : box_sel + 1;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) tma_store_wait<0>();  // all output boxes written before the CTA retires
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// =====================================================================================================
// CTA-pair variant (cta_group::2): the two CTAs of a cluster (one TPC) compute ONE 256 x bn tile.
//
// Why: with a 128 x 256 tile per SM the main loop pulls A 16 KiB + W 32 KiB per 512 tensor-core clocks = 96 B/clk from
// L2 into each SM and reads the same 96 B/clk back out of shared memory for the MMA; 4 stages of 48 KiB cover only
// ~2 k clocks of L2 latency, and the second ncu pass (profiles/r01_cfg2_gemm_v2.md) shows the tensor pipe capped at
// ~85 % with ~3 k clocks lost per tile.  In a pair, each CTA loads its own 128 rows of A and only HALF of the W tile
// (32 KiB per stage, so SIX stages fit), the leader issues tcgen05.mma.cta_group::2 with M = 256, and each CTA's
// tensor core accumulates its 128 rows in its own TMEM: 64 B/clk per SM from L2 and from shared memory.
//
// Protocol (same barriers at the same offsets in both CTAs; rank 0 = leader):
//   full[s]    leader only: arrive.expect_tx by the leader's producer for BOTH CTAs' bytes; both producers' TMA loads
//              complete_tx on it (cp.async.bulk.tensor ... cta_group::2 may signal the peer's mbarrier)
//   empty[s]   each CTA: tcgen05.commit.cta_group::2 ... multicast (mask 0b11) from the leader's MMA thread
//   tfull[a]   each CTA: same multicast commit after the last k-block of a tile
//   tempty[a]  leader only, count 8: the four epilogue warps of BOTH CTAs arrive (the follower's remotely)
constexpr int STAGES2 = 6;
constexpr int B2_STAGE_BYTES = (MAX_BN / 2) * BK * 2;  // 16 KiB: this CTA's half of the W tile
constexpr int GEMM2_SMEM_BYTES = STAGES2 * (A_STAGE_BYTES + B2_STAGE_BYTES) + EPI_BYTES + BIAS_BYTES + 256;

template <int OUT_KIND>
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(GEMM_MAX_REGS)
    gemm_bias_act_2sm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                             const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
                             const __grid_constant__ CUtensorMap tm_o_hi, const __grid_constant__ CUtensorMap tm_o_lo,
                             const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES2 * A_STAGE_BYTES;
  uint8_t* smem_epi = smem_b + STAGES2 * B2_STAGE_BYTES;
  float* smem_bias = reinterpret_cast<float*>(smem_epi + EPI_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_epi + EPI_BYTES + BIAS_BYTES);
  uint64_t* empty_bar = full_bar + STAGES2;
  uint64_t* tfull_bar = empty_bar + STAGES2;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;
  const int total_tiles = p.tiles_m * p.tiles_n;  // tiles_m counts 256-row blocks here
  const int k_iters = p.k_blocks * p.passes;
  const int half_bn = p.bn >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a_hi);
    prefetch_tmap(&tm_w_hi);
    prefetch_tmap(&tm_o_hi);
    if (p.passes > 1) {
      prefetch_tmap(&tm_a_lo);
      prefetch_tmap(&tm_w_lo);
    }
    if (OUT_KIND == NNAM_OUT_BF16_SPLIT) prefetch_tmap(&tm_o_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES2; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 8);  // four epilogue warps of each CTA of the pair
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  // both CTAs' barriers are initialised (and both TMEM allocations done) before any cross-CTA signal
  cluster_arrive_release();
  cluster_wait_acquire();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs; all lanes, one elected)
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = static_cast<uint32_t>(2 * (BM + half_bn) * BK * 2);  // both CTAs' boxes
    for (int tile = pair; tile < total_tiles; tile += n_pairs) {
      const int m_blk = tile / p.tiles_n;
      const int n_blk = tile % p.tiles_n;
      const int row_a = m_blk * (2 * BM) + static_cast<int>(rank) * BM;
      const int row_w = n_blk * p.bn + static_cast<int>(rank) * half_bn;
      for (int pass = 0; pass < p.passes; ++pass) {
        // pass 0: hi.hi;  NNAM_SPLIT_AW: 1 = A_hi.W_lo, 2 = A_lo.W_hi;  NNAM_SPLIT_A: 1 = A_lo.W_hi;  NNAM_SPLIT_W: 1 = A_hi.W_lo
        const CUtensorMap* ma = (pass == 2 || (pass == 1 && p.nsplit == NNAM_SPLIT_A)) ? &tm_a_lo : &tm_a_hi;
        const CUtensorMap* mw = (pass == 1 && p.nsplit != NNAM_SPLIT_A) ? &tm_w_lo : &tm_w_hi;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            const uint32_t full_leader = mapa_shared(smem_u32(&full_bar[stage]), 0);
            if (leader) mbar_expect_tx(&full_bar[stage], tx_bytes);
            tma_load_2d_2sm(smem_a + stage * A_STAGE_BYTES, ma, full_leader, kb * BK, row_a);
            tma_load_2d_2sm(smem_b + stage * B2_STAGE_BYTES, mw, full_leader, kb * BK, row_w);
          }
          __syncwarp();
          if (++stage == STAGES2) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ------------------------------------------------------------ MMA issuer (leader CTA only; all lanes, one elected)
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t idesc = make_idesc_e16_f32(2 * BM, static_cast<uint32_t>(p.bn), p.f16);
      const uint64_t adesc0 = make_sw128_kmajor_desc(smem_u32(smem_a));
      const uint64_t bdesc0 = make_sw128_kmajor_desc(smem_u32(smem_b));
      for (int tile = pair; tile < total_tiles; tile += n_pairs) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);  // no data crosses here: plain wait, tcgen05 fences order the rest
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * MAX_BN);
        for (int it = 0; it < k_iters; ++it) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t ad = adesc0 + static_cast<uint64_t>((stage * A_STAGE_BYTES) >> 4);
            const uint64_t bd = bdesc0 + static_cast<uint64_t>((stage * B2_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < BK / UK; ++k)
              umma_bf16_2sm(tmem_d, ad + static_cast<uint64_t>((k * UK * 2) >> 4),
                            bd + static_cast<uint64_t>((k * UK * 2) >> 4), idesc, (it | k) != 0 ? 1u : 0u);
            umma_commit_2sm(&empty_bar[stage], 0b11);  // frees the slot in both CTAs
            if (it == k_iters - 1) umma_commit_2sm(&tfull_bar[acc], 0b11);
          }
          __syncwarp();
          if (++stage == STAGES2) {
            stage = 0;
            phase ^= 1;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    // -------------------------------------------------------------- epilogue (both CTAs, own 128 rows)
    constexpr int BOX_COLS = OUT_KIND == NNAM_OUT_F32 ? 32 : 64;
    const int q = warp & 3;
    uint8_t* boxes = smem_epi + q * 2 * EPI_BOX_BYTES;
    int box_sel = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = pair; tile < total_tiles; tile += n_pairs) {
      const int m_blk = tile / p.tiles_n;
      const int n_blk = tile % p.tiles_n;
      float* bias_s = smem_bias + acc * MAX_BN;  // staged bias slice of this tile (see the single-CTA kernel)
      if (p.bias != nullptr) {
        for (int c = q * 32 + lane; c < p.bn; c += 128) {
          const int gc = n_blk * p.bn + c;
          bias_s[c] = gc < p.N ? __ldg(p.bias + gc) : 0.0f;
        }
      }
      named_bar_sync_epi();
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * MAX_BN);
      const int row0 = m_blk * (2 * BM) + static_cast<int>(rank) * BM + q * 32;
      for (int c0 = 0; c0 < p.bn; c0 += BOX_COLS) {
        const int col = n_blk * p.bn + c0;
        if (col >= p.N || row0 >= p.M) break;
        float v[BOX_COLS];
        {
          // both 32-column loads of a bf16 box are issued before the one wait (a single epilogue warp per scheduler
          // has nothing else to hide the TMEM latency behind)
          uint32_t r[BOX_COLS / 32][32];
#pragma unroll
          for (int j0 = 0; j0 < BOX_COLS / 32; ++j0) tmem_ld32(taddr + c0 + 32 * j0, r[j0]);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < BOX_COLS; ++j) v[j] = __uint_as_float(r[j >> 5][j & 31]);
        }
        if (p.bias != nullptr) {
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + c0);  // broadcast reads of the staged slice
#pragma unroll
          for (int j = 0; j < BOX_COLS / 4; ++j) {
            const float4 b = b4[j];
            v[4 * j] += b.x;
            v[4 * j + 1] += b.y;
            v[4 * j + 2] += b.z;
            v[4 * j + 3] += b.w;
          }
        }
        apply_act<BOX_COLS>(v, p.act);
        constexpr int N_OUT = OUT_KIND == NNAM_OUT_BF16_SPLIT ? 2 : 1;
#pragma unroll
        for (int o = 0; o < N_OUT; ++o) {
          uint4 chunks[8];
          if (OUT_KIND == NNAM_OUT_F32) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]),
                                     __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
          } else if (OUT_KIND == NNAM_OUT_F16) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_f16x2(v[8 * j], v[8 * j + 1]), pack_f16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_f16x2(v[8 * j + 4], v[8 * j + 5]), pack_f16x2(v[8 * j + 6], v[8 * j + 7]));
          } else {
            if (o == 1) {
#pragma unroll
              for (int j = 0; j < BOX_COLS; ++j) v[j] -= bf16_round(v[j]);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
              chunks[j] = make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
          }
          if (box_crosses_ragged_end<OUT_KIND>(col, p.N)) {  // warp-uniform
            if (row0 + lane < p.M) store_row_prefix<OUT_KIND>(o == 0 ? p.out_hi : p.out_lo, p.ldo, row0 + lane, col,
                                                              p.N - col, chunks);
            continue;
          }
          uint8_t* box = boxes + box_sel * EPI_BOX_BYTES;
          if (lane == 0) tma_store_wait_read<1>();
          __syncwarp();
          stage_row_128B(box, lane, chunks);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(o == 0 ? &tm_o_hi : &tm_o_lo, box, col, row0);
            tma_store_commit();
          }
          box_sel ^= 1;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(mapa_shared(smem_u32(&tempty_bar[acc]), 0));
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) tma_store_wait<0>();
  }

  // neither CTA may retire (or free TMEM) while its peer can still signal it or its tensor core is still in use
  tc_fence_before();
  __syncthreads();
  cluster_arrive_release();
  cluster_wait_acquire();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------ host side
// Tile width: the narrowest multiple of the store box width that covers N in ceil(N / 256) tiles.  Wide tiles win even
// when they pad N (N = 1909 -> 8 x 256, 7 % padding): measured 400 us vs 433 us for 10 x 192 on the cfg2 output layer
// (scripts/gpu_gemm_bench.py), because the A traffic per FLOP falls with the tile width.
static int pick_bn(int n, int box_cols) {
  if (const char* v = getenv("NNAM_GEMM_BN")) {  // tuning aid
    const int bn = atoi(v);
    if (bn >= box_cols && bn <= MAX_BN && bn % box_cols == 0) return bn;
  }
  const int tiles = (n + MAX_BN - 1) / MAX_BN;
  int bn = (n + tiles - 1) / tiles;
  bn = (bn + box_cols - 1) / box_cols * box_cols;
  return bn;
}

template <int OUT_KIND>
static int launch_gemm_2sm(const CUtensorMap (&tm)[6], const GemmParams& p, int grid, cudaStream_t stream) {
  // the attribute is per device and the call is a few hundred ns: set it on every launch rather than caching a flag
  // that several host threads (one per GPU) would race on
  cudaError_t e = cudaFuncSetAttribute(gemm_bias_act_2sm_kernel<OUT_KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       GEMM2_SMEM_BYTES);
  if (e != cudaSuccess) return set_cuda_error(e, "gemm: cudaFuncSetAttribute(2sm)");
  gemm_bias_act_2sm_kernel<OUT_KIND><<<grid, GEMM_THREADS, GEMM2_SMEM_BYTES, stream>>>(tm[0], tm[1], tm[2], tm[3],
                                                                                        tm[4], tm[5], p);
  return check_launch("gemm_bias_act_2sm_kernel");
}

// CTA pairs pay off (+1..7 % on the K >= 1024 shapes of the BASELINE configs) once there are enough 256-row tiles to
// keep every pair busy; NNAM_GEMM_2SM=0 forces the single-CTA kernel (A/B measurements).
static bool use_2sm(int M, int N, int K) {
  // function-local statics with initialisers are initialised once, thread-safely (C++11)
  static const int env = [] {
    const char* v = getenv("NNAM_GEMM_2SM");
    return (v != nullptr && v[0] == '0') ? 0 : 1;
  }();
  // K <= 256 is bound by the output stream in either kernel (80-86 us for a 65,536 x 2048 bf16 output); from K = 512
  // on the pair kernel wins (108.9 vs 123 us) since the accumulator hand-off between the CTAs stopped using
  // cluster-scope release / acquire (MEMBAR.ALL + ERRBAR per epilogue warp and CCTL.IVALL per tile)
  static const int min_k = [] {
    const char* v = getenv("NNAM_GEMM_2SM_MINK");  // tuning aid
    return v != nullptr ? atoi(v) : 384;
  }();
  return env == 1 && M >= 4096 && N >= 128 && K >= min_k;
}

constexpr int gemm_smem_bytes(int st, int nbox) {
  return st * (A_STAGE_BYTES + B_STAGE_BYTES) + 4 * nbox * EPI_BOX_BYTES + BIAS_BYTES + 256;
}

template <int OUT_KIND, int ST, int NBOX>
static int launch_gemm_variant(const CUtensorMap (&tm)[6], const GemmParams& p, int grid, cudaStream_t stream) {
  constexpr int smem = gemm_smem_bytes(ST, NBOX);
  static_assert(smem <= 227 * 1024, "GEMM shared memory over budget");
  cudaError_t e = cudaFuncSetAttribute(gemm_bias_act_kernel<OUT_KIND, ST, NBOX>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return set_cuda_error(e, "gemm: cudaFuncSetAttribute");
  gemm_bias_act_kernel<OUT_KIND, ST, NBOX><<<grid, GEMM_THREADS, smem, stream>>>(tm[0], tm[1], tm[2], tm[3], tm[4],
                                                                                 tm[5], p);
  return check_launch("gemm_bias_act_kernel");
}

// Experiment kept behind NNAM_GEMM_EPI_MAXK=<K>: layers with K <= that value run with 3 stages and 4 store boxes per
// epilogue warp (twice the TMA stores in flight).  Measured no change (K <= 256: 80.5 vs 80.4 us per 65,536 x 2048
// bf16 output), so the output-bound floor is not the number of stores in flight; default off.
template <int OUT_KIND>
static int launch_gemm(const CUtensorMap (&tm)[6], const GemmParams& p, int grid, cudaStream_t stream) {
  static const int max_k = [] {
    const char* v = getenv("NNAM_GEMM_EPI_MAXK");
    return v != nullptr ? atoi(v) : 0;
  }();
  if (p.K * p.passes <= max_k) return launch_gemm_variant<OUT_KIND, 3, 4>(tm, p, grid, stream);
  return launch_gemm_variant<OUT_KIND, STAGES, 2>(tm, p, grid, stream);
}

int gemm_bias_act(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                  long long ldw, const float* bias, void* out_hi, void* out_lo, long long ldo, int M, int N, int K,
                  int act, int out_kind, int nsplit, int elem, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || K <= 0) return set_error(NNAM_ERR_ARG, "gemm: empty problem");
  if (nsplit < NNAM_SPLIT_NONE || nsplit > NNAM_SPLIT_W)
    return set_error(NNAM_ERR_ARG, "gemm: nsplit must be one of NNAM_SPLIT_* (1..4)");
  if (elem != NNAM_ELEM_BF16 && elem != NNAM_ELEM_F16) return set_error(NNAM_ERR_ARG, "gemm: unknown element type %d", elem);
  if (elem == NNAM_ELEM_F16 && nsplit != NNAM_SPLIT_NONE)
    return set_error(NNAM_ERR_ARG, "gemm: the hi/lo split passes are defined for bf16 operands only");
  const bool need_a_lo = nsplit == NNAM_SPLIT_A || nsplit == NNAM_SPLIT_AW;
  const bool need_w_lo = nsplit == NNAM_SPLIT_W || nsplit == NNAM_SPLIT_AW;
  if (lda % 8 || ldw % 8) return set_error(NNAM_ERR_ARG, "gemm: lda/ldw must be multiples of 8 elements (16 B)");
  if (lda < K || ldw < K) return set_error(NNAM_ERR_ARG, "gemm: leading dimension smaller than K");
  if ((need_a_lo && !a_lo) || (need_w_lo && !w_lo)) return set_error(NNAM_ERR_ARG, "gemm: split passes need their lo operands");
  if (out_kind == NNAM_OUT_BF16_SPLIT && !out_lo) return set_error(NNAM_ERR_ARG, "gemm: split output needs out_lo");
  if (ldo < N) return set_error(NNAM_ERR_ARG, "gemm: ldo must be >= N");
  if (out_kind == NNAM_OUT_F32 ? (ldo % 4) : (ldo % 8))
    return set_error(NNAM_ERR_ARG, "gemm: ldo must keep rows 16-byte aligned");
  if ((reinterpret_cast<uintptr_t>(a_hi) | reinterpret_cast<uintptr_t>(w_hi) | reinterpret_cast<uintptr_t>(a_lo) |
       reinterpret_cast<uintptr_t>(w_lo) | reinterpret_cast<uintptr_t>(out_hi) | reinterpret_cast<uintptr_t>(out_lo) |
       reinterpret_cast<uintptr_t>(bias)) & 15)
    return set_error(NNAM_ERR_ARG, "gemm: pointers must be 16-byte aligned");

  if (out_kind != NNAM_OUT_F32 && out_kind != NNAM_OUT_BF16 && out_kind != NNAM_OUT_BF16_SPLIT && out_kind != NNAM_OUT_F16)
    return set_error(NNAM_ERR_ARG, "gemm: unknown out_kind %d", out_kind);
  const bool f32_out = out_kind == NNAM_OUT_F32;
  const int box_cols = f32_out ? 32 : 64;
  GemmParams p;
  p.M = M;
  p.N = N;
  p.K = K;
  const bool pair = use_2sm(M, N, K);
  p.bn = pick_bn(N, box_cols);
  p.tiles_m = pair ? (M + 2 * BM - 1) / (2 * BM) : (M + BM - 1) / BM;
  p.tiles_n = (N + p.bn - 1) / p.bn;
  p.k_blocks = (K + BK - 1) / BK;
  p.nsplit = nsplit;
  p.passes = nsplit == NNAM_SPLIT_AW ? 3 : (nsplit == NNAM_SPLIT_NONE ? 1 : 2);
  p.f16 = elem == NNAM_ELEM_F16;
  p.act = act;
  p.bias = bias;
  p.out_hi = out_hi;
  p.out_lo = out_lo;
  p.ldo = ldo;

  // tm[0..3] = A hi/lo, W hi/lo (loads); tm[4..5] = output hi/lo (stores: 32-row x 128-byte boxes, clipped at M x N)
  CUtensorMap tm[6];
  int rc;
  if ((rc = encode_tmap_bf16_2d(&tm[0], a_hi, K, M, lda, BK, BM))) return rc;
  const int w_box_rows = pair ? p.bn / 2 : p.bn;  // a CTA of a pair loads half of the W tile
  if ((rc = encode_tmap_bf16_2d(&tm[2], w_hi, K, N, ldw, BK, w_box_rows))) return rc;
  tm[1] = tm[0];
  tm[3] = tm[2];
  if (need_a_lo && (rc = encode_tmap_bf16_2d(&tm[1], a_lo, K, M, lda, BK, BM))) return rc;
  if (need_w_lo && (rc = encode_tmap_bf16_2d(&tm[3], w_lo, K, N, ldw, BK, w_box_rows))) return rc;
  if ((rc = encode_tmap_2d(&tm[4], out_hi, f32_out, N, M, ldo, box_cols, 32))) return rc;
  if (out_kind == NNAM_OUT_BF16_SPLIT) {
    if ((rc = encode_tmap_2d(&tm[5], out_lo, false, N, M, ldo, box_cols, 32))) return rc;
  } else {
    tm[5] = tm[4];
  }

  const int total = p.tiles_m * p.tiles_n;
  if (pair) {
    const int pairs = sm_count() / 2;
    const int grid2 = 2 * (total < pairs ? total : pairs);
    switch (out_kind) {
      case NNAM_OUT_F32: return launch_gemm_2sm<NNAM_OUT_F32>(tm, p, grid2, stream);
      case NNAM_OUT_BF16: return launch_gemm_2sm<NNAM_OUT_BF16>(tm, p, grid2, stream);
      case NNAM_OUT_F16: return launch_gemm_2sm<NNAM_OUT_F16>(tm, p, grid2, stream);
      default: return launch_gemm_2sm<NNAM_OUT_BF16_SPLIT>(tm, p, grid2, stream);
    }
  }
  const int grid = total < sm_count() ? total : sm_count();
  switch (out_kind) {
    case NNAM_OUT_F32: return launch_gemm<NNAM_OUT_F32>(tm, p, grid, stream);
    case NNAM_OUT_BF16: return launch_gemm<NNAM_OUT_BF16>(tm, p, grid, stream);
    case NNAM_OUT_F16: return launch_gemm<NNAM_OUT_F16>(tm, p, grid, stream);
    default: return launch_gemm<NNAM_OUT_BF16_SPLIT>(tm, p, grid, stream);
  }
}

}  // namespace nnam
