// K3 -- persistent recurrence kernel (LSTM family; GRU family below) for a whole layer of a whole shard.
//
// Reference semantics: one time step of L.LSTM / F.lstm per Python loop iteration
// (scripts/common/chainer_networks.py:44-62 driven by predict_folds.py:49-61 and
// evaluateModelForTest.py:67-80): gates = upward(x) + lateral(h); the 4H axis is interleaved
// unit-major / gate-minor [a, i, f, o]; c = tanh(a) s(i) + s(f) c; h = s(o) tanh(c); s(x) = tanh(x/2)/2 + 1/2.
// Here upward(x)+b for ALL frames is one K2 GEMM (gx), and this kernel runs the sequential part.
//
// Decomposition
//   * utterances are sorted by length and cut into batches of NB; a batch is stored time-major ("packed"):
//     row(t, u) = row0 + base[t] + u, active utterances at time t are the prefix u < base[t+1]-base[t];
//   * a GROUP of G = 4H / M_ROWS co-resident CTAs owns one (batch, direction) work item at a time; CTA r keeps the
//     M_ROWS lateral-weight rows [r*M_ROWS, (r+1)*M_ROWS) (= M_ROWS/4 whole units, thanks to Chainer's interleaved
//     layout) resident in shared memory as the A operand of tcgen05.mma (K-major, SWIZZLE_128B, loaded by TMA);
//   * per step: every CTA of the group writes its new h slice twice -- into the layer output rows (the next layer's
//     GEMM input) and into a small slot-indexed EXCHANGE buffer (NB x H per lane, double-buffered by step parity).
//     After the group's release/acquire counter, ONE thread pulls the whole h tile back with KB TMA box loads
//     (hardware swizzle, one mbarrier) -- the first versions issued 4096 16-byte cp.async per step from all threads,
//     which cost ~2 k cycles of load/store-unit issue time (profiles/r01_k3_phase_cycles.md).
//     D[M_ROWS x NB] = W_slice . h^T accumulates in TMEM (3 MMAs passes in bf16x3 mode),
//     each thread owns one gate row (TMEM lane), adds gx, applies the nonlinearity, the 4 gates of a unit are
//     exchanged inside a lane quad with a 4x4 shuffle transpose, the cell state lives in registers for the whole
//     utterance, and the new h slice is written (bf16 hi/lo) straight into the layer output rows -- which is what
//     the other CTAs of the group read next step.  A release/acquire counter per group orders the exchange.
//   * a bidirectional layer is ONE launch: forward and backward items are spread over the groups and run
//     concurrently; the backward direction walks t = len-1-s and addresses rows through base[] the same way.
//   * STREAMS: a step is a latency chain (acquire spin -> L2 round trip for h -> tcgen05.mma -> gates -> fence +
//     publish), not a throughput problem, so one CTA runs S independent batches ("streams") at once against the SAME
//     resident weight slice: stream i owns warps [i*WPS, (i+1)*WPS), its own TMEM columns, operand tile, named
//     barrier and group counter.  While one stream waits on its chain the others issue, which is what hides the
//     latency (profiles/r01_k3_phase_cycles.md).
#include <cooperative_groups.h>
#include <type_traits>

#include "recurrent_common.cuh"

namespace nnam {

__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// One kernel for both cell families.
//   CELL   : NNAM_CELL_LSTM | NNAM_CELL_GRU | NNAM_CELL_PEEPHOLE (a second resident block [0, P_i, P_f, P_o] per unit
//            next to the lateral slice, a second operand tile for the cell state, two exchanges per step)
//   M_ROWS : gate rows per CTA (128, or 64 when the slice would not fit in shared memory)
//   NB     : utterance slots per stream (= N of the MMA)
//   NSPLIT : 1 bf16 | 3 bf16x3
//   KBT    : compile-time H / 64 (0 = runtime H)
//   S, WPS : streams per CTA and warps per stream (4 or 8; with 8 two warps share a TMEM lane quarter and split the slots)
template <int CELL, int M_ROWS, int NB, int NSPLIT, bool FAST_TANH, int KBT, int S, int WPS>
__global__ void __launch_bounds__(S * WPS * 32, 1)
    rnn_seq_kernel(const __grid_constant__ RnnTmaps tmaps, const RnnParams p) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int TPS = WPS * 32;        // threads per stream
  constexpr int SUBS = WPS / 4;        // warps sharing one TMEM lane quarter
  constexpr int NBT = NB / SUBS;       // utterance slots per thread
  constexpr int BASE_SMEM = S >= 4 ? 1024 : 2048;  // steps of a batch whose prefix-sum table is mirrored in smem
  static_assert(NBT % 4 == 0 && NBT >= 4, "a thread owns whole lane-quad groups of 4 slots");
  const int group = blockIdx.x / p.group_ctas;
  const int rank = blockIdx.x % p.group_ctas;
  announce_started(p);
  if (group >= p.n_groups) return;

  const int H = KBT > 0 ? KBT * 64 : p.hidden;
  const int KB = KBT > 0 ? KBT : (H >> 6);
  constexpr int W_BLOCK = M_ROWS * 128;
  constexpr int H_BLOCK = NB * 128;
  constexpr int PLANES = NSPLIT == 3 ? 2 : 1;
  const int tid = threadIdx.x;
  const int stream = tid / TPS;
  const int tid_s = tid - stream * TPS;
  const int warp_s = tid_s >> 5;
  const int lane = tid & 31;
  const int quarter = warp_s & 3;  // == (tid >> 5) & 3: the TMEM lane quarter this warp may read
  const int u_lo = (warp_s >> 2) * NBT;

  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  constexpr bool PEEP = CELL == NNAM_CELL_PEEPHOLE;
  constexpr int SETS = PEEP ? 2 : 1;  // resident weight blocks (lateral [+ peephole]) and operand tiles (h [+ c])
  uint8_t* w_hi_s = smem;
  uint8_t* w_lo_s = w_hi_s + (NSPLIT == 3 ? KB * W_BLOCK : 0);
  uint8_t* pw_hi_s = w_lo_s + KB * W_BLOCK;                      // peephole block (PEEP only)
  uint8_t* pw_lo_s = pw_hi_s + (NSPLIT == 3 ? KB * W_BLOCK : 0);
  uint8_t* tiles = w_hi_s + SETS * PLANES * KB * W_BLOCK;
  uint8_t* h_hi_s = tiles + stream * (SETS * PLANES * KB * H_BLOCK);
  uint8_t* h_lo_s = h_hi_s + (NSPLIT == 3 ? KB * H_BLOCK : 0);
  uint8_t* c_hi_s = h_hi_s + PLANES * KB * H_BLOCK;               // cell-state tile (PEEP only)
  uint8_t* c_lo_s = c_hi_s + (NSPLIT == 3 ? KB * H_BLOCK : 0);
  constexpr int UNITS = M_ROWS / 4;              // hidden units per CTA
  constexpr int STAGE_BYTES = NB * UNITS * 2;     // one plane of this stream's freshly computed slice (NB x UNITS bf16)
  uint8_t* stage_hi = tiles + S * (SETS * PLANES * KB * H_BLOCK) + stream * (PLANES * STAGE_BYTES);
  uint8_t* stage_lo = stage_hi + STAGE_BYTES;
  uint8_t* tail = tiles + S * (SETS * PLANES * KB * H_BLOCK) + S * (PLANES * STAGE_BYTES);
  uint64_t* bar_w = reinterpret_cast<uint64_t*>(tail);
  uint64_t* bar_mma = bar_w + 1 + stream;
  uint64_t* bar_h = bar_w + 1 + S + stream;  // this stream's h tile has landed (TMA complete_tx)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_w + 1 + 2 * S);
  int* s_len = reinterpret_cast<int*>(tmem_slot + 2) + stream * NB;
  int* s_base = reinterpret_cast<int*>(tmem_slot + 2) + S * NB + stream * (BASE_SMEM + 1);
  constexpr int TMEM_COLS = SETS * S * NB < 32 ? 32 : SETS * S * NB;  // D1 (lateral . h) [+ D2 (peephole . c)]
  static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM allocations are powers of two");

  if (tid == 0) {
    mbar_init(bar_w, 1);
    for (int i = 0; i < 2 * S; ++i) mbar_init(bar_w + 1 + i, 1);
    fence_mbar_init();
  }
  if (tid < 32) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot + static_cast<uint32_t>(stream * NB);  // this stream's accumulator columns

  auto stream_sync = [&]() {
    if (S == 1)
      __syncthreads();
    else
      named_bar_sync(1 + stream, TPS);
  };

  // TMEM lane <-> gate row of this CTA's slice.  M_ROWS = 128: lane index = row.  M_ROWS = 64: rows 16q..16q+15
  // sit in lanes 32q..32q+15 (the upper half of every subpartition is unused).
  const bool row_valid = (M_ROWS == 128) || (lane < 16);
  const int my_row = (M_ROWS == 128) ? (quarter * 32 + lane) : (quarter * 16 + (lane & 15));
  const int gate = my_row & 3;                           // LSTM: a, i, f, o   GRU: z, r, candidate, pad
  const int unit = rank * (M_ROWS / 4) + (my_row >> 2);  // hidden unit index in [0, H)
  const int gate_col = rank * M_ROWS + my_row;           // column of gx / row of the lateral matrix
  const uint32_t tmem_lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + u_lo;
  const int f16 = NSPLIT == 1 ? p.f16 : 0;  // the split planes of the fp32-accurate mode are always bf16
  const uint32_t idesc = make_idesc_e16_f32(M_ROWS, NB, f16);
  const uint32_t h_hi_sa = smem_u32(h_hi_s), h_lo_sa = smem_u32(h_lo_s);
  const uint32_t c_hi_sa = smem_u32(c_hi_s), c_lo_sa = smem_u32(c_lo_s);
  const uint32_t tmem_d2 = tmem_base + static_cast<uint32_t>(S * NB);  // second accumulator of this stream (PEEP)
  const bool gru_reset = (p.gru_flags & 1) != 0;
  const int gru_act = (p.gru_flags >> 1) & 3;

  const bool prof_on = p.prof != nullptr && tid == 0;  // thread 0 of stream 0
  long long prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long prof_t = 0;
#define PROF_START() do { if (prof_on) prof_t = clock64(); } while (0)
#define PROF_MARK(i) do { if (prof_on) { const long long now = clock64(); prof_acc[i] += now - prof_t; prof_t = now; } } while (0)

  unsigned int steps_done = 0;  // arrivals of this CTA on the lane counter so far
  uint32_t w_phase = 0, mma_phase = 0, h_phase = 0;
  const int lane_id = group * S + stream;  // (group, stream) = one "lane" of the schedule
  unsigned int* counter = p.counters + lane_id;
  int it = p.group_item_start[lane_id];
  const int it_end = p.group_item_start[lane_id + 1];

  // Wait until every CTA of the group has published its slice of the previous exchange, then pull the whole tile
  // (exchange slot `slot` of this lane) into the swizzled B-operand tile: KB (x planes) TMA box loads, one thread.
  // Only the issuing thread waits; the others go on to prefetch gx and meet it again at the MMA barrier.
  auto group_fetch = [&](int slot, bool into_c = false) {
    if (warp_s == 0) {  // warp-uniform loop, one elected lane issues (keeps the TMA operands in uniform registers)
      const unsigned int target = steps_done * static_cast<unsigned int>(p.group_ctas);
      while (ld_acquire_gpu(counter) < target) {
      }
      if (elect_one()) {
        fence_proxy_async_all();  // the peers' generic-proxy stores -> visible to this async-proxy (TMA) read
        mbar_expect_tx(bar_h, static_cast<uint32_t>(KB * H_BLOCK * PLANES));
        const int row = (lane_id * 4 + slot) * NB;
        uint8_t* t_hi = into_c ? c_hi_s : h_hi_s;
        uint8_t* t_lo = into_c ? c_lo_s : h_lo_s;
        for (int kb = 0; kb < KB; ++kb) {
          tma_load_2d(t_hi + kb * H_BLOCK, &tmaps.x_hi, bar_h, kb * 64, row);
          if (NSPLIT == 3) tma_load_2d(t_lo + kb * H_BLOCK, &tmaps.x_lo, bar_h, kb * 64, row);
        }
      }
      __syncwarp();
    }
  };
  // The CTA barrier orders every thread's slice stores before thread 0's release (cumulativity), so one
  // red.release.gpu publishes the whole slice: no per-thread __threadfence (the pattern of a grid barrier).
  auto group_publish = [&]() {
    stream_sync();
    if (tid_s == 0) red_release_gpu_add(counter, 1u);
    ++steps_done;
  };
  // D[M_ROWS x NB] = W_slice . tile^T (3 passes in bf16x3 mode): issue (one thread) ...
  // mode 0: D1 = lateral . h      mode 1 (PEEP): D1 = lateral . h and D2 = peephole . c      mode 2 (PEEP): D2 = peephole . c
  auto mma_issue = [&](bool via_tma, int mode = 0) {
    if (!via_tma) {  // tile staged by the threads with cp.async (initial-state rows of the stateful API)
      cp_async_wait_all();
      fence_proxy_async_smem();
      stream_sync();
    }
    if (warp_s == 0) {
      // All lanes of the issuing warp run this block and one elected lane issues: under `if (tid == 0)` ptxas wraps
      // every tcgen05.mma in an ELECT waterfall loop, which made the 32 MMAs of a step cost ~55 clocks each to issue.
      if (via_tma) mbar_wait(bar_h, h_phase);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int set = 0; set < SETS; ++set) {
          if (set == 0 && mode == 2) continue;
          if (set == 1 && mode == 0) continue;
          const uint64_t wd_hi = make_sw128_kmajor_desc(smem_u32(set == 0 ? w_hi_s : pw_hi_s));
          const uint64_t wd_lo = make_sw128_kmajor_desc(smem_u32(set == 0 ? w_lo_s : pw_lo_s));
          const uint64_t hd_hi = make_sw128_kmajor_desc(set == 0 ? h_hi_sa : c_hi_sa);
          const uint64_t hd_lo = make_sw128_kmajor_desc(set == 0 ? h_lo_sa : c_lo_sa);
          const uint32_t d = set == 0 ? tmem_base : tmem_d2;
          uint32_t accum = 0;
#pragma unroll
          for (int pass = 0; pass < NSPLIT; ++pass) {
            const uint64_t wa = pass == 2 ? wd_lo : wd_hi;
            const uint64_t ha = pass == 1 ? hd_lo : hd_hi;
            if (KBT > 0) {
#pragma unroll
              for (int kb = 0; kb < KBT; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  umma_bf16(d, wa + ((kb * W_BLOCK + k * 32) >> 4), ha + ((kb * H_BLOCK + k * 32) >> 4), idesc, accum);
                  accum = 1;
                }
            } else {
              for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  umma_bf16(d, wa + ((kb * W_BLOCK + k * 32) >> 4), ha + ((kb * H_BLOCK + k * 32) >> 4), idesc, accum);
                  accum = 1;
                }
            }
          }
        }
        umma_commit(bar_mma);
      }
      __syncwarp();
    }
    if (via_tma) h_phase ^= 1;
  };
  // ... and collect: on return acc[] = my (row, slots) of D
  auto tmem_read = [&](uint32_t addr, float (&acc)[NBT]) {
#pragma unroll
    for (int c0 = 0; c0 < NBT; c0 += (NBT >= 16 ? 16 : NBT)) {
      if (NBT >= 16) {
        uint32_t r[16];
        tmem_ld16(addr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[c0 + j] = __uint_as_float(r[j]);
      } else {
        uint32_t r[8];
        tmem_ld8(addr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < (NBT < 8 ? NBT : 8); ++j) acc[c0 + j] = __uint_as_float(r[j]);
      }
    }
  };
  // wait for the MMAs, then read D2 (PEEP) into acc2 -- the caller reads D1 through mma_collect
  auto mma_wait = [&]() {
    mbar_wait(bar_mma, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
  };
  auto mma_collect = [&](float (&acc)[NBT]) {
    mbar_wait(bar_mma, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
    PROF_MARK(3);
#pragma unroll
    for (int c0 = 0; c0 < NBT; c0 += (NBT >= 16 ? 16 : NBT)) {
      if (NBT >= 16) {
        uint32_t r[16];
        tmem_ld16(tmem_lane_addr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[c0 + j] = __uint_as_float(r[j]);
      } else {
        uint32_t r[8];
        tmem_ld8(tmem_lane_addr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < (NBT < 8 ? NBT : 8); ++j) acc[c0 + j] = __uint_as_float(r[j]);
      }
    }
    tc_fence_before();
    PROF_MARK(4);
  };

  for (int d = 0; d < p.n_dirs; ++d) {
    // ---- (re)load this CTA's slice of the direction's lateral weights; all streams work on one direction at a time
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(bar_w, static_cast<uint32_t>(SETS * KB * W_BLOCK * PLANES));
      for (int kb = 0; kb < KB; ++kb) {
        tma_load_2d(w_hi_s + kb * W_BLOCK, &tmaps.w_hi[d], bar_w, kb * 64, rank * M_ROWS);
        if (NSPLIT == 3) tma_load_2d(w_lo_s + kb * W_BLOCK, &tmaps.w_lo[d], bar_w, kb * 64, rank * M_ROWS);
        if (PEEP) {  // the peephole block travels in the (unused) direction-1 slot of the descriptor
          tma_load_2d(pw_hi_s + kb * W_BLOCK, &tmaps.w_hi[1], bar_w, kb * 64, rank * M_ROWS);
          if (NSPLIT == 3) tma_load_2d(pw_lo_s + kb * W_BLOCK, &tmaps.w_lo[1], bar_w, kb * 64, rank * M_ROWS);
        }
      }
    }
    mbar_wait(bar_w, w_phase);
    w_phase ^= 1;
    const bool bwd = d == 1;
    const int h_col0 = d * H;

    for (; it < it_end && p.item_dir[it] == d; ++it) {
      const int b = p.item_batch[it];
      const long long row0 = p.batch_row0[b];
      const int T = p.batch_steps[b];
      const int nutt = p.batch_nutt[b];
      const int* base = p.base + p.batch_base_off[b];
      const int* len = p.utt_len + b * NB;
      // input projection: fp32 in the fp32-accurate mode, bf16 in bf16 mode (halves the largest HBM stream of a layer)
      using GxT = typename std::conditional<NSPLIT == 3, float, __nv_bfloat16>::type;
      const GxT* gx = reinterpret_cast<const GxT*>(p.gx[d]) + gate_col;
      // Exchange slots are reused by the next item: nobody may write one before every CTA of the group has finished
      // the previous item's last step (its TMA read of a slot may still be in flight).  Inside an item the step's
      // own group_fetch gives that guarantee; across items this extra wait does.
      if (steps_done > 0 && warp_s == 0) {
        const unsigned int target = steps_done * static_cast<unsigned int>(p.group_ctas);
        while (ld_acquire_gpu(counter) < target) {
        }
      }
      stream_sync();  // (also: previous item's readers of s_len / s_base are done)
      if (tid_s < NB) s_len[tid_s] = tid_s < nutt ? len[tid_s] : 0;
      const bool base_in_smem = T <= BASE_SMEM;
      if (base_in_smem)
        for (int i = tid_s; i <= T; i += TPS) s_base[i] = __ldg(base + i);
      stream_sync();
      const int* bp = base_in_smem ? s_base : base;
      const bool has_h0 = p.h0_hi != nullptr;
      const int chunks_per_row = H >> 3;

      // Carried initial state (stateful model(x) surface only): the h0 rows of the active utterances go into the swizzled
      // B-operand tile with 16-byte cp.async chunks, one warp per row.  Every later step gets its tile by TMA.
      auto load_h0_tile = [&](int n_act) {
        for (int u = warp_s; u < n_act; u += WPS) {
          const long long off = (static_cast<long long>(b) * NB + u) * (H * p.n_dirs) + h_col0;
          const uint32_t row_so = static_cast<uint32_t>((u >> 3) * 1024 + (u & 7) * 128);
          for (int c = lane; c < chunks_per_row; c += 32) {
            const uint32_t so = static_cast<uint32_t>((c >> 3) * H_BLOCK) + row_so + (((c & 7) ^ (u & 7)) << 4);
            cp_async_16(h_hi_sa + so, p.h0_hi + off + c * 8);
            if (NSPLIT == 3) cp_async_16(h_lo_sa + so, p.h0_lo + off + c * 8);
          }
        }
      };

      // per-thread recurrent state of (utterance u_lo + 4m + gate, unit): LSTM cell state c, GRU hidden state h
      float st_reg[NBT / 4];
#pragma unroll
      for (int m = 0; m < NBT / 4; ++m) {
        const int u = u_lo + 4 * m + gate;
        st_reg[m] = 0.0f;
        if (row_valid && u < nutt) {
          const long long o = (static_cast<long long>(b) * NB + u) * (H * p.n_dirs) + h_col0 + unit;
          if (CELL == NNAM_CELL_LSTM) {
            if (p.c0 != nullptr) st_reg[m] = p.c0[o];
          } else if (CELL == NNAM_CELL_GRU && has_h0) {
            st_reg[m] = e16_to_f32(reinterpret_cast<const uint16_t*>(p.h0_hi)[o], f16) +
                        (NSPLIT == 3 ? __bfloat162float(p.h0_lo[o]) : 0.0f);
          }
        }
      }
      const float ub = (CELL == NNAM_CELL_GRU && row_valid) ? __ldg(p.u_bias[d] + gate_col) : 0.0f;

      // input projection of my gate row for my utterance slots at step s: independent loads (slots beyond the
      // active prefix re-read its last row, so no load is predicated or dependent on another)
      // Raw loads: the fp32 value (fp32-accurate mode) or the 16-bit pattern (16-bit modes) of my gate row for my utterance
      // slots at step s.  Independent loads (slots beyond the active prefix re-read its last row, so no load is predicated
      // or dependent on another); the 16-bit -> fp32 conversion waits until the values are USED, one step later, so the
      // (DRAM-latency) loads never stall the thread that issued them (they cost ~1.3 k cycles per step when the conversion
      // sat right behind the load, profiles/r02_k3_phase_cycles.md).
      auto load_gx = [&](int s, uint32_t (&dst)[NBT]) {
        const int base_s = bp[s];
        const int n_act = bp[s + 1] - base_s;
#pragma unroll
        for (int j = 0; j < NBT; ++j) {
          const int u = u_lo + j;
          const int uu = u < n_act ? u : n_act - 1;
          const long long row = row0 + (bwd ? bp[s_len[uu] - 1 - s] : base_s) + uu;
          if (NSPLIT == 3)
            dst[j] = __float_as_uint(__ldg(reinterpret_cast<const float*>(gx) + row * p.gx_ld));
          else
            dst[j] = __ldg(reinterpret_cast<const uint16_t*>(gx) + row * p.gx_ld);
        }
      };
      auto gx_val = [&](uint32_t raw) -> float {
        return NSPLIT == 3 ? __uint_as_float(raw) : e16_to_f32(static_cast<uint16_t>(raw), f16);
      };
      // my value for (utterance u, my unit) -> staging tile (utterance-major, UNITS bf16 per row, hi [+ lo] planes)
      auto stage_put = [&](int u, float v) {
        const uint16_t hb = f32_to_e16(v, f16);
        reinterpret_cast<uint16_t*>(stage_hi)[u * UNITS + (my_row >> 2)] = hb;
        if (NSPLIT == 3)
          reinterpret_cast<__nv_bfloat16*>(stage_lo)[u * UNITS + (my_row >> 2)] =
              __float2bfloat16_rn(v - e16_to_f32(hb, 0));
      };
      // staging tile -> rows of `dst` (the layer output / the r*h exchange buffer): 16-byte coalesced stores
      // (dst may be NULL: the r*h product of the GRU reset gate only travels through the exchange buffer)
      auto stage_flush = [&](__nv_bfloat16* dst_hi, __nv_bfloat16* dst_lo, int n_act, int s, int slot) {
        constexpr int CPR = UNITS / 8;  // 16-byte chunks per row
        stream_sync();
        for (int q = tid_s; q < n_act * CPR; q += TPS) {
          const int u = q / CPR, j = q - u * CPR;
          const uint4 v_hi = *reinterpret_cast<const uint4*>(stage_hi + (u * UNITS + j * 8) * 2);
          uint4 v_lo = v_hi;
          if (NSPLIT == 3) v_lo = *reinterpret_cast<const uint4*>(stage_lo + (u * UNITS + j * 8) * 2);
          const long long xoff = (static_cast<long long>(lane_id * 4 + slot) * NB + u) * H + rank * UNITS + j * 8;
          *reinterpret_cast<uint4*>(p.xchg_hi + xoff) = v_hi;
          if (NSPLIT == 3) *reinterpret_cast<uint4*>(p.xchg_lo + xoff) = v_lo;
          if (dst_hi != nullptr) {
            const int t_idx = bwd ? (s_len[u] - 1 - s) : s;
            const long long off = (row0 + bp[t_idx] + u) * p.h_ld + h_col0 + rank * UNITS + j * 8;
            *reinterpret_cast<uint4*>(dst_hi + off) = v_hi;
            if (NSPLIT == 3) *reinterpret_cast<uint4*>(dst_lo + off) = v_lo;
          }
        }
      };

      uint32_t gxr[NBT];
      load_gx(0, gxr);
      for (int s = 0; s < T; ++s) {
        PROF_START();
        const int n_s = bp[s + 1] - bp[s];  // active utterances (prefix of the batch), >= 1
        const bool have_h = (s > 0) || has_h0;
        float acc[NBT];
        uint32_t gxn[NBT];
        if (have_h) {
          if (s > 0)
            group_fetch((s - 1) & 1);  // h of step s-1 sits in exchange slot (s-1) & 1
          else
            load_h0_tile(n_s);
          PROF_MARK(1);
          // the next step's input projection is requested while the h tile is still in flight and lands while the
          // tensor core works (tcgen05.mma issue back-pressures the issuing thread, so it must come last)
          if (s + 1 < T) load_gx(s + 1, gxn);
          PROF_MARK(2);
          mma_issue(s > 0, PEEP ? 1 : 0);
          PROF_MARK(0);
          mma_collect(acc);
        } else {
#pragma unroll
          for (int j = 0; j < NBT; ++j) acc[j] = 0.0f;
          if (s + 1 < T) load_gx(s + 1, gxn);
        }

        if (PEEP) {
          // ---- L.StatefulPeepholeLSTM (chainer_networks.py:103-121): i, f see P_i c, P_f c; o sees P_o c' -- the new
          // cell state has to go round the group before the output gate can be formed: two exchanges per step.
          // The c tile still holds c_{s-1} from phase 2 of the previous step, so phase 1 only fetched h.
          const uint32_t lane_addr2 = tmem_d2 + (static_cast<uint32_t>(quarter * 32) << 16) + u_lo;
          float acc2[NBT];
          if (have_h) {
            tc_fence_after();
            tmem_read(lane_addr2, acc2);
            tc_fence_before();
          } else {
#pragma unroll
            for (int j = 0; j < NBT; ++j) acc2[j] = 0.0f;
          }
          float o_pre[NBT / 4];
#pragma unroll
          for (int m = 0; m < NBT / 4; ++m) {
            o_pre[m] = 0.0f;
            if (u_lo + 4 * m >= n_s) break;  // warp-uniform
            float x[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float v = acc[4 * m + i] + gx_val(gxr[4 * m + i]) + ((gate == 1 || gate == 2) ? acc2[4 * m + i] : 0.0f);
              const float t = tanh_sel<FAST_TANH>(gate == 0 ? v : 0.5f * v);
              x[i] = gate == 0 ? t : (gate == 3 ? v : fmaf(t, 0.5f, 0.5f));  // the output gate stays a pre-activation
            }
            quad_transpose(x, gate);  // x = {a, i, f, o_pre} of utterance u = u_lo + 4m + gate
            const int u = u_lo + 4 * m + gate;
            const float c_new = fmaf(x[0], x[1], x[2] * st_reg[m]);
            o_pre[m] = x[3];
            if (row_valid && u < n_s) {
              st_reg[m] = c_new;
              stage_put(u, c_new);
            }
          }
          stage_flush(nullptr, nullptr, n_s, s, 2 + (s & 1));
          group_publish();  // c' slices are out
          group_fetch(2 + (s & 1), true);
          mma_issue(true, 2);  // D2 = peephole block . c'
          mma_wait();
          tmem_read(lane_addr2, acc2);
          tc_fence_before();
#pragma unroll
          for (int m = 0; m < NBT / 4; ++m) {
            if (u_lo + 4 * m >= n_s) break;
            float y[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) y[i] = gate == 3 ? acc2[4 * m + i] : 0.0f;
            quad_transpose(y, gate);  // y[3] = (P_o c')[unit] of utterance u
            const int u = u_lo + 4 * m + gate;
            const float o = fmaf(tanh_sel<FAST_TANH>(0.5f * (o_pre[m] + y[3])), 0.5f, 0.5f);
            const float h_new = o * tanh_sel<FAST_TANH>(st_reg[m]);
            if (row_valid && u < n_s) stage_put(u, h_new);
          }
          stage_flush(p.h_hi, p.h_lo, n_s, s, s & 1);
          PROF_MARK(5);
        } else if (CELL == NNAM_CELL_LSTM) {
          // ---- gates, quad transpose, cell update  (chainer F.lstm: c = tanh(a) s(i) + s(f) c; h = s(o) tanh(c))
#pragma unroll
          for (int m = 0; m < NBT / 4; ++m) {
            if (u_lo + 4 * m >= n_s) break;  // warp-uniform
            float x[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float v = acc[4 * m + i] + gx_val(gxr[4 * m + i]);
              const float t = tanh_sel<FAST_TANH>(gate == 0 ? v : 0.5f * v);
              x[i] = gate == 0 ? t : fmaf(t, 0.5f, 0.5f);
            }
            quad_transpose(x, gate);  // x = {a, i, f, o} of utterance u = u_lo + 4m + gate
            const int u = u_lo + 4 * m + gate;
            const float c_new = fmaf(x[0], x[1], x[2] * st_reg[m]);
            const float h_new = x[3] * tanh_sel<FAST_TANH>(c_new);
            if (row_valid && u < n_s) {
              st_reg[m] = c_new;
              stage_put(u, h_new);
              if (p.c_out != nullptr && s == s_len[u] - 1)
                p.c_out[(static_cast<long long>(b) * NB + u) * (H * p.n_dirs) + h_col0 + unit] = c_new;
            }
          }
          stage_flush(p.h_hi, p.h_lo, n_s, s, s & 1);
          PROF_MARK(5);
        } else {
          // ---- GRU family (MGRU.py:67-85): U terms and their biases exist only when h does (:70-83)
          const float ubs = have_h ? ub : 0.0f;
          const bool two_phase = gru_reset && have_h;  // r must be applied BEFORE the candidate matmul (:73-74)
          float zp[NBT / 4], hp[NBT / 4];
#pragma unroll
          for (int m = 0; m < NBT / 4; ++m) {
            zp[m] = hp[m] = 0.0f;
            if (u_lo + 4 * m >= n_s) break;
            float x[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              x[i] = gx_val(gxr[4 * m + i]) + ubs + ((two_phase && gate == 2) ? 0.0f : acc[4 * m + i]);
            quad_transpose(x, gate);  // x = {z_pre, r_pre, cand_pre, pad} of utterance u_lo + 4m + gate
            zp[m] = x[0];
            hp[m] = x[2];
            if (two_phase) {
              const int u = u_lo + 4 * m + gate;
              const float r = fmaf(tanh_sel<FAST_TANH>(0.5f * x[1]), 0.5f, 0.5f);
              if (row_valid && u < n_s) stage_put(u, r * st_reg[m]);
            }
          }
          if (two_phase) {
            stage_flush(nullptr, nullptr, n_s, s, 2 + (s & 1));
            group_publish();  // r*h slices are out
            group_fetch(2 + (s & 1));
            mma_issue(true);
            mma_collect(acc);  // row 4j+2 now holds U (r*h)
          }
#pragma unroll
          for (int m = 0; m < NBT / 4; ++m) {
            if (u_lo + 4 * m >= n_s) break;
            float cand = hp[m];
            if (two_phase) {
              float y[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) y[i] = gate == 2 ? acc[4 * m + i] : 0.0f;
              quad_transpose(y, gate);
              cand += y[2];
            }
            const int u = u_lo + 4 * m + gate;
            const float z = fmaf(tanh_sel<FAST_TANH>(0.5f * zp[m]), 0.5f, 0.5f);
            const float hb = gru_act == NNAM_ACT_RELU
                                 ? fmaxf(cand, 0.0f)
                                 : (gru_act == NNAM_ACT_SIGMOID
                                        ? fmaf(tanh_sel<FAST_TANH>(0.5f * cand), 0.5f, 0.5f)
                                        : (gru_act == NNAM_ACT_TANH ? tanh_sel<FAST_TANH>(cand) : cand));
            const float h_new = have_h ? fmaf(z, hb, (1.0f - z) * st_reg[m]) : z * hb;
            if (row_valid && u < n_s) {
              st_reg[m] = h_new;
              stage_put(u, h_new);
            }
          }
          stage_flush(p.h_hi, p.h_lo, n_s, s, s & 1);
        }
        group_publish();
        PROF_MARK(6);
#pragma unroll
        for (int j = 0; j < NBT; ++j) gxr[j] = gxn[j];
      }
    }
  }

  if (prof_on) {
    prof_acc[7] = steps_done;
    for (int i = 0; i < 8; ++i) p.prof[blockIdx.x * 8 + i] = prof_acc[i];
  }
#undef PROF_START
#undef PROF_MARK
  tc_fence_before();
  __syncthreads();
  if (tid < 32) {
    tc_fence_after();
    tmem_dealloc(*tmem_slot, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------ host side
// Kernel instances.  (m_rows, slots per stream, nsplit, KBT (0 = runtime H), streams, warps per stream), in order of
// preference for a given (slots, nsplit): the first one whose shared-memory footprint fits is used.
struct RnnCfg {
  int m, nb, ns, kbt, s, wps;
};
#define NNAM_RNN_INSTANCES(X)                                                                      \
  /* H = 512, bf16: the BASELINE geometry */                                                       \
  X(128, 16, 1, 8, 4, 4) X(128, 32, 1, 8, 1, 16) X(128, 64, 1, 8, 1, 16)                           \
  /* H = 512, bf16x3 (fp32-accurate mode): 64-row slices */                                        \
  X(64, 16, 3, 8, 2, 8) X(64, 32, 3, 8, 1, 8)                                                      \
  /* any H, bf16 */                                                                                \
  X(128, 16, 1, 0, 4, 4) X(128, 32, 1, 0, 2, 8) X(128, 64, 1, 0, 1, 8) X(128, 32, 1, 0, 1, 8)      \
  X(64, 16, 1, 0, 2, 8) X(64, 32, 1, 0, 1, 8) X(64, 16, 1, 0, 1, 8)                                \
  /* any H, bf16x3 */                                                                              \
  X(128, 16, 3, 0, 2, 8) X(128, 32, 3, 0, 1, 8) X(64, 16, 3, 0, 2, 8) X(64, 32, 3, 0, 1, 8)        \
  X(64, 16, 3, 0, 1, 8)

// PeepholeLSTM: lateral slice + peephole block + two operand tiles must fit, so 64-row slices only
#define NNAM_PEEP_INSTANCES(X) X(64, 32, 1, 8, 1, 8) X(64, 32, 1, 0, 1, 8) X(64, 16, 1, 0, 1, 8) X(64, 32, 3, 0, 1, 8) X(64, 16, 3, 0, 1, 8)

static const RnnCfg kPeepCfgs[] = {
#define X(M, NBV, NS, KBTV, SV, WPSV) {M, NBV, NS, KBTV, SV, WPSV},
    NNAM_PEEP_INSTANCES(X)
#undef X
};

static const RnnCfg kRnnCfgs[] = {
#define X(M, NBV, NS, KBTV, SV, WPSV) {M, NBV, NS, KBTV, SV, WPSV},
    NNAM_RNN_INSTANCES(X)
#undef X
};

static size_t rnn_smem_bytes(const RnnCfg& c, int hidden, int cell) {
  const size_t kb = hidden / 64;
  const size_t planes = c.ns == 3 ? 2 : 1;
  const size_t sets = cell == NNAM_CELL_PEEPHOLE ? 2 : 1;  // lateral [+ peephole] blocks, h [+ c] tiles
  const size_t base_smem = c.s >= 4 ? 1024 : 2048;
  const size_t stage = planes * static_cast<size_t>(c.s) * c.nb * (c.m / 4) * 2;
  return sets * kb * planes * (static_cast<size_t>(c.m) * 128 + static_cast<size_t>(c.s) * c.nb * 128) + stage +
         8 * (1 + 2 * c.s) + 16 + static_cast<size_t>(c.s) * (c.nb + base_smem + 1) * 4 + 1024;
}

// The instance used for (hidden, slots per stream, precision), or nullptr.  single_stream: only one-stream instances
// qualify (the descriptor was planned for the multicast kernel, which runs one stream, but carried state rules it out).
static const RnnCfg* rnn_pick_cfg(int cell, int hidden, int nb, int nsplit, bool single_stream = false) {
  const int kbt = hidden / 64;
  // the opt-in cluster experiment replaces the single-stream instance
  const bool single = single_stream || ((4 * hidden) % 128 == 0 && rnn_cluster_groups(cell, hidden, nb, nsplit) > 0);
  const RnnCfg* list = cell == NNAM_CELL_PEEPHOLE ? kPeepCfgs : kRnnCfgs;
  const size_t n_list = cell == NNAM_CELL_PEEPHOLE ? sizeof(kPeepCfgs) / sizeof(RnnCfg) : sizeof(kRnnCfgs) / sizeof(RnnCfg);
  for (size_t i = 0; i < n_list; ++i) {
    const RnnCfg& c = list[i];
    if (c.nb != nb || c.ns != nsplit || (c.kbt != 0 && c.kbt != kbt)) continue;
    if (single && c.s != 1) continue;
    if ((4 * hidden) % c.m) continue;
    if (rnn_smem_bytes(c, hidden, cell) > 227 * 1024) continue;
    if (sm_count() < 4 * hidden / c.m) continue;
    return &c;
  }
  return nullptr;
}

template <int CELL, int M_ROWS, int NB, int NSPLIT, int KBT, int S, int WPS>
static int launch_rnn_instance(const RnnTmaps& tm, const RnnParams& p, int grid, size_t smem, cudaStream_t stream) {
  // bf16 mode: MUFU tanh; fp32-accurate mode: tanhf
  auto kern = rnn_seq_kernel<CELL, M_ROWS, NB, NSPLIT, NSPLIT == 1, KBT, S, WPS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return set_cuda_error(e, "rnn: cudaFuncSetAttribute");
  void* args[] = {const_cast<RnnTmaps*>(&tm), const_cast<RnnParams*>(&p)};
  // cooperative launch: every CTA of a group must be co-resident (they wait on one another every step)
  e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kern), dim3(grid), dim3(S * WPS * 32), args, smem, stream);
  if (e != cudaSuccess) return set_cuda_error(e, "rnn: cudaLaunchCooperativeKernel");
  return NNAM_OK;
}

static int launch_rnn(int cell, const RnnCfg& c, const RnnTmaps& tm, const RnnParams& p, int grid, size_t smem,
                      cudaStream_t stream) {
  if (cell == NNAM_CELL_PEEPHOLE) {
#define X(M, NBV, NS, KBTV, SV, WPSV)                                                        \
  if (c.m == M && c.nb == NBV && c.ns == NS && c.kbt == KBTV && c.s == SV && c.wps == WPSV) \
    return launch_rnn_instance<NNAM_CELL_PEEPHOLE, M, NBV, NS, KBTV, SV, WPSV>(tm, p, grid, smem, stream);
    NNAM_PEEP_INSTANCES(X)
#undef X
    return set_error(NNAM_ERR_UNSUPPORTED, "rnn: no peephole kernel instance for this configuration");
  }
#define X(M, NBV, NS, KBTV, SV, WPSV)                                                                         \
  if (c.m == M && c.nb == NBV && c.ns == NS && c.kbt == KBTV && c.s == SV && c.wps == WPSV)                  \
    return cell == NNAM_CELL_GRU ? launch_rnn_instance<NNAM_CELL_GRU, M, NBV, NS, KBTV, SV, WPSV>(tm, p, grid, smem, stream) \
                                 : launch_rnn_instance<NNAM_CELL_LSTM, M, NBV, NS, KBTV, SV, WPSV>(tm, p, grid, smem, stream);
  NNAM_RNN_INSTANCES(X)
#undef X
  return set_error(NNAM_ERR_UNSUPPORTED, "rnn: no kernel instance for this configuration");
}

int rnn_seq(const NnamRnnDesc* d, cudaStream_t stream) {
  if (d == nullptr) return set_error(NNAM_ERR_ARG, "rnn: NULL descriptor");
  if (d->cell != NNAM_CELL_LSTM && d->cell != NNAM_CELL_GRU && d->cell != NNAM_CELL_PEEPHOLE)
    return set_error(NNAM_ERR_UNSUPPORTED, "rnn: cell kind %d not implemented", d->cell);
  if (d->cell == NNAM_CELL_PEEPHOLE && (d->n_dirs != 1 || d->h0_hi || d->c0 || d->c_out || !d->w_hi[1]))
    return set_error(NNAM_ERR_ARG, "rnn: the peephole cell is unidirectional, takes no carried state here, and needs "
                     "its peephole block in w_hi[1]");
  const int H = d->hidden;
  if (H <= 0 || H % 64) return set_error(NNAM_ERR_UNSUPPORTED, "rnn: hidden size must be a multiple of 64 (got %d)", H);
  if (d->n_dirs != 1 && d->n_dirs != 2) return set_error(NNAM_ERR_ARG, "rnn: n_dirs must be 1 or 2");
  if (d->batch != 16 && d->batch != 32 && d->batch != 64 && d->batch != 128)
    return set_error(NNAM_ERR_ARG, "rnn: batch must be 16, 32, 64 or 128");
  if (d->nsplit != 1 && d->nsplit != 3) return set_error(NNAM_ERR_ARG, "rnn: nsplit must be 1 or 3");
  if (d->elem != NNAM_ELEM_BF16 && d->elem != NNAM_ELEM_F16) return set_error(NNAM_ERR_ARG, "rnn: unknown element type %d", d->elem);
  if (d->elem == NNAM_ELEM_F16 && d->nsplit != 1) return set_error(NNAM_ERR_ARG, "rnn: fp16 operands are a single-pass mode (nsplit 1)");
  if (d->n_items <= 0) return NNAM_OK;
  if (d->nsplit == 3 && (d->h_lo == nullptr)) return set_error(NNAM_ERR_ARG, "rnn: bf16x3 needs h_lo");
  if (d->h_ld % 8 || d->w_ld % 8) return set_error(NNAM_ERR_ARG, "rnn: h_ld and w_ld must be multiples of 8");
  // 128 slots per batch: the "wide" kernels (utterances on the MMA's M axis, h streamed through a TMA ring).  The GRU
  // family variant takes gate-blocked rows without padding: 32 * n_gates rows per CTA (recurrent_wide_gru.cu)
  static const RnnCfg kWideCfg1 = {128, 128, 1, 0, 1, 16};
  static const RnnCfg kWideCfg2 = {128, 128, 1, 0, 2, 8};
  static const RnnCfg kWideCfg3 = {128, 128, 1, 0, 3, 4};
  static const RnnCfg kWideGru3 = {96, 128, 1, 0, 2, 8};
  static const RnnCfg kWideGru2 = {64, 128, 1, 0, 2, 8};
  const bool wide = d->batch == 128;
  const bool wide_gru = wide && d->cell == NNAM_CELL_GRU;
  const int gru_gates = (d->flags & 1) ? 3 : 2;
  const RnnCfg& kWideCfg = wide_gru ? (gru_gates == 3 ? kWideGru3 : kWideGru2)
                                    : (rnn_wide_streams() == 3 ? kWideCfg3
                                                               : (rnn_wide_streams() == 2 ? kWideCfg2 : kWideCfg1));
  const int gate_rows = wide_gru ? gru_gates * H : 4 * H;
  if (wide && (d->h0_hi || d->c0 || d->c_out ||
               !(wide_gru ? rnn_wide_gru_applies(H, d->nsplit, gru_gates)
                          : rnn_wide_applies(d->cell, H, d->batch, d->nsplit))))
    return set_error(NNAM_ERR_UNSUPPORTED, "rnn: 128 slots per batch are available for LSTM and the GRU family in "
                     "bf16 mode without carried state only");
  if (wide && (d->h_ld % 16 || d->gx_ld % 16 || (reinterpret_cast<uintptr_t>(d->h_hi) & 31) ||
               (reinterpret_cast<uintptr_t>(d->xchg_hi) & 31) || (reinterpret_cast<uintptr_t>(d->gx[0]) & 31) ||
               (d->n_dirs == 2 && (reinterpret_cast<uintptr_t>(d->gx[1]) & 31))))
    return set_error(NNAM_ERR_ARG, "rnn: 128 slots per batch need 32-byte aligned gx / h / exchange buffers and "
                     "gx_ld, h_ld multiples of 16 (256-bit accesses)");
  // nnam_rnn_plan promises one stream wherever the multicast kernel applies; with carried state that kernel is ruled out
  // and the counter-based kernel must run the same single-stream schedule
  const bool carried = d->h0_hi || d->c0 || d->c_out;
  const bool mc_planned = !wide && rnn_mc_groups(d->cell, H, d->batch, d->nsplit) > 0;
  const RnnCfg* cfg = wide ? &kWideCfg : rnn_pick_cfg(d->cell, H, d->batch, d->nsplit, mc_planned && carried);
  if (!cfg)
    return set_error(NNAM_ERR_UNSUPPORTED,
                     "rnn: no kernel instance holds the lateral weights of H=%d in shared memory with %d slots per "
                     "stream in this precision mode", H, d->batch);
  const int m_rows = cfg->m;
  const int G = gate_rows / m_rows;
  const int max_groups = sm_count() / G;
  if (d->n_groups < 1 || d->n_groups > max_groups)
    return set_error(NNAM_ERR_ARG, "rnn: n_groups %d outside [1, %d]", d->n_groups, max_groups);
  if (d->streams != (mc_planned ? 1 : cfg->s))
    return set_error(NNAM_ERR_ARG, "rnn: descriptor built for %d streams per group, this configuration runs %d "
                     "(ask nnam_rnn_plan)", d->streams, mc_planned ? 1 : cfg->s);
  // experimental DSMEM variant: groups are independent clusters (no carried state through this path)
  const bool use_cluster = m_rows == 128 && cfg->s == 1 && !d->h0_hi && !d->c0 && !d->c_out &&
                           rnn_cluster_groups(d->cell, H, d->batch, d->nsplit) > 0;
  // cluster + TMA-multicast exchange (recurrent_mc.cu): the low-latency kernel for 32-slot batches without carried state
  const int mc_groups = (!wide && !d->h0_hi && !d->c0 && !d->c_out) ? rnn_mc_groups(d->cell, H, d->batch, d->nsplit) : 0;
  const bool use_mc = mc_groups > 0 && d->streams == 1 && d->n_groups <= mc_groups;

  RnnTmaps tm;
  int rc;
  const int n_blocks = d->cell == NNAM_CELL_PEEPHOLE ? 2 : d->n_dirs;  // peephole: [1] is the peephole block
  for (int k = 0; k < n_blocks; ++k) {
    if ((rc = encode_tmap_bf16_2d(&tm.w_hi[k], d->w_hi[k], H, gate_rows, d->w_ld, 64, m_rows))) return rc;
    if (d->nsplit == 3) {
      if (!d->w_lo[k]) return set_error(NNAM_ERR_ARG, "rnn: bf16x3 needs w_lo");
      if ((rc = encode_tmap_bf16_2d(&tm.w_lo[k], d->w_lo[k], H, gate_rows, d->w_ld, 64, m_rows))) return rc;
    } else {
      tm.w_lo[k] = tm.w_hi[k];
    }
  }
  if (n_blocks == 1) {
    tm.w_hi[1] = tm.w_hi[0];
    tm.w_lo[1] = tm.w_lo[0];
  }
  if (!d->xchg_hi || (d->nsplit == 3 && !d->xchg_lo))
    return set_error(NNAM_ERR_ARG, "rnn: the exchange buffer (n_groups * streams * 4 * batch rows of H bf16) is missing");
  const unsigned long long x_rows = static_cast<unsigned long long>(d->n_groups) * cfg->s * 4 * d->batch;
  if ((rc = encode_tmap_bf16_2d(&tm.x_hi, d->xchg_hi, H, x_rows, H, 64, d->batch))) return rc;
  if (d->nsplit == 3) {
    if ((rc = encode_tmap_bf16_2d(&tm.x_lo, d->xchg_lo, H, x_rows, H, 64, d->batch))) return rc;
  } else {
    tm.x_lo = tm.x_hi;
  }
  RnnParams p;
  p.hidden = H;
  p.n_dirs = d->n_dirs;
  p.n_groups = d->n_groups;
  p.group_ctas = G;
  p.gx_ld = d->gx_ld;
  p.h_ld = d->h_ld;
  for (int k = 0; k < 2; ++k) {
    p.gx[k] = d->gx[k];
    p.u_bias[k] = d->u_bias[k];
  }
  p.h_hi = static_cast<__nv_bfloat16*>(d->h_hi);
  p.h_lo = static_cast<__nv_bfloat16*>(d->h_lo);
  p.xchg_hi = static_cast<__nv_bfloat16*>(d->xchg_hi);
  p.xchg_lo = static_cast<__nv_bfloat16*>(d->xchg_lo);
  if (d->cell == NNAM_CELL_GRU) {
    for (int k = 0; k < d->n_dirs; ++k)
      if (!d->u_bias[k]) return set_error(NNAM_ERR_ARG, "rnn: GRU cells need u_bias");
  }
  p.item_batch = d->item_batch;
  p.item_dir = d->item_dir;
  p.group_item_start = d->group_item_start;
  p.batch_row0 = d->batch_row0;
  p.batch_steps = d->batch_steps;
  p.batch_nutt = d->batch_nutt;
  p.batch_base_off = d->batch_base_off;
  p.base = d->base;
  p.utt_len = d->utt_len;
  p.h0_hi = static_cast<const __nv_bfloat16*>(d->h0_hi);
  p.h0_lo = static_cast<const __nv_bfloat16*>(d->h0_lo);
  p.c0 = d->c0;
  p.c_out = d->c_out;
  p.counters = d->counters;
  p.gru_flags = d->flags;
  p.f16 = d->elem == NNAM_ELEM_F16;
  p.prof = static_cast<long long*>(d->debug_cycles);
  p.started = d->started;
  p.started_tag = d->started_tag;
  if (p.h0_hi && d->nsplit == 3 && !p.h0_lo) return set_error(NNAM_ERR_ARG, "rnn: bf16x3 needs h0_lo with h0_hi");

  if (use_mc) return rnn_mc_launch(d->cell, tm, p, G, H, stream);
  if (use_cluster) return rnn_cluster_launch(tm, p, G, H, stream);
  if (wide) {
    cudaError_t ew = cudaMemsetAsync(d->counters, 0, sizeof(unsigned int) * d->n_groups * cfg->s, stream);
    if (ew != cudaSuccess) return set_cuda_error(ew, "rnn: cudaMemsetAsync");
    if (wide_gru) return rnn_wide_gru_launch(tm, p, H, gru_gates, stream);
    return rnn_wide_launch(tm, p, H, stream);
  }
  cudaError_t e = cudaMemsetAsync(d->counters, 0, sizeof(unsigned int) * d->n_groups * cfg->s, stream);
  if (e != cudaSuccess) return set_cuda_error(e, "rnn: cudaMemsetAsync");
  return launch_rnn(d->cell, *cfg, tm, p, d->n_groups * G, rnn_smem_bytes(*cfg, H, d->cell), stream);
}

int rnn_plan(int cell, int hidden, int batch, int nsplit, int* group_ctas, int* max_groups, int* step_cycles,
             int* streams) {
  if (cell != NNAM_CELL_LSTM && cell != NNAM_CELL_GRU && cell != NNAM_CELL_PEEPHOLE)
    return set_error(NNAM_ERR_UNSUPPORTED, "rnn: cell kind %d not implemented", cell);
  if (hidden <= 0 || hidden % 64) return set_error(NNAM_ERR_UNSUPPORTED, "rnn: hidden size must be a multiple of 64");
  if (batch == 128 && cell == NNAM_CELL_GRU) {
    // gate-blocked rows, 32 units per CTA (recurrent_wide_gru.cu); figures for the reset-gate variant (two exchanges)
    if (!rnn_wide_gru_applies(hidden, nsplit, 3))
      return set_error(NNAM_ERR_UNSUPPORTED, "rnn: 128 slots per batch need bf16 mode and a slice that fits");
    *group_ctas = hidden / 32;
    *max_groups = sm_count() / *group_ctas;
    if (step_cycles) *step_cycles = 21500;  // measured, reset-gate variant (11 k without reset gate)
    if (streams) *streams = 2;
    return NNAM_OK;
  }
  if (batch == 128) {
    if (!rnn_wide_applies(cell, hidden, batch, nsplit))
      return set_error(NNAM_ERR_UNSUPPORTED, "rnn: 128 slots per batch are available for LSTM and the GRU family in "
                       "bf16 mode only");
    *group_ctas = 4 * hidden / 128;
    *max_groups = sm_count() / *group_ctas;
    // measured, profiles/r01_k3_phase_cycles.md: per step of ONE stream while all streams of the group are busy
    if (step_cycles) *step_cycles = rnn_wide_streams() == 3 ? 15000 : (rnn_wide_streams() == 2 ? 13800 : 10300);
    if (streams) *streams = rnn_wide_streams();
    return NNAM_OK;
  }
  const RnnCfg* cfg = rnn_pick_cfg(cell, hidden, batch, nsplit);
  if (!cfg)
    return set_error(NNAM_ERR_UNSUPPORTED,
                     "rnn: no kernel instance holds the lateral weights of H=%d in shared memory with %d slots per "
                     "stream in this precision mode", hidden, batch);
  *group_ctas = 4 * hidden / cfg->m;
  *max_groups = sm_count() / *group_ctas;
  // measured SM cycles per recurrence step of ONE stream while all S streams of the CTA are busy
  // (profiles/r01_k3_phase_cycles.md); the host uses it to choose the batch width
  int cycles = cfg->s == 4 ? 12800 : (cfg->s == 2 ? 9500 : (batch == 64 ? 7900 : 6500));
  if (nsplit == 3) cycles = cycles * 7 / 5;
  if (cell == NNAM_CELL_GRU) cycles = cycles * 2;  // measured with the reset gate: 13.0 k (32 slots), 15.2 k (64 slots)
  if (cell == NNAM_CELL_PEEPHOLE) cycles = cycles * 3 / 2;
  const int cl = (cfg->m == 128 && cfg->s == 1) ? rnn_cluster_groups(cell, hidden, batch, nsplit) : 0;
  if (cl > 0) {
    if (cl < *max_groups) *max_groups = cl;
    cycles = 7000;
  }
  int n_streams = cfg->s;
  const int mc = rnn_mc_groups(cell, hidden, batch, nsplit);
  if (mc > 0) {  // cluster + multicast kernel: fewer resident groups (clusters of 16 CTAs), shorter step, one stream
    *group_ctas = 4 * hidden / 128;
    *max_groups = mc;
    n_streams = 1;
    // measured, profiles/r02_k3_phase_cycles.md
    cycles = 4300;
  }
  if (step_cycles) *step_cycles = cycles;
  if (streams) *streams = n_streams;
  return NNAM_OK;
}

// SM cycles per step of a stream whose sibling streams in the CTA group are idle (<= the all-busy figure of rnn_plan):
// the host's lane assignment uses the pair to cost a group as solo * longest lane + (busy - solo) * the other lane.
int rnn_solo_step_cycles(int cell, int hidden, int batch, int nsplit, int* cycles) {
  int g = 0, m = 0, c = 0, s = 0;
  const int rc = rnn_plan(cell, hidden, batch, nsplit, &g, &m, &c, &s);
  if (rc) return rc;
  if (batch == 128 && s >= 2) c = cell == NNAM_CELL_GRU ? 17700 : 11500;  // measured: 10.7 k with one group running, profiles/r01_k3_phase_cycles.md
  *cycles = c;
  return NNAM_OK;
}

}  // namespace nnam
