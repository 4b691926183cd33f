/* nnam_b200 -- C ABI of the B200-native network-output hot path.
 *
 * The reference (OrcusCZ/NNAcousticModeling) has NO FFI/plugin interface: the path sits behind plain
 * Python call surfaces (SURVEY.md 8b).  Each entry point below therefore cites the reference Python
 * symbol whose arithmetic it replaces; the Python host layer (nnacousticmodeling_b200/) binds these
 * with ctypes and keeps the reference's names (get_nn, MLP, LSTM, predict, ...).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns all buffers, kernels never allocate; `stream` is a cudaStream_t passed as void*;
 *   - every function returns 0 on success or a negative NNAM_ERR_* code; nnam_last_error() returns a
 *     thread-local human-readable message for the last failure;
 *   - re-entrant across streams and devices (one host thread per GPU is the intended use).
 *   - 16-bit matrices (bf16 or fp16, see NNAM_ELEM_*) are row-major with a leading dimension in ELEMENTS that is a
 *     multiple of 8.
 */
#ifndef NNAM_B200_H_
#define NNAM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNAM_ABI_VERSION 4

/* error codes */
#define NNAM_OK 0
#define NNAM_ERR_ARG (-1)     /* invalid argument (message says which) */
#define NNAM_ERR_CUDA (-2)    /* CUDA runtime / driver error */
#define NNAM_ERR_UNSUPPORTED (-3)

/* activations (chainer_networks.py: F.relu / F.sigmoid / F.tanh chosen in predict_folds.py:144-152) */
#define NNAM_ACT_NONE 0
#define NNAM_ACT_RELU 1
#define NNAM_ACT_SIGMOID 2 /* Chainer formulation tanh(x/2)/2 + 1/2 */
#define NNAM_ACT_TANH 3

/* output kinds of kernels that can emit GEMM operands */
#define NNAM_OUT_BF16 0       /* bf16 (hi only) */
#define NNAM_OUT_BF16_SPLIT 1 /* bf16 hi + bf16 lo, hi + lo ~= fp32 value (16 mantissa bits) */
#define NNAM_OUT_F32 2        /* fp32 */
#define NNAM_OUT_F16 3        /* IEEE fp16 (hi only), saturating conversion */

/* 16-bit element type of GEMM / recurrence operands.  Both feed tcgen05.mma kind::f16 at the same rate; fp16 carries an
 * 11-bit significand against bf16's 8 (8x smaller rounding error per operand) over a narrower range (|v| <= 65504,
 * conversions saturate), which is what lets the single-pass mode meet north_star's >= 99.5 % frame-argmax agreement.
 * The hi/lo split planes of the fp32-accurate mode are always bf16.  */
#define NNAM_ELEM_BF16 0
#define NNAM_ELEM_F16 1

/* operand passes of nnam_linear_bias_act (`nsplit`): A = A_hi + A_lo, W = W_hi + W_lo, fp32 accumulation in TMEM */
#define NNAM_SPLIT_NONE 1 /* A_hi.W_hi                              (one tensor pass) */
#define NNAM_SPLIT_A 2    /* A_hi.W_hi + A_lo.W_hi                  (activations carry 16 mantissa bits; needs a_lo) */
#define NNAM_SPLIT_AW 3   /* A_hi.W_hi + A_hi.W_lo + A_lo.W_hi      ("bf16x3", fp32-accurate; needs a_lo and w_lo) */
#define NNAM_SPLIT_W 4    /* A_hi.W_hi + A_hi.W_lo                  (weights carry 16 mantissa bits; needs w_lo) */

/* recurrent cell kinds for nnam_rnn_seq */
#define NNAM_CELL_LSTM 0     /* L.LSTM / L.StatefulZoneoutLSTM at inference (chainer_networks.py:44-101) */
#define NNAM_CELL_GRU 1      /* MGRU.py:67-85 family: flags choose reset gate and activation */
#define NNAM_CELL_PEEPHOLE 2 /* L.StatefulPeepholeLSTM (chainer_networks.py:103-121) */

int nnam_abi_version(void);
const char* nnam_last_error(void);
/* Number of SMs of the current device (grid sizing), or a negative error. */
int nnam_sm_count(void);

/* K1 -- context splice + Kaldi feature transform (+ i-vector append), one pass.
 * Replaces prepareBatch (scripts/util/kw_nn_utils.py:19-43) == splicing (scripts/util/kw_utils.py:24-36),
 * applyKaldiFeatureTransform (kw_nn_utils.py:13-17) and the i-vector concatenate (evaluate.py:169-171,
 * train.py:255-258) in the order splice -> transform -> concat.
 *
 *   out[f - f0][w*dim + d] = (x[clamp(f + w - splice, 0, n_total-1)][d] + add_shift[w*dim+d]) * rescale[w*dim+d]
 *   out[f - f0][winlen*dim + j] = ivec[f][j]
 *
 * for f in [f0, f1).  The clamp is at the ends of the WHOLE array (reference quirk Q1), so a shard is
 * described in global frame coordinates: `x` points at global row `x_row0` and holds rows
 * [x_row0, x_row0 + x_rows) which must cover [max(f0-splice,0), min(f1+splice, n_total)).  `ivec` (may be
 * NULL, ivec_dim 0) points at global row f0.  add_shift/rescale may both be NULL (no transform); the
 * add and the multiply are separately rounded (__fadd_rn/__fmul_rn), so fp32 output is bit-exact.
 * out_kind F32: out_hi is float[(f1-f0), ldo]; BF16: out_hi bf16; BF16_SPLIT: out_hi + out_lo.  Columns
 * [winlen*dim + ivec_dim, ldo) are zero-filled.  */
int nnam_splice_transform(const float* x, long long x_row0, long long x_rows, long long n_total, int dim,
                          int splice, const float* add_shift, const float* rescale, const float* ivec,
                          int ivec_dim, long long f0, long long f1, void* out_hi, void* out_lo, long long ldo,
                          int out_kind, void* stream);

/* fp32 -> bf16 (hi) or bf16 hi/lo split of a row-major matrix, zero-padding columns [cols, ldd).
 * Used to stage weights (Chainer npz, (out,in) fp32) and already-spliced inputs of model(x).  */
int nnam_convert_f32(const float* src, long long rows, int cols, long long lds, void* dst_hi, void* dst_lo,
                     long long ldd, int out_kind, void* stream);

/* K2 -- out = act(A . W^T + bias): every L.Linear of chainer_networks.py (F.linear: x.dot(W.T) + b) and the
 * batched `upward` / `W_*` projections of the recurrent links.  A [M,K] (lda), W [N,K] (ldw) bf16 K-major.
 * nsplit: NNAM_SPLIT_* (1 = single pass; 3 = bf16x3 fp32-accurate mode, needs a_lo, w_lo; 2 / 4 = only the activations /
 * only the weights split).  elem: NNAM_ELEM_* of a_hi / w_hi (split passes need NNAM_ELEM_BF16).  bias may be NULL.
 * out_kind selects bf16 / fp16 / bf16 split / fp32 output with leading dimension ldo >= N (rows 16-byte aligned); only
 * columns [0, N) are written.  A may be a column slice of a wider matrix (pointer offset + lda): that is how the
 * TDNN's valid 1 x k convolutions (chainer_networks.py:38-42) run on this kernel without an im2col copy.  */
int nnam_linear_bias_act(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                         long long ldw, const float* bias, void* out_hi, void* out_lo, long long ldo, int M,
                         int N, int K, int act, int out_kind, int nsplit, int elem, void* stream);

/* K4 -- fused ensemble mean -> RPL4 -> minus log-prior -> log-softmax head.
 * Replaces `y - logsum(y, axis=1)` (predict_folds.py:57,88; kw_utils.py:38-43), `y = y - ap` +
 * log-softmax (evaluateModelForTest.py:75-77,110-112), NNWithRPL.__call__ (evaluate.py:35-51), RPL4
 * (RPL.py:68-74) and the dev-mode fold averaging (predict_folds.py:199-219).
 *
 *   h = sum_k weights[k] * (pre_normalize ? log_softmax(logits[k]) : logits[k])
 *   if rpl_w: x = log_softmax(h); g = x + x*rpl_w + rpl_b; h = logaddexp(g, rpl_lb)
 *   if prior: h = h - prior_scale * prior
 *   out = h - logsumexp(h)            (skipped when final_normalize == 0)
 *
 * logits: array of n_inputs DEVICE pointers stored in HOST memory (logits_host[k] -> float[rows, ld_in]).
 * out: float[rows, ld_out] (ld_out == n_classes gives the reference's contiguous (N, C) layout).  */
int nnam_head(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
              int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
              float prior_scale, int final_normalize, float* out, long long ld_out, long long rows,
              int n_classes, void* stream);

/* nnam_head with a scatter map: logits row r is written to out row out_row_map[r]; an entry of -1 drops the row and an
 * entry -2 - q fills out row q with zeros.  Used by the recurrent path, whose rows are time-major "packed"; the zero
 * rows reproduce the reference's unwritten last `timedelay` frames (predict_folds.py:50,60-61, quirk Q4) without a
 * separate pass over the output.  */
int nnam_head_scatter(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                      int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb,
                      const float* prior, float prior_scale, int final_normalize, float* out, long long ld_out,
                      long long rows, int n_classes, const int* out_row_map, void* stream);

/* nnam_head_scatter (out_row_map may be NULL) with the COMPACT TRANSFER FORMAT as output instead of float32 rows:
 *   row_ref[q] = max_c y[q][c]          out16[q][c] = fp16(y[q][c] - row_ref[q])        (q = output row)
 * out16: IEEE fp16 [rows_out, ld16] with ld16 % 8 == 0 (16-byte aligned rows), row_ref: float[rows_out].  Half the bytes
 * of the float32 matrix cross PCIe -- the end-to-end bottleneck of the path (7,636 B per frame) -- and
 * nnam_widen_f16_host rebuilds the reference's (N, C) float32 layout on the host.  What it costs: an entry keeps 11
 * significant bits of its DISTANCE from the row maximum (|error| <= 2^-12 * |y - max|, i.e. <= 4e-3 at a distance of
 * 16), so the best-scoring classes -- the ones the decoder compares -- keep float32-like resolution and the argmax is
 * unchanged.  Used in the 16-bit precision modes (tolerance 5e-2); the fp32-accurate mode transfers float32.  */
int nnam_head_f16(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                  int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
                  float prior_scale, int final_normalize, void* out16, long long ld16, float* row_ref, long long rows,
                  int n_classes, const int* out_row_map, void* stream);

/* nnam_head_scatter scored against frame targets instead of writing rows: with y[q] the row nnam_head_scatter would write
 * to output row q (same arguments, same kernel choice, the same device code),
 *   nll[q]  = -y[q][targets[q]], or 0 when targets[q] == -1 (Chainer's ignore_label)
 *   pred[q] = argmax_c y[q][c], the lowest column on ties
 * An out_row_map entry -1 drops the row (nothing is written) and -2 - q writes nll[q] = 0, pred[q] = -1 (the zero rows of
 * quirk Q4 are no network output).  targets: int[rows_out] in [-1, n_classes) (the host validates them), nll:
 * float[rows_out], pred: int[rows_out].  8 B per row leave the kernel instead of 4 * n_classes.
 * Replaces what training reports per frame (recalled from Chainer upstream, †): F.softmax_cross_entropy (the mean of
 * nll over targets != -1) and F.accuracy, behind L.Classifier as train.py uses it (SURVEY section 2, rows 11-13).  */
int nnam_head_score(const float* const* logits_host, const float* weights_host, int n_inputs, long long ld_in,
                    int pre_normalize, const float* rpl_w, const float* rpl_b, const float* rpl_lb, const float* prior,
                    float prior_scale, int final_normalize, const int* targets, float* nll, int* pred, long long rows,
                    int n_classes, const int* out_row_map, void* stream);

/* K2 + K4 fused for ONE net without RPL: out = log_softmax(A . W^T + bias - prior_scale * prior), i.e. the output
 * L.Linear (chainer_networks.py:21-22, 61-62, ...) followed by `y - logsum(y, axis=1)` (predict_folds.py:57,88) or by
 * `y = y - ap; y - logsum(y)` (evaluateModelForTest.py:75-77,110-112), without the float32 logits ever going to HBM:
 * the CTAs holding the 256-column tiles of a 128-row block form a thread-block cluster and exchange the rows' running
 * max / sum-exp through distributed shared memory (N <= 2048 classes).  Operands as nnam_linear_bias_act.  Exactly one
 * of `out` (float32 rows, leading dimension ld_out >= N, any 4-byte aligned pitch -- the (frames, N) array itself) and
 * `out16` + `row_ref` (the compact transfer format of nnam_head_f16; ld16 % 8 == 0) is given.  out_row_map as in
 * nnam_head_scatter (NULL: row r -> row r; -1: drop; -2 - q: zero-fill row q).  bias / prior may be NULL.  */
int nnam_linear_logsoftmax(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                           long long ldw, const float* bias, const float* prior, float prior_scale, float* out,
                           long long ld_out, void* out16, long long ld16, float* row_ref, const int* out_row_map,
                           int M, int N, int K, int nsplit, int elem, void* stream);

/* nnam_linear_logsoftmax scored against frame targets instead of writing rows: nll / pred / targets and the row map as
 * in nnam_head_score, y the float32 rows nnam_linear_logsoftmax writes with the same operands (the argmax is taken over
 * those written values, not over the logits: rounding bias - lse per column can reorder two near-tied columns).
 * Replaces (recalled from Chainer upstream, †) F.softmax_cross_entropy and F.accuracy behind L.Classifier, as used by
 * train.py, for a net whose output layer runs fused with its head.  */
int nnam_linear_logsoftmax_score(const void* a_hi, const void* a_lo, long long lda, const void* w_hi, const void* w_lo,
                                 long long ldw, const float* bias, const float* prior, float prior_scale,
                                 const int* targets, float* nll, int* pred, const int* out_row_map, int M, int N, int K,
                                 int nsplit, int elem, void* stream);

/* HOST function (no CUDA): dst_host[q][c] = float(src16_host[r][c]) + row_ref_host[r] for r < rows, c < cols, with
 * q = r, or q = dst_rows_host[r] when that map is given (the recurrent path ships a subset of utterances as one
 * contiguous block and scatters its rows to their frame positions here), on `threads` host threads (persistent pool;
 * F16C / AVX2 with non-temporal stores when the CPU has them).  All pointers are HOST pointers; dst_host is the
 * reference-layout float32 output (ld_dst == cols for the contiguous (N, C) array of np.save, predict_folds.py:240).  */
int nnam_widen_f16_host(const void* src16_host, long long ld16, const float* row_ref_host, float* dst_host,
                        long long ld_dst, const long long* dst_rows_host, long long rows, int cols, int threads);

/* Row gather + feature transform (+ i-vector append) for recurrent nets: out[r] = transform(x[row_map[r]]) ++
 * ivec[row_map[r]].  Replaces the per-utterance `np.pad(..., mode="edge")` + applyKaldiFeatureTransform + padded
 * (U, Lmax+timedelay, D) batch assembly of predict_folds.py:34-43 / evaluateModelForTest.py:57-59: row_map lists,
 * in time-major packed order, the source frame of every (utterance, step), repeating the last frame `timedelay`
 * times.  add_shift/rescale have `dim` entries (the shift-0 block) or are NULL.  Output bf16 / bf16 split / f32.
 * A map entry outside [0, n_src) produces a zero row.  */
int nnam_gather_transform(const float* x, long long n_src, int dim, const float* add_shift, const float* rescale,
                          const float* ivec, int ivec_dim, const int* row_map, long long n_rows, void* out_hi,
                          void* out_lo, long long ldo, int out_kind, void* stream);

/* Peephole-LSTM gate arithmetic for ONE time step on n packed rows (L.StatefulPeepholeLSTM via PeepholeLSTM,
 * chainer_networks.py:103-121).  The matrix products around it are nnam_linear_bias_act calls:
 *   g1 = [h | c] . [lateral/W | P]^T   with P rows [0, peep_i, peep_f, 0] per unit (gate-interleaved like lateral/W)
 *   phase 0:  c' = tanh(gx_a + g1_a) s(gx_i + g1_i) + s(gx_f + g1_f) c      -> c_new (fp32) and columns [H, 2H) of out
 *   p2 = c' . peep_o^T
 *   phase 1:  h' = s(gx_o + g1_o + p2) tanh(c')                              -> columns [0, H) of out
 * out_hi/out_lo are the bf16 (hi/lo) [h | c] rows of this step, (n, out_ld >= 2H).  g1 / c_prev may be NULL on the
 * first step (h = None, c = 0).  fast_tanh: 1 = tanh.approx (16-bit modes), 0 = tanhf (fp32-accurate mode).
 * elem: NNAM_ELEM_* of out_hi (out_lo, if given, is the bf16 low half and needs NNAM_ELEM_BF16).  */
int nnam_peephole_cell(int phase, const float* gx, long long gx_ld, const float* g1, long long g1_ld, const float* p2,
                       long long p2_ld, const float* c_prev, float* c_new, void* out_hi, void* out_lo,
                       long long out_ld, int n, int hidden, int fast_tanh, int elem, void* stream);

/* K3 -- persistent recurrence kernel: one launch runs a whole layer (one or both directions) over a whole shard.
 * Replaces the per-time-step Python loop around L.LSTM / F.lstm (chainer_networks.py:44-62 via
 * predict_folds.py:49-61 and evaluateModelForTest.py:67-80).  See csrc/recurrent.cu for the data layout.  */
typedef struct NnamRnnDesc {
  int cell;    /* NNAM_CELL_* */
  int hidden;  /* H (multiple of 64) */
  int n_dirs;  /* 1, or 2 = bidirectional: direction 1 walks every utterance backwards */
  int batch;   /* utterance slots per batch (= per stream): 16, 32, 64, or 128 (LSTM and the GRU family in bf16 mode
                  without carried state: the "wide" kernels, utterances on the MMA's M axis, two streams per group;
                  they need 32-byte aligned gx / h / xchg buffers and gx_ld, h_ld multiples of 16) */
  int streams; /* independent batches a CTA group runs concurrently (from nnam_rnn_plan) */
  int nsplit;  /* 1 = bf16 operands, 3 = bf16x3 (needs the _lo buffers) */
  int flags;   /* GRU family: bit 0 = reset gate, bits 1-2 = candidate activation (NNAM_ACT_*) */
  int elem;    /* NNAM_ELEM_*: element type of w_hi, h_hi, xchg_hi, h0_hi and (nsplit == 1) gx; nsplit == 3 needs BF16 */
  const void* gx[2];   /* per direction: input projection + bias for every packed row, (rows, gx_ld), columns
                          gate-interleaved exactly like Chainer's upward/W rows; fp32 when nsplit == 3, bf16 when
                          nsplit == 1 (in bf16 mode it is the largest HBM stream of a layer) */
  long long gx_ld;
  const void* w_hi[2]; /* per direction: lateral weights (4H, H) bf16 K-major.  LSTM: Chainer lateral/W as is.
                          GRU family: rows interleaved per unit [U_z, U_r (or 0), U, 0]; gx and u_bias likewise.
                          PEEPHOLE (unidirectional): [0] = lateral/W, [1] = peephole block, rows per unit
                          [0, peep_i, peep_f, peep_o] (L.StatefulPeepholeLSTM, chainer_networks.py:103-121).
                          GRU family with batch == 128: gate-BLOCKED rows without padding, (n_g * H, H) with n_g = 3
                          (reset gate) or 2: for every 32 units the 32 rows of U_z, then U_r (if any), then U; gx
                          columns and u_bias in the same order, gx_ld >= n_dirs * n_g * H, and the projection bias
                          already holds W_b + U_b (the kernel subtracts u_bias again at step 0) */
  const void* w_lo[2];
  long long w_ld;
  const float* u_bias[2]; /* GRU family: hidden-side biases, applied from the second step on (MGRU.py:70-83) */
  void* h_hi;          /* layer output (rows, h_ld) bf16; direction d writes columns [d*H, (d+1)*H) */
  void* h_lo;          /* low halves (bf16x3) or NULL */
  long long h_ld;
  void* xchg_hi;       /* exchange buffer, (n_groups * streams * 4 * batch, H) 16-bit, scratch: every CTA of a group
                          publishes its h slice here each step and TMA-loads the whole tile back.  Contents on entry
                          are irrelevant: the kernels never read a slot row they have not written in the same launch
                          (step 0 has no h product; rows beyond the active prefix only feed their own, unused, output
                          columns) -- tests/test_gpu_recurrent.py poisons it with NaNs to hold them to that */
  void* xchg_lo;       /* low halves (bf16x3) or NULL */
  int n_items;                 /* work items = (batch, direction) pairs, grouped by lane = (CTA group, stream);
                                  inside a lane the items are sorted by direction */
  const int* item_batch;       /* device arrays */
  const int* item_dir;
  int n_groups;
  const int* group_item_start; /* n_groups * streams + 1: first item of lane g * streams + s */
  const int* batch_row0;       /* first packed row of each batch */
  const int* batch_steps;      /* steps (= longest utterance) of each batch */
  const int* batch_nutt;       /* utterances in each batch (<= batch) */
  const int* batch_base_off;   /* offset of each batch's prefix-sum table inside `base` */
  const int* base;             /* per batch: base[t] = sum_{t' < t} active(t'), steps + 1 entries */
  const int* utt_len;          /* steps of every utterance in sorted order; batch b owns [b*batch, ...) */
  const void* h0_hi;           /* optional initial hidden state (n_utts, H*n_dirs) bf16 (+ lo), sorted order */
  const void* h0_lo;
  const float* c0;             /* optional initial cell state (n_utts, H*n_dirs) fp32 */
  float* c_out;                /* optional final cell state, same shape */
  unsigned int* counters;      /* n_groups * streams words of scratch */
  unsigned int* started;       /* optional, DEVICE-ACCESSIBLE HOST memory (pinned): thread 0 of every CTA stores started_tag
                                  into started[blockIdx.x] as its first action.  A host that runs two launches side by side
                                  (recurrent_engine.MixedSchedule) polls it to know that THIS launch is resident before it
                                  submits the other one: the multicast kernel runs as clusters of 16 CTAs, which can only
                                  be placed while whole GPCs are still free */
  unsigned int started_tag;
  void* debug_cycles;          /* optional: int64[8] per CTA, per-phase SM cycle totals (profiling builds/tests) */
} NnamRnnDesc;

int nnam_rnn_seq(const NnamRnnDesc* desc, void* stream);
/* sizeof(NnamRnnDesc) as compiled into the library: bindings in other languages check their struct mirror against it. */
int nnam_rnn_desc_size(void);
/* CTAs per group, the number of groups the current device can run concurrently for this cell configuration, and
 * (optional, may be NULL) the measured SM cycles per recurrence step, from which the host picks the batch width, and
 * the number of streams (concurrent batches per group) the kernel instance for `batch` slots runs.
 * NNAM_RNN_CLUSTER=1 in the environment opts LSTM / bf16 / batch 32 into the experimental thread-block-cluster variant
 * (h exchanged through distributed shared memory; measured slower than the L2 exchange on B200).  */
int nnam_rnn_plan(int cell, int hidden, int batch, int nsplit, int* group_ctas, int* max_groups, int* step_cycles,
                  int* streams);
/* SM cycles per step of a stream whose sibling streams in the CTA group are idle (<= step_cycles of nnam_rnn_plan,
 * which is measured with every stream busy).  A scheduler costs a two-stream group as
 * solo * (steps of its longer lane) + (busy - solo) * (steps of the other lane).  */
int nnam_rnn_solo_step_cycles(int cell, int hidden, int batch, int nsplit, int* cycles);

#ifdef __cplusplus
}
#endif
#endif /* NNAM_B200_H_ */
