/* xna_basecaller.h -- C ABI of the B200-native ub-bonito basecalling forward path.
 *
 * One shared library (xna_basecaller_b200/libxna_b200.so), extern "C", plain pointers and sizes, no
 * torch / C++ types.  The reference (CSB5/XNA_Basecaller, ub-bonito) is 100% Python and has no FFI of
 * its own for this path; each entry point below replaces the reference Python symbol cited next to it
 * (paths relative to ub-bonito/bonito/), and INTEGRATION.md shows the ctypes stub a reference
 * maintainer would add.  The Python package xna_basecaller_b200 mirrors the reference's plugin surface
 * (nn.py / crf/model.py / crf/basecall.py / util.py) on top of exactly these calls.
 *
 * Conventions
 *   - every function returns 0 on success, a negative xb_status otherwise; xb_last_error(h) gives the
 *     text (h may be NULL for errors raised before a handle exists).  Nothing throws, nothing exits.
 *   - a handle is bound to one CUDA device; it owns repacked weights and workspace, all allocated in
 *     xb_create / xb_load_weights.  The caller owns every input/output buffer.  A handle is not
 *     thread-safe; distinct handles are independent.  The workspace of a handle (gates, activations,
 *     decode state vectors, scores of the fused route) is shared by all of its calls: issue them on ONE
 *     stream, or order streams externally (events) -- nothing inside a handle orders two streams.
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued asynchronously on it with no host
 *     synchronisation, except the *_host entry points, which synchronise before returning.
 *   - device pointers unless the parameter name ends in _host.
 *   - T = L / stride (stride 5), C = n_base^state_len states, NZ = n_base+1 edges per state,
 *     scores are (T, N, C*NZ) fp32 in the reference's layout (nn.py:122-129).
 *   - activations are fp16 and so are the weights (what the reference itself uses on GPU,
 *     util.py:360-363); XB_FLAG_BF16 rounds the WEIGHTS to bfloat16 (a bf16 checkpoint's own values,
 *     held exactly in fp16 storage) and multiplies them with fp16 activations -- h, the hoisted input
 *     projection and the stem output are bounded, so the 11-bit mantissa of fp16 is the better 16-bit
 *     format for them.  Accumulation, LSTM cell state and scores are fp32.
 */
#ifndef XNA_BASECALLER_H
#define XNA_BASECALLER_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XB_ABI_VERSION 2

typedef struct xb_handle xb_handle;

enum xb_status {
    XB_OK = 0,
    XB_ERR_ARG = -1,        /* bad argument (shape, alignment, null pointer)              */
    XB_ERR_CUDA = -2,       /* a CUDA runtime / driver call failed                         */
    XB_ERR_STATE = -3,      /* call order (e.g. encoder before xb_load_weights)            */
    XB_ERR_UNSUPPORTED = -4,/* alphabet / state_len / feature size without a compiled kernel */
    XB_ERR_NOMEM = -5
};

enum xb_flags {
    XB_FLAG_BF16 = 1,            /* weights rounded to bfloat16 (activations stay float16)     */
    XB_FLAG_NO_ENCODER = 2,      /* decode-only handle: no encoder workspace is allocated      */
    XB_FLAG_TRAIN = 8            /* keep transposed bf16 weight copies for xb_encoder_bwd      */
    /* (4 was the one-launch-per-step LSTM of round 1; it exists only in -DXB_EXPERIMENTS builds) */
};

enum xb_signal_dtype { XB_SIG_F32 = 0, XB_SIG_F16 = 1, XB_SIG_I16 = 2 };

/* Number of weight tensors xb_load_weights expects: the reference state_dict in key order
 * (SURVEY.md section 5): encoder.{0,1,2}.conv.{weight,bias}, encoder.{4..8}.rnn.{weight_ih_l0,
 * weight_hh_l0,bias_ih_l0,bias_hh_l0}, encoder.9.linear.{weight,bias}. */
#define XB_NUM_WEIGHTS 28

int xb_abi_version(void);
const char *xb_last_error(const xb_handle *h);

/* Handle life cycle.  alphabet: n_base+1 letters, blank first ("NACGTX").  Replaces the state the
 * reference keeps in Model / CTC_CRF objects (crf/model.py:24-36, 224-237). */
int xb_create(xb_handle **out, int device, int max_N, int max_T, int n_base, int state_len,
              const char *alphabet, int flags);
int xb_destroy(xb_handle *h);

/* util.load_model's load_state_dict (util.py:324-366): 28 fp32 device tensors in reference layout,
 * repacked here into kernel layouts (gate-interleaved LSTM rows, K-major 16-bit GEMM operands).
 * scale / blank_score / expand_blanks are LinearCRFEncoder's (nn.py:90-96). */
int xb_load_weights(xb_handle *h, const float *const *tensors, int n_tensors, float scale,
                    float blank_score, int expand_blanks, void *stream);

/* The same, one module at a time (what nn.Convolution x3 / nn.LSTM / nn.LinearCRFEncoder hold,
 * nn.py:57-68,176-235,87-110), so that a single layer can be driven without the whole encoder.
 * layer in 0..4 selects the weight slot xb_lstm_fwd reads; b (head bias) may be NULL. */
int xb_load_conv_weights(xb_handle *h, const float *w1, const float *b1, const float *w2, const float *b2,
                         const float *w3, const float *b3, void *stream);
int xb_load_lstm_weights(xb_handle *h, int layer, const float *w_ih, const float *w_hh, const float *b_ih,
                         const float *b_hh, void *stream);
int xb_load_head_weights(xb_handle *h, const float *w, const float *b, float scale, float blank_score,
                         int expand_blanks, void *stream);

/* nn.Convolution x3 + nn.Permute([2,0,1]) (nn.py:57-68,156-167; crf/model.py:148-151).
 * signal (N, L) of sig_dtype -> out (T, N, 768) 16-bit. */
int xb_conv_stem_fwd(xb_handle *h, const void *signal, int sig_dtype, int N, int L, void *out_tnc,
                     void *stream);

/* nn.LSTM / RNNWrapper.forward (nn.py:176-235), layer in 0..4 (= encoder.4 .. encoder.8);
 * x, y (T, N, 768) 16-bit; reverse walks time backwards by indexing (no flips). */
int xb_lstm_fwd(xb_handle *h, int layer, const void *x_tnc, void *y_tnc, int T, int N, int reverse,
                void *stream);

/* the five layers with the reference's directions reverse,fwd,reverse,fwd,reverse (crf/model.py:152-154);
 * x is overwritten (ping-pong with handle workspace); result in y. */
int xb_lstm_stack_fwd(xb_handle *h, void *x_tnc, void *y_tnc, int T, int N, void *stream);

/* nn.LinearCRFEncoder.forward (nn.py:112-133): x (T,N,768) 16-bit -> scores (T,N,C*NZ) fp32 (or
 * (T,N,C*n_base) when expand_blanks was 0). */
int xb_crf_head_fwd(xb_handle *h, const void *x_tnc, float *scores, int T, int N, void *stream);

/* Model.forward (crf/model.py:212-213): signal (N, L) -> scores (T, N, C*NZ) fp32. */
int xb_encoder_fwd(xb_handle *h, const void *signal, int sig_dtype, int N, int L, float *scores,
                   void *stream);

/* CTC_CRF.logZ (crf/model.py:41-46), Log semiring: logz (N). */
int xb_crf_logz(xb_handle *h, const float *scores, int T, int N, float *logz, void *stream);

/* CTC_CRF.forward_scores / backward_scores (crf/model.py:51-61), Log semiring: (T+1, N, C). */
int xb_crf_forward_scores(xb_handle *h, const float *scores, int T, int N, float *alpha, void *stream);
int xb_crf_backward_scores(xb_handle *h, const float *scores, int T, int N, float *beta, void *stream);

/* The same three with the semiring argument the reference's methods take (S: semiring = Log, crf/model.py:41,51,57):
 * XB_SEMIRING_MAX gives the best path's score / the Max-semiring forward and backward vectors. */
enum xb_semiring { XB_SEMIRING_LOG = 0, XB_SEMIRING_MAX = 1 };
int xb_crf_logz_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *logz, void *stream);
int xb_crf_forward_scores_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *alpha, void *stream);
int xb_crf_backward_scores_s(xb_handle *h, const float *scores, int T, int N, int semiring, float *beta, void *stream);

/* SequenceDist.posteriors(scores, Max) (what CTC_CRF.viterbi arg-maxes, crf/model.py:92-95): the one-hot tensor at the
 * arg-max edge of every step's max-marginals (first flat index c*NZ + k on ties).  edges_nt (N, T) int32 receives the
 * edge indices; post (T, N, C*NZ) fp32 the one-hot tensor itself, may be NULL. */
int xb_crf_posteriors_max(xb_handle *h, const float *scores, int T, int N, int32_t *edges_nt, float *post, void *stream);

/* SequenceDist.posteriors(scores, Log) (crf/model.py:216): post (T, N, C*NZ) fp32. */
int xb_crf_posteriors(xb_handle *h, const float *scores, int T, int N, float *post, void *stream);

/* CTC_CRF.viterbi (crf/model.py:92-95): labels (N, T) int8 in 0..n_base (already transposed). */
int xb_crf_viterbi(xb_handle *h, const float *scores, int T, int N, int8_t *labels_nt, void *stream);

/* SeqdistModel.decode_batch (crf/model.py:215-218) + the left-packing of compute_scores
 * (crf/basecall.py:56-76): seq / qstring (N, T) int8 zero padded (ascii letters / 'O'), lens (N).
 * qstring, labels_nt, post may be NULL. */
int xb_crf_decode(xb_handle *h, const float *scores, int T, int N, int8_t *seq, int8_t *qstring,
                  int32_t *lens, int8_t *labels_nt, float *post, void *stream);

/* Beam-search decode for any alphabet (the role koi.decode.beam_search plays at crf/basecall.py:33-46; koi itself is
 * ACGT-only and switched off for the UB models, util.py:299-313): a beam of beam_width <= 32 (emitted sequence, lattice
 * state) pairs that sums the alignments of a sequence and is guided by the exact backward scores; candidates further than
 * beam_cut below the leader are dropped.  scores (T, N, C*NZ) fp32 as for xb_crf_decode.  seq / qstring (N, T) int8
 * left-packed letters and phred+33 qualities, moves (N, T) int8 = 1 at the steps that emitted a base, lens (N);
 * qstring and moves may be NULL.  Algorithm and its checker: csrc/beam_search.cu, oracle/c/crf_exact.c. */
int xb_crf_beam_search(xb_handle *h, const float *scores, int T, int N, int beam_width, float beam_cut, int8_t *seq,
                       int8_t *qstring, int8_t *moves, int32_t *lens, void *stream);

/* The fused route's hand-over format.  decode_batch is computed in the linear domain (sums / maxima of products of
 * E = exp(score), see csrc/crf_decode_lin.cu); when encoder and decode run back to back the CRF head writes E itself
 * -- one bit-reproducible exponential per edge instead of one in each of the three decode sweeps -- and the decode
 * reads it.  xb_crf_head_fwd_exp is xb_crf_head_fwd with that exponential applied (blank included),
 * xb_crf_decode_exp is xb_crf_decode on such a tensor; xb_crf_decode_exp(xb_crf_head_fwd_exp(x)) returns the bits of
 * xb_crf_decode(xb_crf_head_fwd(x)).  Scores outside [-80, 80] are clamped before the exponential on both routes. */
int xb_crf_head_fwd_exp(xb_handle *h, const void *x_tnc, float *escores, int T, int N, void *stream);
int xb_crf_decode_exp(xb_handle *h, const float *escores, int T, int N, int8_t *seq, int8_t *qstring,
                      int32_t *lens, int8_t *labels_nt, float *post, void *stream);

/* compute_scores between its two copies (crf/basecall.py:47-76) for chunks already on the device: encoder + decode over
 * signal (N, L) of sig_dtype -> seq / qstring (N, T) int8 left-packed, lens (N); qstring may be NULL.  The scores
 * stay in handle workspace (in the hand-over format above). */
int xb_basecall_chunks(xb_handle *h, const void *signal, int sig_dtype, int N, int L, int8_t *seq, int8_t *qstring,
                       int32_t *lens, void *stream);

/* CTC_CRF.ctc_loss(reduction='none') forward (crf/model.py:118-131): targets (N, Lmax) int32 1-based
 * 0-padded, lengths (N) int32 -> loss (N) fp32 = -logz / length.  normalise as in the reference. */
int xb_ctc_crf_loss_fwd(xb_handle *h, const float *scores, int T, int N, const int32_t *targets,
                        int Lmax, const int32_t *lengths, int normalise, float *loss, void *stream);

/* Backward of the above (what loss.backward() propagates to the scores in Trainer.train_one_step,
 * training.py:91-117, through seqdist's Logspace gradients): grad_scores (T, N, C*NZ) fp32 =
 * grad_loss[n] * (P_full[t,n,e] * normalise - P_target[t,n,e]) / lengths[n], P_full the edge posteriors of the
 * whole lattice, P_target those of the target's alignment lattice.  grad_loss (N) fp32 is the upstream gradient
 * per sequence (1/N for reduction='mean'); alpha_ws is caller-owned scratch of (T+1) * N * (Lmax - state_len + 1)
 * floats. */
int xb_ctc_crf_loss_bwd(xb_handle *h, const float *scores, int T, int N, const int32_t *targets,
                        int Lmax, const int32_t *lengths, int normalise, const float *grad_loss,
                        float *alpha_ws, float *grad_scores, void *stream);

/* The encoder half of Trainer.train_one_step (training.py:91-117) on a handle created with XB_FLAG_TRAIN:
 *   xb_encoder_fwd_train  = scores_ = model(data_): xb_encoder_fwd that also keeps the layer inputs and the LSTM gate /
 *                           cell values of every step in handle workspace (N must be a multiple of 8);
 *   xb_encoder_bwd        = what loss.backward() does below the scores: dscores (T,N,C*NZ) fp32 (from
 *                           xb_ctc_crf_loss_bwd) -> fp32 gradients of the XB_NUM_WEIGHTS parameter tensors, in
 *                           xb_load_weights' order and the reference's layouts -- except encoder.2.conv.weight, whose
 *                           gradient is (768, 320) = [out][tap*16 + in] (the caller reshapes to (768,16,19)).
 * signal and scores are the buffers of the matching forward call. */
int xb_encoder_fwd_train(xb_handle *h, const void *signal, int sig_dtype, int N, int L, float *scores, void *stream);
int xb_encoder_bwd(xb_handle *h, const void *signal, int sig_dtype, const float *scores, const float *dscores,
                   float *const *grads, int n_tensors, void *stream);

/* Dropout in the training step (rnn_encoder(drop_rate_bottom=...), crf/model.py): the forward of xb_encoder_fwd_train with
 * torch.nn.Dropout(p[s]) applied at XB_DROPOUT_SITES sites, in the order the reference applies them:
 *   0 conv1 output, 1 conv2 output, 2 conv3 output, 3..6 outputs of LSTM layers 0..3.
 * p is a host array of XB_DROPOUT_SITES probabilities, each 0 <= p < 1 (else XB_ERR_ARG); NULL or all zero is exactly
 * xb_encoder_fwd_train (same kernels, same bits).  The mask is a pure function of (seed, site, element index): Philox4x32-10
 * keyed by the 64-bit seed, written out in csrc/xb_dropout.cuh.  Kept values are scaled by (float)(1 / (1 - p)), dropped
 * ones are 0 -- torch.nn.Dropout's distribution, not torch's random stream.  The handle records (p, seed), and the next
 * xb_encoder_bwd regenerates the same masks; its signature does not change. */
#define XB_DROPOUT_SITES 7
int xb_encoder_fwd_train_dropout(xb_handle *h, const void *signal, int sig_dtype, int N, int L, const float *p, uint64_t seed,
                                 float *scores, void *stream);

/* The keep flags (1 kept, 0 dropped) of elements 0 .. n-1 of one dropout site under (seed, p), computed on the current
 * device by the device function the training kernels use.  keep: n bytes of device memory.  Needs no handle. */
int xb_dropout_keep(uint64_t seed, int site, float p, int64_t n, uint8_t *keep, void *stream);

/* The optimiser half of Trainer.train_one_step (training.py:112-115): torch.nn.utils.clip_grad_norm_(max_norm) followed by
 * one torch.optim.AdamW step (training.py:183-184; decoupled weight decay, bias-corrected moments) over n_tensors fp32
 * tensors given as host arrays of device pointers.  max_norm <= 0 disables clipping; step >= 1 counts this update;
 * grad_norm (device, 1 float) receives the total gradient norm before clipping; scratch is device memory of
 * 4 * (sum_i ceil(numel[i] / 65536) + 1) bytes.  Needs no handle. */
int xb_adamw_step(float *const *params, float *const *grads, float *const *exp_avg, float *const *exp_avg_sq,
                  const int64_t *numel, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                  float max_norm, int64_t step, float *grad_norm, float *scratch, void *stream);

/* Local alignment counts for validation accuracy (util.accuracy, bonito/util.py:402-424): for each pair p, the best local
 * alignment of query seq[p] (seq_len[p] bytes of row p, rows seq_stride bytes apart) against reference ref[p] under the
 * contract written in csrc/align.cu (+5 for identical bytes, -4 otherwise, a gap of length k costs 8 + 4 (k - 1), fixed
 * tie rules).  counts (n_pairs, 5) int32 on the device receives (score, eq, x, ins, del): matching and mismatching
 * columns, query bases aligned to a gap and reference bases aligned to a gap; all zero for an empty alignment.
 * seq / ref are letter codes as xb_crf_decode writes them (left-packed rows); seq_len / ref_len are device arrays.
 * The lengths are copied to the host and checked (0 <= len <= 32767 and len <= row stride, else XB_ERR_ARG), so the
 * call synchronises the stream once before it enqueues the kernel.  Needs no handle. */
int xb_align_counts(const int8_t *seq, int seq_stride, const int32_t *seq_len, const int8_t *ref, int ref_stride,
                    const int32_t *ref_len, int n_pairs, int32_t *counts, void *stream);

/* util.stitch over left-packed chunks (util.py:169-188; crf/basecall.py:15-24): for each read r,
 * concatenates slices of its chunks' packed rows.  chunk_first[r], chunk_count[r], read_len[r]
 * (samples) describe the reads; rows are (n_chunks_total, T) int8; out is (n_reads, out_stride) int8,
 * out_len (n_reads).  reverse != 0 is the reference's reverse=True branch (util.py:180-184; `bonito basecaller
 * --reverse`): chunks walked backwards, slices taken from the end of each row with Python's negative-index rules. */
int xb_stitch(xb_handle *h, const int8_t *rows, int T, const int32_t *chunk_first,
              const int32_t *chunk_count, const int32_t *read_len, int n_reads, int chunksize,
              int overlap, int stride, int reverse, int8_t *out, int out_stride, int32_t *out_len, void *stream);

/* util.chunk (util.py:152-166) for a whole read set resident on the device: signal holds the reads back to back
 * (sig_dtype XB_SIG_F32 or XB_SIG_I16), read r occupies [read_offset[r], read_offset[r] + read_len[r]); chunk c is
 * samples [chunk_start[c], chunk_start[c] + L) of read chunk_read[c], zero where that runs off the read (a negative
 * start is the left padding of a short read).  out (n_chunks, L) fp32. */
int xb_gather_chunks(xb_handle *h, const void *signal, int sig_dtype, const int64_t *read_offset,
                     const int32_t *read_len, const int32_t *chunk_read, const int32_t *chunk_start, int n_chunks,
                     int L, float *out, void *stream);

/* Per-read signal pre-processing (the reference's Read.__init__, fast5.py:88-100: DAC -> pA scaling, trim :149-172, then
 * med/MAD normalisation, or norm_by_noisiest_section for reads of <= 8000 samples after trimming).  raw: concatenated int16
 * DAC samples, read r = [read_offset[r], read_offset[r] + read_len[r]); scaling[r] = range / digitisation, offset[r] the
 * channel offset.  out: float32 with the same layout -- the trimmed, normalised signal of read r starts at
 * out[read_offset[r]] and has out_len[r] samples (feed out / read_offset / out_len to xb_gather_chunks).  stats
 * (n_reads, 4) float32: trim start, med, mad, mode (0 whole read, 1 noisiest section, 2 nothing left). */
int xb_preprocess_reads(xb_handle *h, const int16_t *raw, const int64_t *read_offset, const int32_t *read_len,
                        const double *scaling, const int32_t *offset, int n_reads, float *out, int32_t *out_len,
                        float *stats, void *stream);

/* crf.basecall.compute_scores end to end with HOST buffers (crf/basecall.py:27-82): H2D of the
 * chunk batch, encoder, decode, D2H of the packed sequences; synchronises.  signal_host (N, L) fp32,
 * seq_host (N, T) int8, lens_host (N).  Pinned host memory makes the copies asynchronous. */
int xb_compute_scores_host(xb_handle *h, const float *signal_host, int N, int L, int8_t *seq_host,
                           int32_t *lens_host, void *stream);

/* Pipelined form of xb_compute_scores_host for a stream of batches (the reference overlaps its stages with one thread per
 * stage, crf/basecall.py:96-119): submit() enqueues the H2D copy, encoder, decode and D2H copy of one batch into slot 0 or 1
 * and returns; wait() blocks until that slot's seq_host / lens_host are filled.  Submit batch i+1 before waiting for batch i
 * and the copies hide under the kernels.  A slot must be waited for before it is submitted again; the host buffers (pinned
 * for the copies to be asynchronous) must stay valid until then. */
int xb_compute_scores_submit(xb_handle *h, int slot, const float *signal_host, int N, int L, int8_t *seq_host,
                             int32_t *lens_host, void *stream);
int xb_compute_scores_wait(xb_handle *h, int slot);

/* Introspection used by tests / bench: number of kernels this library launched on the handle so far. */
int64_t xb_launch_count(const xb_handle *h);

/* Per-stage device timing with CUDA events on the launching stream (bench.py's roofline numbers).
 * Stages: 0 conv1+conv2+im2col, 1 conv3 GEMM, 2 LSTM input-projection GEMMs, 3 LSTM recurrence,
 * 4 CRF head GEMM, 5 CRF alpha sweep, 6 CRF backward sweep, 7 CRF Viterbi sweep + packing;
 * of xb_encoder_bwd: 8 BPTT step kernels, 9 transposed copies (+ bias gradients), 10 weight-gradient GEMMs (K = T*N),
 * 11 input-gradient GEMMs, 12 head and convolution-stem backward kernels.
 * xb_stage_times synchronises, adds the elapsed milliseconds and launch-span counts of every span
 * recorded since the last call into ms[XB_NUM_STAGES] / spans[XB_NUM_STAGES], and clears them. */
#define XB_NUM_STAGES 13
int xb_set_profiling(xb_handle *h, int on);
int xb_stage_times(xb_handle *h, float *ms, int *spans);

/* Standalone tensor-core GEMM self-test hook: D (M,N) fp32 = A (M,K) x B (N,K)^T, fp16 operands. */
int xb_gemm_selftest(xb_handle *h, const void *A, const void *B, float *D, int M, int N, int K,
                     void *stream);

#ifdef __cplusplus
}
#endif
#endif /* XNA_BASECALLER_H */
