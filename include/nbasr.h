/*
 * nbasr.h -- C ABI of libnbasr.so: the B200 (sm_100a) kernels behind the NAS-Bench-ASR
 * candidate train/eval step.
 *
 * The reference (SamsungLabs/nb-asr) has no FFI of its own: its hot path is a chain of
 * torch library calls (SURVEY.md 2.2).  Each entry point below therefore cites the reference
 * call site(s) it replaces (paths under /root/reference/nasbench_asr/).  INTEGRATION.md shows
 * the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *   - caller allocates all outputs/workspaces; no hidden allocation, no sync, no host<->device
 *     copies; every launch goes to the `stream` argument (a cudaStream_t passed as void*);
 *   - return 0 on success, non-zero on error (nbasr_last_error() gives the message);
 *   - dtype codes: NBASR_F32 = 0, NBASR_BF16 = 1, NBASR_F16 = 2.
 *
 * 16-bit mode ("bf16" precision of the engine): FORWARD activations and the weight operands that multiply them are
 * IEEE fp16 (10-bit mantissa: bf16 storage of every activation costs 2-4e-2 on the logits of this 80-layer net, fp16
 * 0.8-1.5e-2, DESIGN.md 4), stored multiplied by a power-of-two `act_scale` so that small activations stay out of the
 * fp16 subnormal range; GRADIENTS and the operands that multiply them are bf16 (range).  One tcgen05.mma needs both
 * operands in the same format (mixed f16 x bf16 faults, tools/experiments/README.md), so tensors that feed a weight
 * gradient are additionally written as an unscaled bf16 copy by their producer (training plans only).
 *
 * Activation layout ("frames x channels", channels-last): a tensor of one encoder block is
 * (B, Tp, C) contiguous with Tp = T + NBASR_PAD_L + NBASR_PAD_R; frame t of utterance b is row
 * b*Tp + NBASR_PAD_L + t.  Pad rows are zero and are never written, so every (dilated /
 * strided) convolution tap is a plain row offset and zero padding comes for free.
 */
#ifndef NBASR_H
#define NBASR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NBASR_F32 0
#define NBASR_BF16 1
#define NBASR_F16 2
#define NBASR_PAD_L 8
#define NBASR_PAD_R 4
#define NBASR_MAX_ADD 3

/* Fused output stage shared by the dense GEMM, grouped-conv and element-wise kernels.
 * For an accumulator value v at output row rho, column n:
 *   v  = v*acc_scale + bias[n]*bias_scale          (ops.py:26,45 bias of Conv1d / Linear; scales: see below)
 *   m  = (0 < v <= relu_hi); v = min(max(v,0),relu_hi)   (ops.py:27-28,46-47 ReLU + clamp_max 20)
 *   keep ~ Bernoulli(1-p); m &= keep; v = keep ? v/(1-p) : 0   (ops.py:22,29,40,48 Dropout)
 *   v += add[0][rho,n] + add[1][rho,n] + ...       (model.py:16-22 skip-connection sum)
 *   out[rho,n] = v ; mask_out bit(rho,n) = m
 *   out2[rho,n] = bit(mask2,rho,n) ? v*scale2 : 0  (backward: gradient through ReLU20/Dropout)
 * All row-indexed tensors share the row mapping of the call; ld_out is the row pitch in elements.
 * Gate-bit masks are PLANE-major bit arrays: columns are cut into planes of `w` columns (w = 32 -> 4-byte
 * entries, w = 40/48 -> 8-byte entries; the producer kernel's natural slab width), plane p holds one entry per
 * row: byte address of (row, col) = ((col / w) * mask_rows + row) * entry_bytes + (col % w) / 8, bit col % 8.
 * Consecutive rows are contiguous, so every producer/consumer reads and writes masks coalesced. */
typedef struct nbasr_epilogue {
  const float* bias;
  int32_t relu20;
  float drop_p;
  uint64_t drop_seed;           /* per-call salt */
  const uint64_t* drop_step;    /* optional device counter mixed into the seed (graph replay) */
  int32_t n_add;
  const void* add[NBASR_MAX_ADD];
  int32_t add_dtype;
  void* out;
  int32_t out_dtype;
  int64_t ld_out;
  uint32_t* mask_out;
  void* out2;
  int32_t out2_dtype;
  const uint32_t* mask2;
  float scale2;
  int64_t mask_rows;    /* rows per mask plane (same for mask_out and mask2) */
  int32_t mask_w;       /* plane width of mask_out: 32, 40 or 48 */
  int32_t mask2_w;      /* plane width of mask2 */
  int32_t accumulate;   /* out += v instead of out = v (fp32 out only, SIMT path) */
  /* Scaled fp16 activations: a kernel whose A operand holds act_scale*x produces act_scale*(W x) in its accumulator.
   * Forward edges stay in the scaled domain (acc_scale 1, bias_scale = act_scale, relu_hi = 20*act_scale, skip tensors
   * and `out` scaled alike; out2 with scale2 = 1/act_scale and mask2 = NULL is the unscaled bf16 copy for the weight
   * gradient); a consumer that wants true values (LSTM input projection) sets acc_scale = 1/act_scale.
   * 0 means "unset": acc_scale 1, bias_scale 1, relu_hi 20. */
  float acc_scale;
  float bias_scale;
  float relu_hi;
} nbasr_epilogue;

/* Dense GEMM  C[(b,r), n] = sum_k A[(b,r), k] * W[n, k]  followed by the epilogue.
 * A element (b,r,k) is a[b*a_bs + r*a_rs + k]; rows may overlap (a_rs < K), which is how the
 * k=8 time-reduction convolutions (model.py:82-89 -> ops.py:25-26) become one GEMM with
 * K = 8*C_in over the zero-padded channels-last input (stride 2: a_rs = 2*C_in).
 * Output row rho = o_r0 + b*o_bs + r*o_rs.  Replaces: nn.Conv1d(groups=1) (ops.py:26),
 * nn.Linear edge (ops.py:45), LSTM input projection (model.py:100), and their input-gradients
 * (W pre-packed by nbasr_pack_weight).  dtype BF16 -> tcgen05/TMEM/TMA kernel; F32 -> SIMT. */
typedef struct nbasr_gemm {
  int32_t dtype;          /* of A and W: F32 (SIMT), BF16 or F16 (tcgen05; both operands share the format) */
  const void* a;
  int64_t a_bs, a_rs;
  int32_t nb, nr, K, N;
  const void* w;
  int64_t ldw;
  int64_t o_r0, o_bs, o_rs;
  nbasr_epilogue epi;
} nbasr_gemm;

int nbasr_gemm_tn(const nbasr_gemm* p, void* stream);

/* Weight-gradient GEMM  dW[m, n] += sum_{b,r} dY[(b,r), m] * X[(b,r), n]   (fp32, atomic add)
 * dY element (b,r,m) = dy[b*dy_bs + r*dy_rs + m]; X element = x[b*x_bs + r*x_rs + n] (overlapping
 * rows give all conv taps at once: n = tap*C_in + c_in).  Replaces the weight-gradient half of
 * autograd for Conv1d/Linear/LSTM (trainer.py:223 `_regu_loss.backward()`). */
typedef struct nbasr_wgrad {
  int32_t dtype;
  const void* dy;
  int64_t dy_bs, dy_rs;
  const void* x;
  int64_t x_bs, x_rs;
  int32_t nb, nr, M, N;
  float* dw;
  int64_t ldw;
  float* dbias;           /* optional: dbias[m] += sum_{b,r} dY[(b,r), m] (bias gradient, fused) */
} nbasr_wgrad;

int nbasr_gemm_wgrad(const nbasr_wgrad* p, void* stream);

/* Grouped (groups = C/cpg) 1-D convolution edge, channels-last, taps at row offsets
 * off0 + j*dstep (j < ktaps):  ops.py:73-76 conv5/conv5d2/conv7/conv7d2 (groups=100).
 * w is (C, cpg, ktaps) fp32 in the reference layout (forward) or the group-transposed pack
 * made by nbasr_pack_gconv_dgrad (input gradient, with negated offsets). */
#define NBASR_W_STABLE 2
typedef struct nbasr_gconv {
  int32_t dtype;          /* of x and of the packed weights: F32 / BF16 / F16 */
  const void* x;          /* (B, Tp, C) padded activation, pointer to row 0 of the buffer */
  int32_t B, T, Tp, C, cpg, ktaps, off0, dstep;
  const void* w;          /* w_packed = 0: fp32 (C, cpg, ktaps)  -> SIMT kernel (any dtype)
                             w_packed & 1: bf16 block-diagonal pack of nbasr_pack_gconv_mma -> tcgen05 kernel (BF16)
                             w_packed & 2 (NBASR_W_STABLE): the pack was not written by the launch immediately before this
                             one on the stream; the kernel may then fetch it before its programmatic launch dependency
                             resolves (never set it right after nbasr_pack_gconv_mma on the same stream) */
  int32_t w_packed;
  nbasr_epilogue epi;     /* rows rho = b*Tp + PAD_L + t */
} nbasr_gconv;

int nbasr_gconv_fwd(const nbasr_gconv* p, void* stream);
int nbasr_pack_gconv_dgrad(const float* w, float* wt, int C, int cpg, int ktaps, void* stream);
/* bf16 block-diagonal operand for the tcgen05 grouped-conv kernel: [slab][tap][48][64], slabs of 48 (cpg 6/8/12)
 * or 40 (cpg 10) channels; transposed = 1 gives the input-gradient operand (group-transposed, taps flipped).
 * nbasr_gconv_mma_pack_elems returns the number of bf16 elements of the pack. */
int nbasr_pack_gconv_mma(const float* w, void* out, int out_dtype, int C, int cpg, int ktaps, int transposed, void* stream);
int64_t nbasr_gconv_mma_pack_elems(int C, int cpg, int ktaps);
/* dw[c_out][i][j] += sum_{b,t} dz[b,t,c_out] * x[b, t+off0+j*dstep, g*cpg+i];  dbias[c] += sum_{b,t} dz[b,t,c]
 * (dbias may be NULL). BF16 -> tcgen05 kernel, F32 -> SIMT. */
int nbasr_gconv_wgrad(int dtype, const void* dz, const void* x, int B, int T, int Tp, int C, int cpg,
                      int ktaps, int off0, int dstep, float* dw, float* dbias, void* stream);
/* The same with X in its own format, multiplied by x_scale as it is read: the scaled fp16 forward activations (S*x, nbasr.h
 * "scaled fp16") with x_scale = 1/S, so that a 16-bit plan needs no bf16 copy of them.  dz_dtype BF16 takes x_dtype BF16 or
 * F16; F32 takes F32.  nbasr_gconv_wgrad(dtype, ...) is nbasr_gconv_wgrad_x(dtype, dz, x, dtype, 1, ...). */
int nbasr_gconv_wgrad_x(int dz_dtype, const void* dz, const void* x, int x_dtype, float x_scale, int B, int T, int Tp, int C,
                        int cpg, int ktaps, int off0, int dstep, float* dw, float* dbias, void* stream);

/* Element-wise pass through the epilogue: v = src ? src[rho,n] : 0 over rows (b,t) of a padded
 * (B,Tp,C) geometry.  Used for `zero` main ops (ops.py:62-68), the LSTM input dropout
 * (model.py:99) and gradient masking. */
int nbasr_eltwise(int src_dtype, const void* src, int64_t ld_src, int B, int T, int Tp, int C,
                  const nbasr_epilogue* epi, void* stream);

/* column sums  out[c] += sum_{b,t} x[b,t,c]  (bias gradients). */
int nbasr_colsum(int dtype, const void* x, int B, int T, int Tp, int C, float* out, void* stream);

/* LayerNorm over channels, eps given (model.py:47,92: nn.LayerNorm(C, eps=1e-3)), biased
 * variance, affine.  Saves mean / rstd per row for the backward pass.
 * y = (gamma * xhat + beta) * out_scale in `dtype`; optional y2 = (gamma * xhat + beta) as bf16 (the unscaled copy a
 * weight gradient reads; NULL in eval plans).  With scaled fp16 input (x = s*x_true) the caller passes eps * s^2: xhat
 * is then exactly that of the unscaled tensor, and the saved mean / rstd are those of the scaled one. */
int nbasr_layernorm_fwd(int dtype, const void* x, void* y, int B, int T, int Tp, int C,
                        const float* gamma, const float* beta, float eps, float* mean, float* rstd,
                        float out_scale, void* y2, void* stream);
/* dx (+ optional dx2 = dx * bit(mask2) * scale2), dgamma += , dbeta +=.  dy / dx / dx2 have dtype `dtype` (BF16 in
 * 16-bit mode), x has x_dtype; x_scale = s when x (and the saved mean / rstd) are those of the scaled tensor s*x_true:
 * the gradient wrt x_true is s times the gradient wrt the stored tensor. */
int nbasr_layernorm_bwd(int dtype, const void* dy, const void* x, int x_dtype, float x_scale, const float* mean,
                        const float* rstd, const float* gamma, int B, int T, int Tp, int C, void* dx, void* dx2,
                        const uint32_t* mask2, float scale2, int64_t mask_rows, int mask2_w, float* dgamma,
                        float* dbeta, void* stream);

/* (B, F, T) fp32 channel-first input (trainer.py:210) -> padded channels-last (B, Tp, F), multiplied by `scale`. */
int nbasr_transpose_in(const float* audio, void* out, int dtype, int B, int F, int T, int Tp, float scale, void* stream);
/* The inverse: padded channels-last fp32 (B, Tp, F), frame t at row b*Tp + PAD_L + t -> (B, F, T) fp32 (the input
 * gradient of the model). */
int nbasr_transpose_out(const float* in, float* out, int B, int F, int T, int Tp, void* stream);

/* Weight packing: out[n][q*M + m] = w[m*ws_m + n*ws_n + (t0 + q*tstep)*ws_t],  q < nq.
 * Produces the bf16 / fp32 operand copies (plain, transposed, tap-flipped) used by gemm_tn. */
int nbasr_pack_weight(const float* w, void* out, int out_dtype, int M, int N, int nq, int t0, int tstep,
                      int64_t ws_m, int64_t ws_n, int64_t ws_t, void* stream);
int nbasr_convert(const float* src, void* dst, int dst_dtype, int64_t n, void* stream);

/* LSTM (model.py:100 nn.LSTM(1200,500,batch_first), zero initial state, gates i,f,g,o).
 * gx: (B, T, 4H) fp32 input projection incl. both biases; w_hh (4H, H) fp32.
 * Outputs: h_seq (B, Tp?, ld_h) act dtype written at row b*h_bs + t*h_rs; saves gates (B,T,4H)
 * post-activation and c (B,T,H) for BPTT.  work: 2*B*H floats (h ping-pong). Cooperative launch. */
int nbasr_lstm_fwd(const float* gx, const float* w_hh, int T, int B, int H, void* h_seq, int h_dtype,
                   int64_t h_bs, int64_t h_rs, int64_t ld_h, float* gates, float* cstate,
                   const void* w_hh_packed, float* work, void* stream);
/* w_hh_packed (optional): bf16 [16][gate*32+unit][512] pack of W_hh (nbasr_pack_batch kind 4).  When given and
 * h_dtype is BF16 the recurrence runs on tcgen05 tensor cores in 16-CTA clusters (bf16 h / W_hh operands, fp32
 * accumulation, gates and cell state); otherwise the fp32 SIMT kernel is used. */
/* BPTT: dh_seq (same addressing as h_seq, fp32) -> dgx (B,T,4H) fp32 (gradient of gx).
 * dW_hh / dW_ih / biases then follow from nbasr_gemm_wgrad / nbasr_colsum over dgx. */
int nbasr_lstm_bwd(const float* dh_seq, int64_t dh_bs, int64_t dh_rs, int64_t ld_dh, const float* w_hh,
                   const float* gates, const float* cstate, int T, int B, int H, float* dgx, float* work,
                   const void* w_hh_packed, void* dgx_bf16, void* stream);
/* w_hh_packed given -> tcgen05 / cluster kernel (bf16 recurrent operands); it can also emit dgx as bf16 (dgx_bf16). */

/* Classifier + log-softmax: logits = h W^T + b (model.py:101 nn.Linear(500,49)),
 * logp = log_softmax(logits) (trainer.py:218). h rows at b*h_bs + t*h_rs, pitch implied by strides. */
int nbasr_head_fwd(int h_dtype, const void* h, int64_t h_bs, int64_t h_rs, int B, int T, int K, int V,
                   const float* w, const float* bias, float* logits, float* logp, void* stream);
/* dlogits (B,T,V) fp32 -> dh (fp32, same addressing as h), dw += , db += */
int nbasr_head_bwd(int h_dtype, const void* h, int64_t h_bs, int64_t h_rs, int B, int T, int K, int V,
                   const float* w, const float* dlogits, float* dh, int64_t dh_bs, int64_t dh_rs,
                   float* dw, float* db, void* stream);

/* Input-gradient half of the classifier backward only: dh = dlogits W (fp32, same addressing as nbasr_head_bwd), plus
 * (optional) dl16 = dlogits as bf16 padded to 64 columns, (B*T, 64): the dY operand with which nbasr_gemm_wgrad then
 * computes dW (and db) on the tensor cores against the bf16 h_seq. */
int nbasr_head_bwd_dh(int B, int T, int K, int V, const float* w, const float* dlogits, float* dh, int64_t dh_bs,
                      int64_t dh_rs, void* dl16, void* stream);

/* CTC (trainer.py:36-44: F.ctc_loss(reduction='none', zero_infinity=True) / output_len, mean).
 * logp (B,T,V) fp32, blank 0; targets (B,S) int32 zero padded; lens int64 (audio_len is the INPUT
 * length; output_len = audio_len / len_div, trainer.py:219 uses 4).  Outputs: nll[b] (already
 * zero-infinity'd, NOT divided), loss (scalar mean of nll/output_len), and, if dlogits != NULL,
 * d loss / d logits (B,T,V) (log-softmax backward folded in).  work: 2*B*T*(2S+1) floats. */
int nbasr_ctc(const float* logp, int B, int T, int V, const int32_t* targets, int S,
              const int64_t* audio_len, int len_div, const int64_t* targets_len, float* nll, float* loss,
              float* dlogits, float* work, void* stream);

/* CTC forced alignment: the Viterbi path of the known target sequence through the CTC trellis (where each phone of the
 * transcript sits in time; what torchaudio.functional.forced_align computes one utterance at a time).  Inputs exactly as
 * nbasr_ctc: T_b = min(T, audio_len[b] / len_div) frames, S_b = min(S, targets_len[b]) tokens.
 *   alpha_0(0) = logp[0, 0], alpha_0(1) = logp[0, ext[1]], other states -inf; over the 2S_b + 1 extended states
 *   alpha_t(s) = max(alpha_{t-1}(s), alpha_{t-1}(s-1), alpha_{t-1}(s-2) [ext[s] != blank, ext[s] != ext[s-2]]) + logp[t, ext[s]]
 *   (one fp32 add after an exact max).  Ties go to the smaller jump (stay, then s-1, then s-2); at the end the trailing
 *   blank 2S_b wins over the last label 2S_b - 1 unless the label is strictly better.
 * Outputs: score[b] = alpha at the chosen end state = max over CTC paths of sum_t logp[t, path_t] (-inf: no path, i.e.
 * T_b < S_b + adjacent repeats with finite log-probs; 0 for T_b = S_b = 0); labels (B,T) class of each frame on the path
 * (0 = blank), tok (B,T) index j of the target token the frame emits (-1: blank), start / end (B,S) first frame and one
 * past the last frame of token j.  Frames t >= T_b, tokens j >= S_b and every output of a row without a path are -1.
 * A target id outside [1, V) is found on the device: that row gets score NaN and -1 outputs (the call returns 0).
 * Error (non-zero return): S > 511.  work: nbasr_ctc_align_work_bytes(B, T, S) bytes = 8 * B * T * ceil((2S+1)/32) when
 * the backpointers (2 bits per frame and state) do not fit in shared memory, i.e. ceil((2S+1)/32) * (T + 32) > 25 600;
 * 0 otherwise, and work may then be NULL. */
int nbasr_ctc_align(const float* logp, int B, int T, int V, const int32_t* targets, int S,
                    const int64_t* audio_len, int len_div, const int64_t* targets_len,
                    int32_t* labels, int32_t* tok, int32_t* start, int32_t* end, float* score,
                    void* work, void* stream);
int64_t nbasr_ctc_align_work_bytes(int B, int T, int S);

/* Greedy CTC decode + fold + Levenshtein PER (trainer.py:229-247 with beam search replaced by
 * argmax/merge-repeats/drop-blank, tf/metrics/ctc.py:76-81; fold encoder.py:64-74 via `lut`
 * (V entries) or NULL).  Outputs: hyp (B,T) int32 folded hypotheses, hyp_len (B), dist (B) edit
 * distances, per[0] = mean_b dist/ref_len in fp64 (sequential), per[1] = same as fp32 in a float
 * slot.  work: B*(S+2) int32. */
int nbasr_greedy_per(const float* logp, int B, int T, int V, const int64_t* audio_len, int len_div,
                     const int32_t* targets, int S, const int64_t* targets_len, const int32_t* lut,
                     int32_t* hyp, int32_t* hyp_len, int32_t* dist, double* per, int32_t* work,
                     void* stream);

/* CTC prefix beam search + fold + Levenshtein PER: what Trainer.decode calls in the reference (trainer.py:71,236:
 * ctcdecode.CTCBeamDecoder(labels, beam_width=12, log_probs_input=True), defaults cutoff_top_n=40, no LM).  Same
 * arguments as nbasr_greedy_per plus beam_width (<= 16) and cutoff_top_n (<= 0: all classes); raw (B,T) / raw_len (B)
 * receive the unfolded best prefix of every utterance. */
int nbasr_beam_per(const float* logp, int B, int T, int V, const int64_t* audio_len, int len_div, int beam_width,
                   int cutoff_top_n, const int32_t* targets, int S, const int64_t* targets_len, const int32_t* lut,
                   int32_t* raw, int32_t* raw_len, int32_t* hyp, int32_t* hyp_len, int32_t* dist, double* per,
                   int32_t* work, void* stream);

/* Phone error breakdown: the Levenshtein alignment behind nbasr_greedy_per / nbasr_beam_per's dist, per utterance b.
 *   hyp = hyp[b, :min(H, hyp_len[b])] exactly as those calls write it (folded, no zeros; NOT folded again: the effective
 *   fold table is not idempotent); ref = targets[b, :min(S, targets_len[b])] mapped through lut (V entries, or NULL) with
 *   the tokens that map to 0 dropped -- what greedy_per compares against.  n = |hyp|, m = |ref|.
 *   D(i, j) over hyp prefix i and ref prefix j: D(i, 0) = i, D(0, j) = j,
 *   D(i, j) = min(D(i-1, j-1) + [hyp[i-1] != ref[j-1]], D(i, j-1) + 1, D(i-1, j) + 1);  D(n, m) = dist.
 *   A diagonal step is a hit (equal labels) or a substitution, a step j-1 a DELETION (ref token aligned to nothing), a step
 *   i-1 an INSERTION (hyp token aligned to nothing).  Tie rule: backtrace from (n, m) taking at each cell the first move on
 *   an optimal path in the order diagonal, deletion, insertion (on the borders the only move) -- among all minimum-cost
 *   alignments, the one whose move sequence read from the end is lexicographically smallest.
 * Outputs: counts (B, 4) = [hits, substitutions, deletions, insertions] (hits + S + D = m, hits + S + I = n,
 * S + D + I = dist); ref_at (B, H) ref position aligned to each hyp position (-1: insertion, and past n); hyp_at (B, S) hyp
 * position aligned to each ref position (-1: deletion, and past m); positions are those of the compared sequences.
 * confusion (V, V) is ADDED INTO (sum a corpus over calls): confusion[ref class * V + hyp class] += 1 per aligned pair, row
 * 0 counting insertions and column 0 deletions.  Integer atomics: deterministic.
 * A row with a target id outside [0, V) (before or after lut) or a hyp id outside [1, V) is refused on the device: counts
 * and alignments -1, nothing added to confusion (the call returns 0).  Errors (non-zero return): H or S >= 32 768, V > 64,
 * or the sequences and three anti-diagonals, H + 7S + 6 bytes, exceeding 220 KB of shared memory.
 * work: nbasr_edit_align_work_bytes(B, H, S) bytes = 8 * B * (H + S + 1) * ceil((S + 1) / 32) when the backpointers (2 bits
 * per cell) do not fit in shared memory beside the sequences; 0 otherwise, and work may then be NULL. */
int nbasr_edit_align(const int32_t* hyp, const int32_t* hyp_len, int H, const int32_t* targets, int S,
                     const int64_t* targets_len, const int32_t* lut, int B, int V, int32_t* counts, int32_t* ref_at,
                     int32_t* hyp_at, uint64_t* confusion, void* work, void* stream);
int64_t nbasr_edit_align_work_bytes(int B, int H, int S);

/* Optimiser tail of Trainer.step (trainer.py:221-225): regulariser 0.01*sum_i ||W_i||_F over the
 * PadConvRelu weights (segments), clip_grad_norm_(5), Adam(eps=1e-7).  Flat fp32 buffers of n
 * elements.  seg_off/seg_len (nseg, int64, device) delimit the regularised tensors.
 * seg_chunks = sum_s ceil(seg_len[s]/16384) (grid size of the per-segment kernels).
 * state: [0]=step count (as float), [1]=lr, [2]=||grad||^2, [3]=clip coef, [4..4+nseg) per-segment ||W||^2, then
 *        scratch from [8+nseg): 592 + seg_chunks per-block partial sums -> 8 + nseg + 592 + seg_chunks floats in all.
 *        All on device, so the step is graph-replayable.  Reductions are deterministic (partials summed in a fixed
 *        order): replicas fed the same all-reduced gradient stay bit-identical. */
int nbasr_optim_step(float* param, float* grad, float* m, float* v, int64_t n, const int64_t* seg_off,
                     const int64_t* seg_len, int nseg, int64_t seg_chunks, float reg_coef, float max_norm,
                     float beta1, float beta2, float eps, float* state, void* stream);

/* Per-tensor statistics of the zero-cost architecture proxies over the same flat fp32 buffers and segment table format as
 * nbasr_optim_step: out[2*s] = sum g^2 and out[2*s + 1] = sum |param * grad| over segment s, products and sums in fp64.
 * part: 2 * seg_chunks doubles of scratch.  Deterministic: fixed 16384-element chunks, partials summed in chunk order. */
int nbasr_param_stats(const float* param, const float* grad, const int64_t* seg_off, const int64_t* seg_len, int nseg,
                      int64_t seg_chunks, double* part, double* out, void* stream);

/* Gradient signal-to-noise of the ZiCo proxy (Li et al. 2023) over N gradient samples of the same flat buffer
 * (2 <= N <= 16; other N is an error): sample k of parameter i is g[k*g_stride + i].  Per parameter, in fp64:
 *   m = sum_k g_k / N,  var = sum_k (g_k - m)^2 / N,  included iff var > 0 (the samples are not all equal),
 *   r = (sum_k |g_k| / N) / sqrt(var).
 * out[2*s] = sum of r over the included parameters of segment s, out[2*s + 1] = their number (an exact double).
 * Segment table, part (2 * seg_chunks doubles) and determinism as in nbasr_param_stats. */
int nbasr_grad_snr(const float* g, int64_t g_stride, int N, const int64_t* seg_off, const int64_t* seg_len, int nseg,
                   int64_t seg_chunks, double* part, double* out, void* stream);

/* Row Gram matrix and row sums of a (B, D) fp32 matrix with row pitch ld (B <= 128), in fp64:
 * gram[i*B + j] = sum_d x[i*ld + d] * x[j*ld + d],  rowsum[i] = sum_d x[i*ld + d].
 * work: ceil(D / 256) * (B*(B+1)/2 + B) doubles.  Deterministic (256-column chunks summed in chunk order).
 * Used on a padded channels-last input gradient (ld = D = Tp*C): its zero pad rows add nothing. */
int nbasr_row_gram(const float* x, int B, int64_t D, int64_t ld, double* gram, double* rowsum, double* work, void* stream);

/* One ReLU layer of the NASWOT proxy: a gate-bit mask in the plane-major format of nbasr_epilogue (mask_out) over the
 * padded rows of one encoder block; frame t of utterance b is row b*Tp + NBASR_PAD_L + t. */
typedef struct nbasr_gate_layer {
  const void* mask;
  int64_t mask_rows;    /* rows per plane */
  int32_t w;            /* plane width: 32 (4-byte entries), 40 or 48 (8-byte entries) */
  int32_t C;            /* channels: columns >= C of the last plane and bits >= w of an entry are ignored */
  int32_t Tp;           /* rows per utterance */
  int32_t T;            /* frames of the block */
  int32_t s;            /* valid frames of utterance b: L = min(T, ceil(audio_len[b] / 2^s)) */
  int32_t reserved;
} nbasr_gate_layer;

/* NASWOT kernel matrix (Mellor et al. 2021) over gate bits m = (0 < z <= relu_hi):
 *   K[i*B + j] = sum over layers, frames t < min(L_i, L_j), channels c < C of [m_i(t, c) == m_j(t, c)]   (both triangles).
 * layers: DEVICE array of nlayers (<= 1024) entries; audio_len (B) int64; 1 <= B <= 128 (larger B is an error).
 * work: nbasr_gate_gram_work_elems(B) uint64.  Exact integer sums: deterministic.  Every entry of K is written. */
int nbasr_gate_gram(const nbasr_gate_layer* layers, int nlayers, const int64_t* audio_len, int B, uint64_t* K,
                    uint64_t* work, void* stream);
int64_t nbasr_gate_gram_work_elems(int B);

/* Batched operand refresh: ONE launch executes a device-resident table of pack jobs (what
 * nbasr_convert / nbasr_pack_weight / nbasr_pack_gconv_mma / nbasr_pack_gconv_dgrad do one at a time).
 * jobs: device array of n nbasr_pack_job; blockmap: device int32 pairs (job, chunk), one per thread block.  A chunk is
 * 4096 consecutive output elements (ceil(n_out / 4096) chunks per job), except for kind 1 (transposes), where a chunk is
 * one 64 x 64 (m, n) tile of one tap: nq * ceil(M / 64) * ceil(N / 64) chunks, tile_n fastest, then tile_m, then q;
 * and for kind 2, where chunks walk the C * cpg * ktaps SOURCE weights and only the diagonal blocks of the pack are
 * rewritten (the caller zero-fills the pack buffer once). */
typedef struct nbasr_pack_job {
  int32_t kind;          /* 0 convert, 1 pack_weight, 2 pack_gconv_mma, 3 pack_gconv_dgrad, 4 LSTM W_hh cluster pack (a[0]=H) */
  int32_t out_dtype;
  const float* src;
  void* dst;
  int64_t n_out;         /* output elements */
  int32_t a[8];          /* kind 1: M,N,nq,t0,tstep ; kind 2: C,cpg,ktaps,transposed ; kind 3: C,cpg,ktaps */
  int64_t s[3];          /* kind 1: ws_m, ws_n, ws_t */
} nbasr_pack_job;
int nbasr_pack_batch(const nbasr_pack_job* jobs, int n, const int32_t* blockmap, int64_t blocks, void* stream);

/* Log-mel front end (training/torch/timit.py:90-95: torchaudio MelSpectrogram(16 kHz, n_fft = win = 400, hop 160,
 * 80 mels) -> log -> (x - mean) / (var + eps), then the zero padding of collate_fn, timit.py:104).
 * wav (B, L) fp32 zero padded, len[b] samples (> 200); dft (402, 400) fp32 = Hann-windowed cos | -sin rows,
 * melfb (80, 208) fp32 = transposed HTK filterbank (201 bins, zero padded); mean / var (80).
 * out (B, 80, T) fp32 with T >= 1 + L / 160: frames t < 1 + len[b] / 160 hold the features, the rest 0.
 * work: nbasr_logmel_work_floats(B, L) floats. */
int nbasr_logmel(const float* wav, const int64_t* len, int B, int64_t L, const float* dft, const float* melfb,
                 const float* mean, const float* var, float eps, float* out, int T, float* work, int64_t work_floats,
                 void* stream);
int64_t nbasr_logmel_work_floats(int B, int64_t L);

/* misc */
int nbasr_fill_u32(uint32_t* p, uint32_t val, int64_t n, void* stream);
int nbasr_version(void);
int nbasr_sm_count(void);
const char* nbasr_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
