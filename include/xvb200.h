/*
 * xvb200.h -- C ABI of libxvb200.so, the B200 (sm_100a) x-vector extraction / back-end scoring
 * library that stands in for the hot path of Snowdar/asv-subtools.
 *
 * The reference has no native FFI for this path: its "kernels" are ATen calls issued from
 * Python (SURVEY.md section 2).  The entry points below are therefore what a ctypes stub in the
 * reference tree would bind to replace those calls; each one cites the reference code whose
 * arithmetic it takes over (paths relative to the reference root).  INTEGRATION.md shows the
 * stub.  Conventions:
 *
 *   - plain C, no C++/torch types; every pointer is a raw device pointer unless the name ends
 *     in _host; sizes are explicit; nothing is allocated behind the caller's back except by
 *     the xvb_extractor_* object, which owns its packed weights and workspace;
 *   - every function returns 0 on success or a negative XVB_E* code; xvb_last_error() gives
 *     the message (thread-local);
 *   - device functions are asynchronous on the caller-supplied cudaStream_t (passed as void*);
 *   - frame matrices are channel-contiguous "(B, T, C)" (the reference is (B, C, T); Kaldi
 *     features arrive as (T, F), so no transpose is needed on the way in);
 *   - "split planes": an fp32 tensor stored as two bf16 tensors hi = bf16(x), lo = bf16(x-hi)
 *     (same bytes as fp32).  The tcgen05 GEMM consumes them as x*w ~= hi*whi + lo*whi + hi*wlo
 *     with fp32 accumulation in TMEM (|error| <= ~3 * 2^-18 |x w| per product), which is what
 *     keeps the stack within the 1e-4 parity budget at bf16 tensor-core rate.
 *
 * There is no CPU fallback anywhere in this library: on a machine without an sm_100 device
 * every compute entry point fails with XVB_ENODEVICE.
 */
#ifndef XVB200_H_
#define XVB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XVB_VERSION 100

/* error codes */
#define XVB_OK 0
#define XVB_EINVAL (-1)    /* bad argument (shape, alignment, null pointer) */
#define XVB_ECUDA (-2)     /* a CUDA runtime/driver call failed; see xvb_last_error() */
#define XVB_ENODEVICE (-3) /* no sm_100 GPU visible */
#define XVB_ESTATE (-4)    /* object used in the wrong state (e.g. extract before finalize) */

/* epilogue flags for xvb_tdnn_affine* (order is fixed: +bias -> ReLU -> BN affine) */
#define XVB_RELU 1 /* components.py:410-416 (_relu_bn_forward): ReLU first ... */
#define XVB_BN 2   /* ... then eval-mode BatchNorm folded to y*scale[c] + shift[c] */
#define XVB_SIGMOID 4 /* ... then sigmoid (SE gate, ecapa_tdnn_xvector.py:97-106) */
#define XVB_TANH 8    /* ... then tanh (attention bottleneck, ecapa_tdnn_xvector.py:164-168) */

#define XVB_MAX_TAPS 16

int xvb_version(void);
const char* xvb_last_error(void);
/* 0 if the current device is sm_100 (B200); XVB_ENODEVICE otherwise. */
int xvb_device_check(void);

/* ---------------------------------------------------------------------------------------------
 * Frame-matrix staging
 * ------------------------------------------------------------------------------------------- */

/* fp32 (rows, C) with row pitch ldx  ->  split planes (rows, ldp); columns [C, ldp) are zeroed.
 * Replaces the torch.tensor(input)/unsqueeze/transpose staging of for_extract_embedding,
 * pytorch/libs/nnet/framework.py:28-33.  ldp % 8 == 0. */
int xvb_split_f32(const float* x, int64_t rows, int C, int64_t ldx, uint16_t* hi, uint16_t* lo, int64_t ldp,
                  void* stream);

/* Pack a TdnnAffine weight.  w: (Cout, Cin, tot_context) fp32 exactly as stored in the
 * reference state_dict, *including* the masked taps (pytorch/libs/nnet/components.py:62,
 * :78-83); only the taps listed in context[] are kept (the weight*mask of :133-138).
 * Output planes are K-major (Cout, ntaps*cin_p16) with cin_p16 = round_up(Cin,16) and
 * K index = tap*cin_p16 + c.  Size in elements: xvb_packed_weight_elems(). */
/* (B, T, C) fp32 frames -> split planes with `pad_front` / `pad_back` zero frames around every
 * utterance: planes are (B, pad_front + T + pad_back, ldp).  The zero frames are F.pad of
 * TdnnAffine.forward (components.py:117) made explicit, for the im2col view of xvb_tdnn_args_t. */
int xvb_split_frames(const float* x, int B, int T, int C, uint16_t* hi, uint16_t* lo, int64_t ldp, int pad_front,
                     int pad_back, void* stream);
int64_t xvb_packed_weight_elems(int Cout, int Cin, int ntaps);
int xvb_pack_tdnn_weight(const float* w, int Cout, int Cin, int tot_context, int left_context, const int* context_host,
                         int ntaps, uint16_t* w_hi, uint16_t* w_lo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * TDNN layer:  y[b,t,:] = epilogue( bias + sum_{c in context} W_c . x[b,t+c,:] ),  x = 0 outside
 * [0,T) -- TdnnAffine.forward (components.py:107-149) fused with ReLU/BatchNorm of
 * _BaseActivationBatchNorm (components.py:410-431).
 *
 * xvb_tdnn_affine: tcgen05 (bf16x3 split, fp32 accumulate in TMEM) GEMM with M = B*T frames,
 * K = ntaps*Cin, N = Cout; the context splice is done by TMA (3-D tensor map (C,T,B), time
 * coordinate offset per tap, out-of-bounds zero fill == F.pad).  Outputs: split planes
 * (y_hi,y_lo; may be NULL) and/or fp32 (y_f32; may be NULL); the TMA store clips ragged T / B /
 * Cout.  Requirements: ldx % 8 == 0, ldy % 8 == 0, ldyf % 4 == 0; pointers 16-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int xvb_tdnn_affine(const uint16_t* x_hi, const uint16_t* x_lo, int64_t ldx, const uint16_t* w_hi,
                    const uint16_t* w_lo, const float* bias, const float* bn_scale, const float* bn_shift, int flags,
                    const int* context_host, int ntaps, uint16_t* y_hi, uint16_t* y_lo, int64_t ldy, float* y_f32,
                    int64_t ldyf, int B, int T, int Cin, int Cout, void* stream);

/* Extended form of the same kernel (everything xvb_tdnn_affine does, plus what ECAPA-TDNN and the
 * PLDA scorer need).  Zero-initialise the struct; unused pointers stay NULL.
 *   x2_*      : second A source with the same shape; computes W.(x + x2) by accumulating both
 *               sources into the same TMEM accumulator (Res2Net "sp + spx[i+1]",
 *               pytorch/model/ecapa_tdnn_xvector.py:66-71) -- no elementwise pass, no extra launch;
 *   row_bias  : per frame (B*T) additive term (PLDA row term);
 *   utt_bias  : per utterance x column (B, Cout) additive term, pitch ld_utt_bias (the
 *               time-constant [mean,std] part of AttentiveStatsPool's first conv, :173-180);
 *   both plane and fp32 outputs may be requested together. */
typedef struct xvb_tdnn_args {
  const uint16_t* x_hi; const uint16_t* x_lo; int64_t ldx;
  const uint16_t* x2_hi; const uint16_t* x2_lo; int64_t ldx2;
  const uint16_t* w_hi; const uint16_t* w_lo;
  const float* bias; const float* bn_scale; const float* bn_shift;
  const float* row_bias;
  const float* utt_bias; int64_t ld_utt_bias;
  int flags;
  const int* context_host; int ntaps;
  uint16_t* y_hi; uint16_t* y_lo; int64_t ldy;
  float* y_f32; int64_t ldyf;
  int B, T, Cin, Cout;
  /* Fused statistics pooling (no other output): the epilogue reduces each tile's frames per
   * utterance and writes [mean | centred sum of squares] partials, (num_blocks, B, 2*Cout) fp32 with
   * num_blocks = xvb_pool_partial_blocks(B, T, &frames_per_block); merge with xvb_pool_finalize. */
  float* pool_partial;
  /* 0: utterance b starts at row b*T of the x planes.  Otherwise the element distance between
   * utterances, and ldx may then be smaller than Cin: row t is the Cin-long window starting at
   * x[b*x_batch_stride + t*ldx] -- an im2col VIEW of consecutive context taps over a time-padded
   * frame matrix (ntaps = 1, Cin = taps*channels), so a [-2..2] layer over 80 channels streams 7
   * channel blocks of 64 instead of 5 x (64 + 16).  Requires x2_* == NULL. */
  int64_t x_batch_stride;
  /* Ragged batch: (B) int32 on the device, utterance b has lengths[b] valid frames (1 <= lengths[b] <= T);
   * NULL: all T frames are valid.  Rows t >= lengths[b] of the plane / fp32 outputs are stored as exact
   * zeros, so the next layer's taps past the end read what F.pad (components.py:117) gives the
   * reference's one-utterance-at-a-time extraction (extract_embeddings.py:73-83); with pool_partial the
   * epilogue counts lengths[b] frames (merge with the extractor's ragged path).  Ignored by the
   * segment-level (T == 1, split-K) layers. */
  const int32_t* lengths;
} xvb_tdnn_args_t;
int xvb_tdnn_affine_ex(const xvb_tdnn_args_t* args, void* stream);
/* Time blocking the fused-pooling epilogue will use for a (B, T) batch. */
int xvb_pool_partial_blocks(int B, int T, int* frames_per_block);
/* Merge the fused-pooling partials into StatisticsPooling's output (mode as in xvb_stats_pool_ex):
 * Chan's parallel update over the time blocks, i.e. the two-pass result of pooling.py:58-67
 * without ever materialising the (B, T, C) tensor. */
int xvb_pool_finalize(const float* partial, int num_blocks, int frames_per_block, int B, int T, int C, float eps,
                      int mode, float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

/* Same layer on CUDA cores in plain fp32 straight from the *unpacked* reference weight
 * (Cout, Cin, tot_context).  Slow; exists so the tensor-core path and the weight packer can
 * be cross-checked on the device and for shapes the tcgen05 path rejects. */
int xvb_tdnn_affine_simt(const float* x, int64_t ldx, const float* w, int tot_context, int left_context,
                         const float* bias, const float* bn_scale, const float* bn_shift, int flags,
                         const int* context_host, int ntaps, float* y, int64_t ldy, int B, int T, int Cin, int Cout,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * Statistics pooling: StatisticsPooling.forward, no-lengths branch
 * (pytorch/libs/nnet/pooling.py:58-67): out[b, 0:C] = mean_t x, out[b, C:2C] =
 * sqrt(max(sum_t (x-mean)^2 / T, eps)).  x: (B, T, C) fp32 pitch ldx (ldx % 4 == 0, C % 4 == 0).
 * One HBM read of x.  out: (B, 2C) fp32; out_hi/out_lo (optional, pitch ldo % 8 == 0) receive
 * the same values as split planes for the following segment-level GEMM.
 * ------------------------------------------------------------------------------------------- */
int xvb_stats_pool(const float* x, int64_t ldx, int B, int T, int C, float eps, float* out, uint16_t* out_hi,
                   uint16_t* out_lo, int64_t ldo, void* stream);

/* mode 0 = xvb_stats_pool; mode 1 = the global context of ECAPA's AttentiveStatsPool
 * (pytorch/model/ecapa_tdnn_xvector.py:175-178): std = sqrt(unbiased_var + eps). */
int xvb_stats_pool_ex(const float* x, int64_t ldx, int B, int T, int C, float eps, int mode, float* out,
                      uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ECAPA-TDNN pieces that are not contractions (pytorch/model/ecapa_tdnn_xvector.py)
 * ------------------------------------------------------------------------------------------- */

/* Mean over time of a split-plane tensor (B,T,C) -> (B,C) fp32 and/or planes: the
 * AdaptiveAvgPool1d(1) of SE_Connect (:100).  C % 8 == 0. */
int xvb_plane_mean(const uint16_t* x_hi, const uint16_t* x_lo, int64_t ldx, int B, int T, int C, float* out,
                   uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

/* Res2NetBlock.forward (pytorch/model/ecapa_tdnn_xvector.py:61-75) as ONE persistent kernel: chunk 0
 * of x passes through; step i = TDNN 128->128, context [-d,0,d], ReLU, BN on (x chunk i+1 [+ y chunk i]),
 * written to y chunk i+1.  A CTA owns whole utterances and walks them through all scale-1 steps, so the
 * serial chain needs no grid-wide synchronisation and no per-step launches.  x, y: split planes
 * (B,T,scale*128) with pitches ldx/ldy (distinct tensors).  w_hi/w_lo: the scale-1 packed weights
 * (xvb_pack_tdnn_weight, each (128, 3*128)) stacked along rows; bias/bn_scale/bn_shift: (scale-1, 128). */
int xvb_res2net_block(const uint16_t* x_hi, const uint16_t* x_lo, int64_t ldx, const uint16_t* w_hi, const uint16_t* w_lo,
                      const float* bias, const float* bn_scale, const float* bn_shift, int dilation, int scale,
                      uint16_t* y_hi, uint16_t* y_lo, int64_t ldy, int B, int T, void* stream);

/* Strided row copy (16-byte granularity): the pass-through of Res2Net's first chunk
 * (ecapa_tdnn_xvector.py:63-64) between two channel-slice views. */
int xvb_copy_rows(const void* src, int64_t src_pitch_bytes, void* dst, int64_t dst_pitch_bytes, int64_t rows,
                  int64_t row_bytes, void* stream);

/* out = z * gate[b,:] + in  and optionally next = in + out, all split planes (B,T,C): the SE
 * scaling + residual of SE_Res2Block.forward (:109-111, :149) fused with the running sums
 * x+x1, x+x1+x2 of ECAPA_TDNN.extract_embedding (:405-408).  gate: (B,C) fp32. */
int xvb_se_apply(const uint16_t* z_hi, const uint16_t* z_lo, int64_t ldz, const uint16_t* in_hi, const uint16_t* in_lo,
                 int64_t ldin, const float* gate, uint16_t* out_hi, uint16_t* out_lo, int64_t ldout, uint16_t* next_hi,
                 uint16_t* next_lo, int64_t ldnext, int B, int T, int C, void* stream);

/* AttentiveStatsPool.forward tail (:183-188): alpha = softmax_T(logits); mean = sum alpha x;
 * std = sqrt(max(sum alpha x^2 - mean^2, floor)); out (B,2C) = [mean | std].  One streaming pass
 * over logits and x (both (B,T,C) fp32) with an online softmax. */
int xvb_attn_stats_pool(const float* logits, int64_t ldl, const float* x, int64_t ldx, int B, int T, int C, float floor_,
                        float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

/* LDEPooling.forward (libs/nnet/pooling.py:130-162): x (B,T,C) fp32, dictionary mu (C,K) fp32 as the state_dict stores
 * it, neg_beta[k] = -(s_k^2 + eps); w[t,k] = softmax_k(neg_beta[k] * sum_c (x[t,c] - mu[c,k])^2) (distances summed directly
 * in fp32), out[b, c*K + k] = mean_t w[t,k] (x[t,c] - mu[c,k]); out (B, C*K) fp32, optionally also split planes.
 * w_scratch: (B*T, K) fp32.  K <= 64. */
int xvb_lde_pool(const float* x, int64_t ldx, int B, int T, int C, const float* mu, int K, const float* neg_beta,
                 float* w_scratch, float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

/* Segment-level affine on CUDA cores, fp32 throughout: y[b,n] = epi(bias[n] + sum_k w[n,k] x[b,k]) for the few rows
 * (one per utterance) of the SE gate's two 1x1 convolutions (ecapa_tdnn_xvector.py:97-111), the time-constant half of
 * the attention's first conv (:179-181) and fc2 (:412-422).  x (B, >=K) fp32 pitch ldx, w (N, K) fp32 exactly as the
 * state_dict stores a kernel-size-1 conv weight; flags XVB_RELU | XVB_BN | XVB_SIGMOID | XVB_TANH applied in that
 * order after the bias; y fp32 (pitch ldy) and/or split planes (pitch ldplane).  K % 4 == 0. */
int xvb_small_affine(const float* x, int64_t ldx, const float* w, int B, int K, int N, const float* bias,
                     const float* bn_scale, const float* bn_shift, int flags, float* y, int64_t ldy, uint16_t* y_hi,
                     uint16_t* y_lo, int64_t ldplane, void* stream);

/* The attention poolings of libs/nnet/pooling.py with shared / per-head weights: AttentiveStatisticsPooling
 * (:322-368), MultiHeadAttentionPooling (:371-440), Global / MultiResolution multi-head (:443-587).  logits
 * (B,T,G) fp32 are the output of AttentionAlphaComponent's last affine (:300-319; temperature folded into its
 * weights); output channel o in [0,O) pools input channel o % C of x (B,T,C) with alpha = softmax_T(logits[:,:,o/gdiv]):
 * mean = sum alpha x, std = sqrt(max(sum alpha x^2 - mean^2, floor)) (unweighted_var = 1: the `stddev_attention=False`
 * branch, mean_T((x-mean)^2)).  out (B,2O) = [mean | std], optionally also as split planes. */
int xvb_attn_head_stats_pool(const float* logits, int64_t ldl, int G, const float* x, int64_t ldx, int B, int T, int C,
                             int O, int gdiv, float floor_, int unweighted_var, float* out, uint16_t* out_hi,
                             uint16_t* out_lo, int64_t ldo, void* stream);
/* The xi-vector pooling (xivec_stdinit_softplus2_prec_pooling, pooling.py:165-212) on the same kernel: softplus2log = 1
 * turns the raw logit z (output of `lin2`) into a frame log-precision 2 log(softplus(z)) (:189-190); prior_logit / prior_x
 * (C each, may be NULL) add the prior as a (T+1)-th element of the softmax and of the weighted sums (:194-202).  out =
 * [phi | sqrt(max(sum w x^2 - phi^2, floor))]: the post-mean variant uses the first half. */
int xvb_attn_head_stats_pool_prior(const float* logits, int64_t ldl, int G, const float* x, int64_t ldx, int B, int T, int C,
                                   int O, int gdiv, float floor_, int unweighted_var, const float* prior_logit,
                                   const float* prior_x, int softplus2log, float* out, uint16_t* out_hi, uint16_t* out_lo,
                                   int64_t ldo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Feature-side front-end (SURVEY 8f rank 1) on a ragged batch: utterance u owns rows
 * offsets[u] .. offsets[u+1] of the (sum_T, F) fp32 matrix x.
 * ------------------------------------------------------------------------------------------- */

/* Energy VAD: TorchAsvExtractor::ComputeVadEnergy, runtime/extractor/torch_asv_extractor.cc:14-62
 * (column 0 = log-energy; threshold += mean_scale * mean(log-energy); a frame is voiced when at least
 * proportion_threshold of its +-frames_context neighbours exceed the threshold).  voiced: (sum_T)
 * bytes 0/1; voiced_counts: (U) number of voiced frames per utterance. */
int xvb_vad_energy(const float* x, const int32_t* offsets, int num_utts, int F, float energy_threshold,
                   float energy_mean_scale, int frames_context, float proportion_threshold, uint8_t* voiced,
                   int32_t* voiced_counts, void* stream);

/* Cepstral mean normalisation, no variance norm.  window <= 0: per-utterance mean
 * (torch_asv_extractor.cc:99-101).  window > 0: Kaldi apply-cmvn-sliding --center=true
 * --cmn-window=window as used by pytorch/pipeline/extract_xvectors_for_pytorch.sh:105-111. */
int xvb_cmn(const float* x, const int32_t* offsets, int num_utts, int F, int window, float* y, void* stream);

/* Keep the voiced frames of every utterance, order preserved (torch_asv_extractor.cc:103-107,
 * Kaldi select-voiced-frames).  out_offsets (U+1) = exclusive prefix sum of the voiced counts. */
int xvb_select_frames(const float* x, const int32_t* offsets, const uint8_t* voiced, const int32_t* out_offsets,
                      int num_utts, int F, float* y, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Back-end scoring
 * ------------------------------------------------------------------------------------------- */

/* y = (x - mean) / ||x - mean||_2 per row.  mean may be NULL.  Covers `submean` + `norm` of
 * score/process.sh:181-203 (ivector-subtract-global-mean, ivector-normalize-length
 * --scaleup=false). */
int xvb_center_length_norm(const float* x, const float* mean, float* y, int64_t rows, int D, void* stream);

/* Column mean of (rows, D): `getmean`, score/process.sh:169-179 (ivector-mean). */
int xvb_column_mean(const float* x, int64_t rows, int D, float* mean, void* stream);

/* Per-trial dot products: score/score.sh:82-97 (ivector-compute-dot-products).
 * scores[i] = <enroll[trial_e[i]], test[trial_t[i]]>. */
int xvb_cosine_trials(const float* enroll, const float* test, int D, const int32_t* trial_e, const int32_t* trial_t,
                      int64_t num_trials, float* scores, void* stream);

/* Per-speaker mean of embeddings: `mean` of score/process.sh:156-167 (ivector-mean ark:spk2utt).
 * CSR lists: speaker s owns rows members[offsets[s] .. offsets[s+1]) of x (N,D); out (S,D).
 * num_utts[s] = offsets[s+1]-offsets[s] is known to the caller. */
int xvb_speaker_mean(const float* x, int D, const int32_t* offsets, const int32_t* members, int num_spk, float* out,
                     void* stream);

/* Score normalisation (score/ScoreNormalization.py).  xvb_topn_mean_std: per row of a cohort score
 * matrix S (rows, ncoh), mean and unbiased std of the top_n largest entries (top_n <= 0: all) --
 * groupby().head(top_n) + .mean()/.std() of :151-166 (AS-norm) / :93-98 (S-norm).  xvb_snorm_trials:
 * out = 0.5*((s-mean_e[e])/std_e[e] + (s-mean_t[t])/std_t[t]) per listed trial (:101-104, :172-173). */
int xvb_topn_mean_std(const float* S, int64_t lds, int64_t rows, int ncoh, int top_n, float* mean, float* stdv,
                      void* stream);
/* The same with the divisor of the variance stated: ddof = 1 is pandas' .std() (ScoreNormalization.py:163-166),
 * ddof = 0 is np.std of subtools2/egrecho/score/asnorm.py:137-140 (`compute_cohort_stats`). */
int xvb_topn_mean_std_ddof(const float* S, int64_t lds, int64_t rows, int ncoh, int top_n, int ddof, float* mean,
                           float* stdv, void* stream);
int xvb_snorm_trials(const float* scores, const int32_t* trial_e, const int32_t* trial_t, int64_t num_trials,
                     const float* mean_e, const float* std_e, const float* mean_t, const float* std_t, float* out,
                     void* stream);

/* Per-trial bilinear scores with optional per-row / per-column terms:
 * scores[i] = <enroll[te[i]], test[tt[i]]> + row_term[te[i]] + col_term[tt[i]]  (terms may be NULL).
 * With enroll := E.(Lambda+Lambda^T) and the xvb_plda_terms() vectors this is PLDAScoring
 * (score/pyplda/gaussian-plda-scoring.py:23-29) for each listed trial (main loop :78-84). */
int xvb_bilinear_trials(const float* enroll, const float* test, int D, const int32_t* trial_e, const int32_t* trial_t,
                        int64_t num_trials, const float* row_term, const float* col_term, float* scores, void* stream);

/* y (rows, Dout) = x (rows, D) . M^T with M (Dout, D) row-major, Dout % 4 == 0: the small
 * projections of the back-end (PLDA's E.(Lambda+Lambda^T); `lda`/`whiten` transforms applied by
 * ivector-transform in score/process.sh:205-233).  Runs on the tcgen05 layer kernel. */
int xvb_project(const float* x, int64_t rows, int D, const float* M, int Dout, float* y, void* stream);

/* All-pairs score matrix S (Ne, Nt) = enroll . test^T (BASELINE config 4). */
int xvb_cosine_matrix(const float* enroll, int64_t Ne, const float* test, int64_t Nt, int D, float* S, int64_t lds,
                      void* stream);

/* Two-covariance PLDA, score/pyplda/gaussian-plda-scoring.py:23-29 in matrix form:
 * S[i,j] = e_i^T L2 t_j + row[i] + col[j],  L2 = Lambda + Lambda^T (D,D) fp32,
 * row = diag(E G E^T) + E c, col likewise (see xvb_plda_terms). */
int xvb_plda_terms(const float* x, int64_t rows, int D, const float* gamma, const float* c, float* term, void* stream);
int xvb_plda_matrix(const float* enroll, int64_t Ne, const float* test, int64_t Nt, int D, const float* L2,
                    const float* row, const float* col, float* S, int64_t lds, void* stream);

/* AS-norm with cross selection (score/ScoreNormalization.py:146-160, --cross-select true): the statistics of
 * the enroll side of trial (e, t) are taken over the cohort utterances that are the top_n of the TEST side and
 * vice versa.  xvb_topn_indices: idx (rows, top_n) int32 = cohort indices of every row's top_n scores, best
 * first (ncoh <= 16384); xvb_snorm_cross_trials: out[i] = 0.5 ((s - mu_e)/sd_e + (s - mu_t)/sd_t) with
 * mu_e, sd_e over enroll_cohort[e, top_test[t, :]] and mu_t, sd_t over test_cohort[t, top_enroll[e, :]],
 * std with ddof = 1 like pandas. */
int xvb_topn_indices(const float* S, int64_t lds, int64_t rows, int ncoh, int top_n, int32_t* idx, void* stream);
int xvb_snorm_cross_trials(const float* scores, const int32_t* trial_e, const int32_t* trial_t, int64_t num_trials,
                           const float* enroll_cohort, int64_t lde, const float* test_cohort, int64_t ldt,
                           const int32_t* top_enroll, const int32_t* top_test, int top_n, float* out, void* stream);

/* out (M, N) = a (M, K) . b (N, K)^T + row_bias[i] + col_bias[j] (biases may be NULL), fp32 row-major in
 * and out, N % 4 == 0: the general form behind xvb_project / xvb_cosine_matrix / xvb_plda_matrix. */
int xvb_matmul_nt(const float* a, int64_t M, const float* b, int64_t N, int K, const float* row_bias,
                  const float* col_bias, float* out, int64_t ldo, void* stream);

/* PLDA training on the GPU (score/pyplda/plda_base.py: PldaStats.add_samples :50-66, PldaEstimation
 * .get_stats_from_class_mean :262-287).  The D x D algebra (Cholesky, eigh, inverses) stays on the host in
 * float64; the O(N D^2) parts are Gram products X^T X, computed as xvb_matmul_nt(X^T, X^T) on transposed
 * operands these two kernels emit:
 *   xvb_center_rows_transposed: out[d][i] = sqrt_weight[spk[i]] * (x[i][d] - means[spk[i]][d])   (D, ldo >= N)
 *     -> offset_scatter = out . out^T  (the weighted within-class scatter, without the cancellation of
 *        sum x x^T - n m m^T);
 *   xvb_plda_em_rows: per class k, in the basis where within_var = I and between_var = diag(psi),
 *     what = n psi/(1 + n psi) * u;  what_T[d][k] = sqrt(w_k) what;  resid_T[d][k] = sqrt(w_k n_k) (u - what)
 *     -> the rank-one sums of one EM iteration are what_T . what_T^T and resid_T . resid_T^T. */
int xvb_center_rows_transposed(const float* x, const int32_t* spk, const float* means, const float* sqrt_weight,
                               int64_t N, int D, float* out, int64_t ldo, void* stream);
int xvb_plda_em_rows(const float* u, const float* n, const float* weight, const float* psi, int S, int D, float* what_T,
                     float* resid_T, int64_t ldo, void* stream);

/* Kaldi-style PLDA scoring in the diagonalised space, the arithmetic of ivector-plda-scoring as restated by the
 * reference's score/pyplda/plda_base.py (PLDA.transform_ivector :93-107, get_normalization_factor :151-158,
 * log_likelihood_ratio :109-136; called from score/score.sh:99-121 through the Kaldi binary):
 *   u = transform . x + offset                       -> xvb_matmul_nt with col_bias = offset
 *   u *= sqrt(D / sum_d u_d^2 / (psi_d + 1/n))       -> xvb_plda_normalize_rows (simple: sqrt(D)/||u||)
 *   LLR(i,j) = [t_j^2 | t_j] . [-1/(2 v_i) | m_i/v_i] + term_i + term_j,  m = n psi/(n psi+1) u, v = 1 + psi/(n psi+1)
 *     -> xvb_plda_llr_operands(side 0 = enroll with num_examples n, side 1 = test) writes the (rows, 2D) operand
 *        and the per-row term; the score matrix is xvb_matmul_nt(enroll_operand, test_operand, row, col), listed
 *        trials xvb_bilinear_trials. */
int xvb_plda_normalize_rows(float* u, const float* psi, const float* num_examples, int64_t rows, int D,
                            int simple_length_norm, void* stream);
int xvb_plda_llr_operands(const float* u, const float* psi, const float* num_examples, int64_t rows, int D, int side,
                          float* operand, float* term, void* stream);

/* Fused consumer for score matrices too large to store (BASELINE configs 4/5: 10^12 cosine trials,
 * 10^10 PLDA trials; SURVEY Appendix A "fused consumer"): every score
 *   s(i,j) = <enroll[i], test[j]> + row_term[i] + col_term[j]        (terms may be NULL)
 * is binned in the GEMM epilogue by trial class -- target when enroll_spk[i] == test_spk[j], the
 * trials file's third column (score/score.sh:82-97, computeEER.sh:21-22) -- and only the counters
 * leave the SM.  hist is (2, nbins) uint64 [nontarget | target] and is ACCUMULATED into (zero it
 * first; several calls / shards / GPUs add up).  Bins: w = (hi-lo)/(nbins-2);
 *   bin 0: s < lo;  bin k (1..nbins-2): lo+(k-1)w <= s < lo+kw;  bin nbins-1: s >= hi,
 * evaluated in fp32 as 1 + floor((s - lo) * ((nbins-2)/(hi-lo))).  4 <= nbins <= 2048.
 * symmetric != 0 (needs Ne == Nt, one set on both sides): only pairs j > i are counted, tiles
 * below the diagonal are skipped.  Row sharding for multi-GPU: this call walks the 256-row units
 * unit_first, unit_first + unit_stride, ... of enroll (rank r of W passes r, W). */
int xvb_trial_histogram(const float* enroll, int64_t Ne, const int32_t* enroll_spk, const float* test, int64_t Nt,
                        const int32_t* test_spk, int D, const float* row_term, const float* col_term, int symmetric,
                        int unit_first, int unit_stride, float lo, float hi, int nbins, unsigned long long* hist,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * Whole-model extractor (x-vector TDNN family): owns packed weights + workspace on the current
 * device; replaces Xvector.extract_embedding (pytorch/model/xvector.py:77-98) for a whole batch
 * of equal-length utterances, and the model-loading role of runtime/ (torch_asv_model.cc:8-17).
 * ------------------------------------------------------------------------------------------- */
typedef struct xvb_extractor xvb_extractor_t;

int xvb_extractor_create(xvb_extractor_t** out, int feat_dim);
/* Append a frame-level layer (before pooling) / a segment-level layer (after pooling).
 * w_host: (Cout, Cin, tot_context) fp32 host; bias_host (Cout) or NULL; bn_scale_host/
 * bn_shift_host (Cout) or NULL (folded eval BatchNorm); flags: XVB_RELU | XVB_BN. */
int xvb_extractor_add_frame_layer(xvb_extractor_t* h, int Cout, const int* context_host, int ntaps,
                                  const float* w_host, const float* bias_host, const float* bn_scale_host,
                                  const float* bn_shift_host, int flags);
int xvb_extractor_add_segment_layer(xvb_extractor_t* h, int Cout, const float* w_host, const float* bias_host,
                                    const float* bn_scale_host, const float* bn_shift_host, int flags);
int xvb_extractor_finalize(xvb_extractor_t* h, float pooling_eps);
int xvb_extractor_embed_dim(const xvb_extractor_t* h);
/* feats (B, T, feat_dim) fp32 on the device -> emb (B, embed_dim) fp32 on the device. */
int xvb_extractor_extract(xvb_extractor_t* h, const float* feats, int B, int T, float* emb, void* stream);
/* Same through host buffers (H2D of feats, D2H of emb inside; synchronises the stream). */
int xvb_extractor_extract_host(xvb_extractor_t* h, const float* feats_host, int B, int T, float* emb_host,
                               void* stream);
/* Pipelined host-buffer path: submit returns as soon as the work is queued (H2D on a private copy
 * stream into one of two device slots, the stack and the D2H on `stream`), so the host->device
 * copy of batch i+1 overlaps the kernels of batch i.  feats_host / emb_host must stay valid (and
 * should be pinned) until xvb_extractor_wait(h, slot) returns.  Typical loop:
 *   submit(batch0, slot0); for i>=1 { submit(batch_i, i&1); wait((i-1)&1); } wait(last). */
int xvb_extractor_submit_host(xvb_extractor_t* h, const float* feats_host, int B, int T, float* emb_host, int slot,
                              void* stream);
int xvb_extractor_wait(xvb_extractor_t* h, int slot);
/* A whole shard of N equal-length utterances -- the caller loop of the reference
 * (pytorch/pipeline/onestep/extract_embeddings.py:73-83, one utterance per iteration; sharded over `nj` jobs by
 * extract_xvectors_for_pytorch.sh:125-136) as ONE call: ceil(N / batch) batches through the stack back to back.
 *   _shard      : feats (N, T, feat_dim) and emb (N, embed_dim) on the device; asynchronous on `stream`;
 *   _shard_host : the same through host buffers (pinned, so that the copies overlap): batch i+1 crosses the link
 *                 while batch i runs (the submit/wait protocol above); returns when emb_host is complete.
 * Launch plans (tensor maps, tile geometry) are cached per batch shape, so a batch costs its launches only. */
int xvb_extractor_extract_shard(xvb_extractor_t* h, const float* feats, int64_t N, int T, int batch, float* emb,
                                void* stream);
int xvb_extractor_extract_shard_host(xvb_extractor_t* h, const float* feats_host, int64_t N, int T, int batch,
                                     float* emb_host, void* stream);
/* ---------------------------------------------------------------------------------------------
 * Ragged batches: utterances of different lengths in one call.  The reference extracts one utterance at a time
 * (pytorch/pipeline/onestep/extract_embeddings.py:73-83), every TdnnAffine zero-padding its own input
 * (libs/nnet/components.py:117), and StatisticsPooling averages over that utterance's frames (pooling.py:58-67).
 * A ragged batch reproduces this per utterance: utterance b (L_b >= 1 frames) is padded to Tq = round_up(max L, 32),
 * frame-layer rows t >= L_b are stored as exact zeros, and pooling counts L_b frames.  TDNN x-vector extractors with
 * fused pooling only (XVB_ESTATE if it is switched off or a gather table is set).
 *   _extract_ragged : feats (offsets_host[B], feat_dim) fp32 on the device, utterance b = rows offsets_host[b] ..
 *                     offsets_host[b+1]; emb (B, embed_dim) on the device; asynchronous on `stream` (the lengths are
 *                     uploaded on it from a pinned staging buffer the extractor owns).
 *   _ragged_shard_host : N utterances in host memory (pinned, so that the copies overlap), int64 offsets (N+1)
 *                     into feats_host; batches as xvb_ragged_plan cuts them with max_frames (<= 0: 262144) through
 *                     the pipeline of xvb_extractor_extract_shard_host; emb_host (N, embed_dim) in INPUT order,
 *                     complete when the call returns.
 * Launch plans are cached per (B, Tq); at most 64 ragged ones per extractor lane (then they are rebuilt). */
int xvb_extractor_extract_ragged(xvb_extractor_t* h, const float* feats, const int32_t* offsets_host, int B, float* emb,
                                 void* stream);
int xvb_extractor_extract_ragged_shard_host(xvb_extractor_t* h, const float* feats_host, const int64_t* offsets_host,
                                            int64_t N, int batch, int64_t max_frames, float* emb_host, void* stream);
/* The batching policy of ragged shards, host only (no device needed): stable sort of the N utterances by length
 * (offsets_host (N+1) int64), then consecutive batches of <= `batch` utterances with B * round_up(max L, 32) <=
 * max_frames (<= 0: 262144); an utterance longer than that forms a batch of its own.  order_out (N): utterance index
 * per sorted position; batch k is order_out[batch_first_out[k] .. batch_first_out[k+1]), batch_first_out needs N+1
 * entries; *num_batches_out = number of batches.  Replaces the exact-length buckets of the batching CLIs. */
int xvb_ragged_plan(const int64_t* offsets_host, int64_t N, int batch, int64_t max_frames, int32_t* order_out,
                    int64_t* batch_first_out, int64_t* num_batches_out);

/* ---------------------------------------------------------------------------------------------
 * The embedding table of BASELINE configs[3] on every GPU of a node without a collective after extraction
 * (SURVEY 8e; replaces the `cat xvector.*.scp` of extract_xvectors_for_pytorch.sh:147-151 and the NCCL all-gather
 * of the plain path).  Each rank allocates its copy of the (world x n, D) table with xvb_ipc_alloc, exports it
 * (64-byte CUDA IPC handle, exchanged by the caller -- torch.distributed, MPI, a file), and maps its peers' copies
 * with xvb_ipc_open (NVLink peer access).  xvb_extractor_set_gather / xvb_ecapa_set_gather then make the shard calls
 * store every batch's embeddings into ALL copies at row0 + (row inside the shard) as soon as the batch's last layer
 * has produced them (xvb_scatter_rows on the batch's stream), overlapped with the following batches; the caller ends
 * the step with a barrier.  tables[k], k < ntables: base pointers valid in THIS process (own copy included);
 * ntables = 0 turns it off.  `emb` of the shard call still receives the rank's own rows.
 * ------------------------------------------------------------------------------------------- */
#define XVB_MAX_PEERS 16
#define XVB_IPC_HANDLE_BYTES 64
int xvb_ipc_alloc(void** ptr, size_t bytes);
int xvb_ipc_free(void* ptr);
int xvb_ipc_export(void* ptr, void* handle64);
int xvb_ipc_open(const void* handle64, void** ptr);
int xvb_ipc_close(void* ptr);
int xvb_scatter_rows(const float* src, int64_t rows, int D, float* const* tables, int ntables, int64_t row0, int64_t ld,
                     void* stream);
int xvb_extractor_set_gather(xvb_extractor_t* h, float* const* tables, int ntables, int64_t row0, int64_t ld);

/* Per-kernel timing with CUDA events recorded on the launching stream around every kernel of
 * the next extract calls.  xvb_extractor_kernel_times() waits for the last call and returns the
 * number of kernels n (<= max_n) and their durations in ms, in launch order: split, frame layers,
 * stats pooling, segment layers.  After xvb_extractor_extract_shard the events of ALL its batches are kept: per batch
 * the same kernel intervals followed by the interval to the next batch's first event. */
int xvb_extractor_set_profiling(xvb_extractor_t* h, int enable);
int xvb_extractor_kernel_times(xvb_extractor_t* h, float* ms_host, int max_n);
/* Fused pooling (default on): the last frame layer's epilogue reduces over time itself and the
 * (B,T,C_last) fp32 tensor is never written.  Off: last layer -> fp32 -> xvb_stats_pool. */
int xvb_extractor_set_fused_pooling(xvb_extractor_t* h, int enable);
/* Number of kernels the last extract call launched (bench.py's gpu_launches). */
int xvb_extractor_last_launches(const xvb_extractor_t* h);
/* Device pointer/pitch of a frame layer's fp32 output from the last call (debug/tests; only
 * the last frame layer keeps fp32), or the pooled statistics (layer = -1). */
const float* xvb_extractor_debug_f32(const xvb_extractor_t* h, int which);
void xvb_extractor_destroy(xvb_extractor_t* h);

/* ---------------------------------------------------------------------------------------------
 * Kaldi-compatible fbank / MFCC from raw waveforms (the feature step of the reference's online
 * path: KaldiFeature, pytorch/libs/egs/kaldi_features.py:69-135 -> torchaudio.compliance.kaldi
 * fbank/mfcc; C++ runtime: runtime/kaldifeat/csrc/feature-fbank.cc).  snip_edges framing, no
 * dither (the launchers force dither = 0 for extraction), no VTLN, window rounded up to 2^k.
 * Field names and defaults are torchaudio's / Kaldi's.  num_ceps > 0 selects MFCC.
 * ------------------------------------------------------------------------------------------- */
#define XVB_WINDOW_POVEY 0
#define XVB_WINDOW_HAMMING 1
#define XVB_WINDOW_HANNING 2
#define XVB_WINDOW_RECTANGULAR 3
#define XVB_WINDOW_BLACKMAN 4
typedef struct {
  float sample_frequency, frame_length_ms, frame_shift_ms, preemphasis_coefficient, low_freq, high_freq,
      energy_floor, cepstral_lifter, blackman_coeff;
  int num_mel_bins, num_ceps, use_energy, raw_energy, remove_dc_offset, use_log_fbank, use_power, htk_compat,
      window_type;
} xvb_fbank_opts_t;
typedef struct xvb_fbank xvb_fbank_t;
void xvb_fbank_default_opts(xvb_fbank_opts_t* opts);
/* Builds window / twiddle / mel / DCT tables (double precision, stored fp32) on the current device. */
int xvb_fbank_create(xvb_fbank_t** out, const xvb_fbank_opts_t* opts);
int xvb_fbank_dim(const xvb_fbank_t* h);                            /* columns of the feature matrix */
int64_t xvb_fbank_num_frames(const xvb_fbank_t* h, int64_t num_samples); /* 1 + (n - window) / shift, or 0 */
/* wave: all utterances back to back (device, fp32, Kaldi i.e. int16-range scale if the model was
 * trained that way); sample_offsets (U+1) int64 and frame_offsets (U+1) int32 on the device, with
 * frame_offsets[u+1]-frame_offsets[u] = xvb_fbank_num_frames(len_u); feats (total_frames, dim). */
int xvb_fbank_compute(xvb_fbank_t* h, const float* wave, const int64_t* sample_offsets, const int32_t* frame_offsets,
                      int num_utts, int64_t total_frames, float* feats, void* stream);
void xvb_fbank_destroy(xvb_fbank_t* h);

/* ---------------------------------------------------------------------------------------------
 * Whole-model extractor for ECAPA-TDNN (pytorch/model/ecapa_tdnn_xvector.py, ECAPA_TDNN.extract_embedding
 * :403-426; canonical c1024 parameters runEcapaXvector_online.py:221-263).  Layers are set by name with the
 * weights as the state_dict stores them (host fp32 (Cout, Cin, tot_context); eval BatchNorm folded to
 * scale/shift; flags XVB_RELU | XVB_BN):
 *   "layer1"; for L in 2..4: "layerL.bn1", "layerL.res0".."layerL.res6" (128 -> 128, [-d,0,d]),
 *   "layerL.bn2", "layerL.se1" (ReLU), "layerL.se2"; "mfa"; "att_x" = the first attention conv's columns
 *   over x with its ReLU + BatchNorm, "att_gs" = its columns over [mean | std] plus its bias (:179),
 *   "att2"; "fc2" with bn_stats folded into the weight (and fc2's own BatchNorm for position "near").
 * channels must be 1024 (Res2Net scale 8 x width 128, the chain kernel's shape).
 * ------------------------------------------------------------------------------------------- */
typedef struct xvb_ecapa xvb_ecapa_t;
int xvb_ecapa_create(xvb_ecapa_t** out, int feat_dim, int channels, int mfa_dim, int att_hidden, int embed_dim);
int xvb_ecapa_set_layer(xvb_ecapa_t* h, const char* name, int Cout, int Cin, const int* context_host, int ntaps,
                        const float* w_host, const float* bias_host, const float* bn_scale_host,
                        const float* bn_shift_host, int flags);
int xvb_ecapa_finalize(xvb_ecapa_t* h);
int xvb_ecapa_embed_dim(const xvb_ecapa_t* h);
int xvb_ecapa_feat_dim(const xvb_ecapa_t* h);
/* feats (B, T, feat_dim) fp32 on the device -> emb (B, embed_dim) fp32 on the device; asynchronous. */
int xvb_ecapa_extract(xvb_ecapa_t* h, const float* feats, int B, int T, float* emb, void* stream);
/* Same through host buffers (H2D of feats, D2H of emb inside; synchronises the stream). */
int xvb_ecapa_extract_host(xvb_ecapa_t* h, const float* feats_host, int B, int T, float* emb_host, void* stream);
/* Whole shard of N equal-length utterances in `batch`-utterance batches (extract_embeddings.py:73-83's loop as one
 * call): device-resident and asynchronous, or through pinned host buffers with the copies overlapped. */
int xvb_ecapa_extract_shard(xvb_ecapa_t* h, const float* feats, int64_t N, int T, int batch, float* emb, void* stream);
/* the replicated-table form of the shard calls, see xvb_extractor_set_gather */
int xvb_ecapa_set_gather(xvb_ecapa_t* h, float* const* tables, int ntables, int64_t row0, int64_t ld);
int xvb_ecapa_extract_shard_host(xvb_ecapa_t* h, const float* feats_host, int64_t N, int T, int batch, float* emb_host,
                                 void* stream);
int xvb_ecapa_last_launches(const xvb_ecapa_t* h);
/* "XVBE0001" model files: the named layers as handed to xvb_ecapa_set_layer. */
int xvb_ecapa_save(const xvb_ecapa_t* h, const char* path);
int xvb_ecapa_load(xvb_ecapa_t** out, const char* path);
void xvb_ecapa_destroy(xvb_ecapa_t* h);

/* Load a finalized extractor from an .xvbm model file (written by asv_subtools_b200.ops.Extractor.save:
 * the layers exactly as the reference's state_dict stores them, eval BatchNorm folded) -- what
 * torch::jit::load does for the reference's runtime (runtime/extractor/torch_asv_model.cc:8-17). */
int xvb_extractor_load(xvb_extractor_t** out, const char* path);
/* Feature dimension recorded in an .xvbm file (> 0), or a negative XVB_E* code.  Host only. */
int xvb_extractor_feat_dim(const char* path);

/* ---------------------------------------------------------------------------------------------
 * Kaldi ark/scp I/O on the host (no GPU needed): the byte formats of the reference's
 * pytorch/libs/support/kaldi_io.py -- read_key :148-163, _read_mat_binary :495-525 (FM/DM),
 * _read_compressed_mat :527-569 (CM), ascii matrices :478-493, write_vec_flt :367-399 (FV),
 * open_or_fd :43-73 (files, "-", "cmd |", "| cmd", "file:offset").
 * rspecifier: "ark:<src>" | "scp:<list>" | "<src>";  wspecifier: "ark:<dst>" | "ark,t:<dst>" |
 * "ark,scp:<ark file>,<scp file>".
 * ------------------------------------------------------------------------------------------- */
typedef struct xvb_ark_reader xvb_ark_reader_t;
typedef struct xvb_ark_writer xvb_ark_writer_t;
int xvb_ark_reader_open(xvb_ark_reader_t** out, const char* rspecifier);
/* Next matrix as fp32 row-major (DM is converted, CM decoded with the reference's fp32 steps).
 * Returns 1 (2 if the matrix was stored in double precision, which the reference's extractor rejects,
 * SURVEY Appendix B.1) and fills the outputs (owned by the reader, valid until the next call), 0 at the
 * end of the stream, a negative XVB_E* code on malformed input. */
int xvb_ark_reader_next(xvb_ark_reader_t* r, const char** key, int* rows, int* cols, const float** data);
void xvb_ark_reader_close(xvb_ark_reader_t* r);
int xvb_ark_writer_open(xvb_ark_writer_t** out, const char* wspecifier);
int xvb_ark_writer_put_vector(xvb_ark_writer_t* w, const char* key, const float* v, int dim);
/* Flushes and closes; fails if the stream or the pipe command failed. */
int xvb_ark_writer_close(xvb_ark_writer_t* w);

#ifdef __cplusplus
}
#endif
#endif /* XVB200_H_ */
