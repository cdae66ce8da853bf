/*
 * speecht5_b200 -- C ABI of the B200 (sm_100a) kernel library for the SpeechT5 forward/backward hot path.
 *
 * The reference (microsoft/SpeechT5, SpeechT5/speecht5/models/modules/*.py) has no FFI of its own: every device op is
 * a PyTorch library call made from the nn.Module forward()s. This header is the boundary a maintainer binds instead
 * (ctypes stub shown in INTEGRATION.md); each entry point names the reference code it replaces (file:line under
 * /root/reference/SpeechT5/).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); nothing is allocated or freed here;
 *   - `stream` is a cudaStream_t (pass torch.cuda.current_stream().cuda_stream);
 *   - return value 0 = ok, >0 = cudaError_t, <0 = library argument error; st5_last_error() gives the text
 *     (allocation failures contain the literal "out of memory", which fairseq/trainer.py:725 greps for);
 *   - `dtype`: ST5_F32 = 0, ST5_BF16 = 1 is the activation storage type; statistics, biases, LayerNorm/BatchNorm
 *     parameters, probabilities returned to the caller and all gradients of parameters are fp32;
 *   - dropout is counter based: one Philox4x32-7(seed, offset, i/8) call yields eight 16-bit lanes; element i is kept
 *     iff lane i%8 >= p*65536, i = linear index in the logical tensor (attention probabilities: row pitch rounded up
 *     to a multiple of 32 keys), so forward and backward regenerate identical masks without storing them.
 *     If bit 63 of `offset` is set, `seed` is the device address of a uint64 holding the seed (lets a captured CUDA
 *     graph draw fresh masks on every replay).
 */
#ifndef SPEECHT5_B200_H
#define SPEECHT5_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ST5_F32 0
#define ST5_BF16 1
#define ST5_ACT_NONE 0
#define ST5_ACT_RELU 1
#define ST5_ACT_GELU 2
#define ST5_ACT_TANH 3
#define ST5_ACT_GELU_TANH 4 /* tanh-form GELU on the MUFU unit: |error| <= 4.8e-4 vs the erf form; bf16 throughput mode */
#define ST5_ACT_GATE 5      /* actgrad_act only: actgrad_pre already holds the multiplier (written by ..._GATE below) */
#define ST5_ACT_GELU_TANH_GATE 6 /* act only (bf16 output, N % 8 == 0, c_pre != NULL): C = dropout(gelu_tanh(x)) and c_pre
                                    receives keep * scale * gelu_tanh'(x), the factor of the FFN's dH GEMM in backward */

int st5_version(void);
const char* st5_last_error(void);
/* sm_100a only: returns 0 when the current device can run the library, else a negative code. */
int st5_device_ok(void);

/* ------------------------------------------------------------------------------------------------- GEMM
 * D[z][m][n] = epi( alpha * sum_k A[z][m][k] * B[z][n][k] ), bf16 operands, fp32 accumulation in TMEM
 * (TMA + tcgen05.mma). Replaces every nn.Linear / torch.bmm / F.conv1d on the path:
 *   models/modules/multihead_attention.py:213-231 (q/k/v), :340 (QK^T), :389 (PV), :397 (out_proj);
 *   models/modules/transformer_layer.py:127-132, 385-391 (fc1/fc2);
 *   models/modules/speech_decoder_prenet.py:41-47,69-72; speech_decoder_postnet.py:31-32,39-51 (Conv1d as an
 *   overlapping-window GEMM over a zero-padded channels-last buffer); and their backward contractions.
 * Operand storage: *_mn = 0 -> row-major [rows][ld] with k contiguous; *_mn = 1 -> [K][ld] with the row index
 * contiguous (the operand is used transposed without a copy). ld / batch strides are in elements and must be
 * multiples of 8 (16 bytes); base pointers 16-byte aligned. Batch index z = b2 * nb1 + b1.
 * epi(v) = dropout(act(v + c_old*accumulate + bias[n] + bias2[m / bias2_rows][n])) + residual[m][n]; the value before
 * act() is also stored to c_pre when non-null.
 * accumulate: 0 = overwrite; 1 = c += (read-modify-write in the epilogue, FP32 c); 2 = c += as a TMA reduce-add at the
 * L2 (FP32 c, 16-byte aligned rows): batch entries may then SHARE one output (c_bs = 0) -- a contraction split over the
 * batch dimension (weight gradients: a_bs / b_bs step along K) -- and nothing reads c first. */
typedef struct st5_gemm_args {
  int32_t M, N, K, nb1, nb2;
  int32_t a_mn, b_mn, c_fp32, act, accumulate, bias2_rows;
  const void* a; int64_t a_ld, a_bs1, a_bs2;
  const void* b; int64_t b_ld, b_bs1, b_bs2;
  void* c; int64_t c_ld, c_bs1, c_bs2;
  void* c_pre;
  const float* bias;
  const float* bias2;
  const void* residual;
  float alpha;
  float drop_p;
  uint64_t drop_seed, drop_offset;
  const void* actgrad_pre;   /* optional: result *= act'(actgrad_pre[m][n]) (type actgrad_act), applied after the */
  int32_t actgrad_act;       /* dropout mask: fuses the activation backward into the dX GEMM of the next layer   */
} st5_gemm_args;
int st5_gemm_bf16(const st5_gemm_args* args, void* stream);

/* fp32 -> bf16 cast of a strided 2-D view. lo != NULL additionally writes the bf16 residual x - float(hi(x)), which
 * lets callers form hi*hi + hi*lo + lo*hi with three accumulate passes of st5_gemm_bf16 (fp32-grade "parity mode"). */
int st5_cast_bf16(const float* src, int64_t src_ld, void* hi, void* lo, int64_t dst_ld, int64_t rows, int64_t cols,
                  void* stream);

/* ------------------------------------------------------------------------------------------------- pre-nets
 * y[b,t,:] = dropout( (tokens ? E[tokens[b,t]] : x[b,t,:]) + alpha * pe[t,:] ).
 * text_encoder_prenet.py:36-45 (Embedding -> espnet ScaledPositionalEncoding), speech_decoder_prenet.py:52-67. */
int st5_posenc_fwd(const int64_t* tokens, const float* emb, const void* x, const float* pe, const float* alpha,
                   void* y, int dtype, int64_t B, int64_t T, int64_t C, float drop_p, uint64_t seed, uint64_t offset,
                   void* stream);
/* Backward: dx (same dtype, may be NULL), demb += (fp32 scatter-add, skipping padding_idx), dalpha += sum(dy*pe). */
int st5_posenc_bwd(const void* dy, const int64_t* tokens, int64_t padding_idx, const float* pe, void* dx, float* demb,
                   float* dalpha, int dtype, int64_t B, int64_t T, int64_t C, float drop_p, uint64_t seed,
                   uint64_t offset, void* stream);

/* ------------------------------------------------------------------------------------------------- LayerNorm
 * s = residual + dropout(x); y = LN(s) * gamma + beta. Saves s (for backward), mean and rstd.
 * transformer_layer.py:112-132 (post-LN encoder layer), :343-391 (decoder layer), encoder.py:226-227. */
int st5_ln_fwd(const void* x, const void* residual, const float* gamma, const float* beta, void* y, void* s_out,
               float* mean, float* rstd, int dtype, int64_t rows, int64_t C, float eps, float drop_p, uint64_t seed,
               uint64_t offset, void* stream);
/* Same with an fp32 RESIDUAL STREAM next to the bf16 activations (throughput mode): residual_f32 (may be NULL) replaces
 * `residual` as the addend, y_f32 (may be NULL) receives the un-rounded output. The GEMMs keep reading the bf16 `y`; the
 * next block's residual add reads y_f32, so the post-LN stream of transformer_layer.py:112-132 / :343-391 is never
 * rounded to bf16 between layers (the reference keeps it in fp32 on the CPU path / fp16 storage + fp32 LayerNorm on GPU). */
int st5_ln_fwd_stream(const void* x, const void* residual, const float* residual_f32, const float* gamma,
                      const float* beta, void* y, float* y_f32, void* s_out, float* mean, float* rstd, int dtype,
                      int64_t rows, int64_t C, float eps, float drop_p, uint64_t seed, uint64_t offset, void* stream);
/* ds = LN backward wrt s; dx = dropout-backward(ds) (may alias / be NULL when drop_p == 0 and caller reuses ds);
 * dgamma/dbeta are accumulated (+=) in fp32. `dxsum` (may be NULL; fp32 [C], accumulated +=) receives the column sums
 * of dx (of ds when dx is NULL): in the post-LN tail y = LN(residual + dropout(W a + b)) that is the gradient of b, so
 * the bias gradient of out_proj / fc2 (transformer_layer.py:112-132) costs no launch of its own.
 * st5_ln_bwd_blocks is kept for ABI stability (returns 1; no scratch is needed). */
int64_t st5_ln_bwd_blocks(int64_t rows);
int st5_ln_bwd(const void* dy, const void* s, const float* mean, const float* rstd, const float* gamma, void* ds,
               void* dx, float* dgamma, float* dbeta, float* dxsum, int dtype, int64_t rows, int64_t C, float drop_p,
               uint64_t seed, uint64_t offset, void* stream);

/* HiFi-GAN operand staging (SpeechUT/fairseq/fairseq/models/text_to_speech/hifigan.py:70-100, 154-170: F.leaky_relu
 * before every convolution): out[b][m][:] = leaky_relu(x[b][ph + d*m - pad][:], slope) for source frames inside [0, T),
 * zeros outside -- the zero-padded (d = 1) or de-interleaved (phase ph of dilation d) bf16 operand of the window GEMM in
 * one pass. x [B, T, C], out [B, n_in, C], C a multiple of 8; slope = 1 copies. */
int st5_lrelu_pad(const void* x, void* out, int64_t B, int64_t T, int64_t C, int64_t n_in, int32_t d, int32_t ph,
                  int32_t pad, float slope, void* stream);

/* y = dropout(x) (also its own backward when applied to the gradient). fairseq/modules/fairseq_dropout.py:23-37
 * (F.dropout semantics: keep with probability 1-p, scale by 1/(1-p)); mask = the counter-based generator above. */
int st5_dropout(const void* x, void* y, int dtype, int64_t n, float drop_p, uint64_t seed, uint64_t offset,
                void* stream);
/* y = act(x), stand-alone: the GELU behind the per-frame LayerNorm of layers 1..6 of the "layer_norm" waveform
 * extractor (speech_encoder_prenet.py:308-318). x, y 16-byte aligned. */
int st5_act_fwd(const void* x, void* y, int dtype, int act, int64_t n, void* stream);
/* dpre = dropout-backward(dy) * act'(pre): backward of activation_fn + activation dropout
 * (transformer_layer.py:127-129, speech_decoder_prenet.py:41-47 via espnet Prenet). */
int st5_act_bwd(const void* dy, const void* pre, void* dpre, int dtype, int act, int64_t n, float drop_p, uint64_t seed,
                uint64_t offset, void* stream);
/* out[g][n] (+)= sum_{m in group g} x[m][n], groups of `group_rows` consecutive rows: bias gradients of every
 * nn.Linear on the path (and, per utterance, of the x-vector term of speech_decoder_prenet.py:69-72); also the reduction
 * of split-K partial products. */
int st5_colsum(const void* x, int64_t ld, float* out, int dtype, int64_t rows, int64_t cols, int64_t group_rows,
               int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------- attention
 * multihead_attention.py:232-405. q/k/v are read in place from the fused projection outputs:
 *   element (b, t, h, c) of q lives at q[b * q_bs + t * q_ld + h * 64 + c] (same for k, v with their strides).
 * scores = scale * q.(k + pe_k[clamp(i-j,-maxpos,maxpos-1)+maxpos]) (RPE, encoder.py:40-59,239-246) ;
 * causal => j <= i; key_pad[b][j] != 0 => -inf; P = softmax_fp32; out = dropout(P) v.
 * probs (optional) receives P: [B,H,Tq,p_ld] in `probs_dtype` (fp32 when returned to the user: need_head_weights).
 * Head dim is fixed at 64 (Base and Large). */
typedef struct st5_attn_args {
  int32_t B, H, Tq, Tk, dtype, causal, maxpos, probs_dtype;
  const void* q; int64_t q_ld, q_bs;
  const void* k; int64_t k_ld, k_bs;
  const void* v; int64_t v_ld, v_bs;
  const uint8_t* key_pad;      /* [B][Tk] or NULL */
  const float* pe_k;           /* [2*maxpos][64] fp32 or NULL */
  void* out; int64_t o_ld, o_bs;
  void* probs; int64_t p_ld;   /* may be NULL in forward only */
  float scale, drop_p;
  uint64_t seed, offset;
  /* backward only */
  const void* dout;            /* same layout as out */
  const float* dprobs_ext;     /* optional external gradient wrt P, [B,H,Tq,p_ld] fp32 */
  float* ds;                   /* scratch [B,H,Tq,p_ld] fp32 */
  void* dq; void* dk; void* dv;/* same layouts as q, k, v */
  float* dpe_k;                /* [2*maxpos][64] fp32, accumulated (+=) */
  /* fused / flash forward only: > 0 = write `probs` for heads < probs_heads only (the caller reads no others: the
   * guided-attention loss, text_to_speech_loss.py:210-212); the rest of the buffer is left untouched */
  int32_t probs_heads;
} st5_attn_args;
int st5_attn_fwd(const st5_attn_args* args, void* stream);
int st5_attn_bwd(const st5_attn_args* args, void* stream);

/* Fused tcgen05 attention forward (bf16, Tk <= 320): QK^T -> masks -> softmax -> dropout -> PV in ONE launch, scores
 * resident in TMEM. Uses the q/k/v/out/probs/key_pad/scale/dropout fields of st5_attn_args exactly like st5_attn_fwd;
 * additionally writes lse[b][h][i] = log sum_j exp(scale*q_i.k_j) (may be NULL). probs (optional, only when the caller
 * wants them: need_head_weights) receives the undropped normalised probabilities in probs_dtype.
 * What the backward pass reads back (both optional, but together): psave [B,H,Tq,p_ld] BF16 = exp(s - rowmax), NOT
 * normalised, with the SIGN BIT set on elements dropout removed (probabilities are non-negative; a dropped zero is -0),
 * and inv_l [B,H,Tq] = 1 / rowsum. p_ld must be a multiple of 8, psave 16-byte aligned. out_f32 (optional)
 * [B,Tq,H*64] FP32 receives the un-rounded output: the backward's row constant delta = dO.O is the subtrahend of a
 * cancelling difference (dS = P (dP - delta)) and must not carry the BF16 rounding of `out`.
 * Relative positions (encoder.py:239-246): pe_k != NULL selects the skewed-bias variant; here pe_k must point to a
 * BF16 copy of the [2*maxpos][64] table, and Tq, Tk <= maxpos <= 160 (clamp(i-j) never clips), no causal mask. */
int st5_attn_fused_fwd(const st5_attn_args* args, float* lse, void* psave, float* inv_l, float* out_f32, void* stream);
/* Streaming ("flash") tcgen05 attention forward for ANY Tq / Tk (bf16): 128-key blocks, the row maximum is made final
 * in a first sweep over the key blocks (scores only), a second sweep computes exp / dropout / P V with the output
 * accumulating in TMEM, a third one (only when args->probs != NULL, which must then be FP32) writes the normalised
 * probabilities. Same arguments, outputs and psave / inv_l / out_f32 contract as st5_attn_fused_fwd, so
 * st5_attn_fused_bwd is its backward. Relative positions: pe_k = BF16 copy of the [2*maxpos][64] table, any Tq / Tk --
 * clamp(i - j, -maxpos, maxpos - 1) clips as encoder.py:40-59 does; no causal mask together with pe_k. */
int st5_attn_flash_fwd(const st5_attn_args* args, float* lse, void* psave, float* inv_l, float* out_f32, void* stream);
/* Fused tcgen05 attention backward (multihead_attention.py:340-389 differentiated). psave / inv_l are what
 * st5_attn_fused_fwd wrote: probabilities and dropout decisions are read back instead of recomputed (no exponential, no
 * Philox), so every step needs one score-sized MMA (dP = dO V^T) and the kernel double buffers dP, the dropout(P)/dS
 * operand tiles, dQ and the Q/dO tiles. Reads q/k/v, out (forward result), dout and drop_p; optional dprobs_ext (then
 * args->probs must be the FP32 probabilities the forward returned); writes dq/dk/dv (same layouts as q/k/v).
 * ext_heads > 0: dprobs_ext is known to be zero for heads >= ext_heads (the guided-attention loss reads the first two
 * heads of every layer, text_to_speech_loss.py:210-212) -- those heads skip its loads. out_f32 (optional): what the
 * forward wrote there. Scratch: delta [B*H*Tq] floats, dq_acc [B*Tq*H*64] floats.
 * Relative positions (pe_k != NULL): args->ds additionally receives dS as BF16 [B,H,Tq,p_ld] for st5_attn_dqp_scatter
 * and the two table GEMMs; dq then holds only the q.k part of the gradient. */
int st5_attn_fused_bwd(const st5_attn_args* args, const void* psave, const float* inv_l, const float* out_f32,
                       float* delta, float* dq_acc, int32_t ext_heads, void* stream);

/* Tensor-core (bf16) attention path: the contractions run on st5_gemm_bf16 (batched over heads and utterances, q/k/v
 * read in place from the fused projection buffers); these three row kernels are the non-GEMM steps between them.
 * Row index = (b*H + h)*Tq + i everywhere; row pitch p_ld (multiple of 8, >= Tk); dropout indices as in st5_attn_fwd.
 *   softmax_fwd: P = softmax(S + QP[i][clamp(i-j)+maxpos] + masks); writes P (bf16), optionally fp32 probabilities
 *                (may alias s) and dropout(P) (bf16). s already holds scale*q.k, qp (optional) scale*q.pe_k^T [rows][2*maxpos].
 *   ds:          dS = P * (dropout_bwd(dP) + dP_ext - rowsum(P * (...))) (bf16); optionally re-emits dropout(P).
 *   dqp_scatter: dQP[row][r] = sum over keys j with clamp(i-j)+maxpos == r of dS[row][j]  (gradient wrt QP); output rows
 *                in the order of dS ((b, h, i)), or with h_major != 0 as (h, b, i). */
int st5_attn_softmax_fwd(const float* s, const float* qp, int64_t qp_ld, const uint8_t* key_pad, void* p_bf16,
                         float* probs_f32, void* pdrop_bf16, int32_t B, int32_t H, int32_t Tq, int32_t Tk, int64_t p_ld,
                         int32_t causal, int32_t maxpos, float drop_p, uint64_t seed, uint64_t offset, void* stream);
int st5_attn_ds(const void* p_bf16, const float* dp, const float* dp_ext, void* ds_bf16, void* pdrop_bf16, int32_t B,
                int32_t H, int32_t Tq, int32_t Tk, int64_t p_ld, float drop_p, uint64_t seed, uint64_t offset,
                void* stream);
int st5_attn_dqp_scatter(const void* ds_bf16, void* dqp_bf16, int32_t B, int32_t H, int32_t Tq, int32_t Tk,
                         int64_t p_ld, int32_t maxpos, int32_t h_major, void* stream);

/* ------------------------------------------------------------------------------------------------- BatchNorm1d
 * espnet Tacotron2 Postnet block (speech_decoder_postnet.py:39-51): y = dropout(tanh?(BN(x))) on channels-last
 * rows [rows][C]; training statistics over all rows (padded frames included, as in the reference). */
int st5_bn_fwd(const void* x, int64_t x_ld, const float* gamma, const float* beta, float* running_mean,
               float* running_var, float* save_mean, float* save_rstd, void* y, int64_t y_ld, void* y_pre, int dtype,
               int64_t rows, int64_t C, int training, float momentum, float eps, int act, float drop_p, uint64_t seed,
               uint64_t offset, float* scratch, void* stream);
int st5_bn_bwd(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, const void* y_pre, const float* gamma,
               const float* save_mean, const float* save_rstd, void* dx, int64_t dx_ld, float* dgamma, float* dbeta,
               int dtype, int64_t rows, int64_t C, int act, float drop_p, uint64_t seed, uint64_t offset,
               float* scratch, void* stream);

/* ------------------------------------------------------------------------------------------------- waveform front end
 * (speech-input branch, SURVEY section 8a row 2)
 * Layer 0 of ConvFeatureExtractionModel in mode "default" (speech_encoder_prenet.py:290-327,349-354): Conv1d(1 -> C, K
 * taps, `stride`, no bias) + Fp32GroupNorm(C groups: statistics per utterance and channel over time) + GELU
 * (fairseq/modules/gelu.py:24), fused. wave [B, n_samples] fp32; w [C, K]; y [B, T0, C] channels-last in `dtype`,
 * T0 = (n_samples - K) / stride + 1; mean / rstd [B, C] are saved for the backward. The convolution is recomputed from
 * the waveform in every pass, so the [B, T0, C] tensor is written once (forward) and dy read twice (backward).
 * ws: st5_conv0_ws_floats(...) floats of scratch. act: ST5_ACT_GELU or ST5_ACT_GELU_TANH. C <= 1024, K <= 16.
 * Backward: dw [C, K], dgamma [C], dbeta [C] are ACCUMULATED (+=); the input is the waveform: no input gradient. */
int64_t st5_conv0_ws_floats(int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride);
int st5_conv0_gn_gelu_fwd(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                          float* mean, float* rstd, float* ws, int32_t B, int64_t n_samples, int32_t C, int32_t K,
                          int32_t stride, float eps, int act, void* stream);
int st5_conv0_gn_gelu_bwd(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                          const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws,
                          int dtype, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride, int act,
                          void* stream);

/* Layer 0 in extractor mode "layer_norm" (t5_transformer_large, models/speecht5.py:1421; block builder
 * speech_encoder_prenet.py:308-318): Conv1d(1 -> C, K taps, `stride`, no bias) + Fp32LayerNorm over the C channels of
 * each frame + GELU, fused in ONE pass (a warp per frame). y [B, T0, C] channels-last in `dtype`; mean / rstd [B * T0]
 * are saved for the backward. C even, C <= 512, K <= 16. Backward: dw [C, K], dgamma [C], dbeta [C] are ACCUMULATED
 * (+=); ws: st5_conv0_ln_ws_floats(...) floats of scratch; no input gradient (the input is the waveform). */
int64_t st5_conv0_ln_ws_floats(int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride);
int st5_conv0_ln_gelu_fwd(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                          float* mean, float* rstd, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride,
                          float eps, int act, void* stream);
int st5_conv0_ln_gelu_bwd(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                          const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws,
                          int dtype, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride, int act,
                          void* stream);

/* ------------------------------------------------------------------------------------------------- CTC
 * (speech-input branch, SURVEY section 8a row 18)
 * Replaces F.log_softmax + F.ctc_loss(reduction="sum") of speech_to_text_loss.py:303-335 on the encoder's CTC head.
 * logits fp32, element (t, b, k) at t*ld_t + b*ld_b + k; targets: flat int64 labels, utterance b's at
 * targets[tgt_offsets[b] .. + target_lengths[b]); nll [B] receives the per-utterance negative log-likelihood (+inf for
 * an infeasible utterance, or 0 with zero_infinity); grad (optional, same addressing as logits) receives
 * d(sum_b nll_b)/d logits, zero for t >= input_lengths[b] and for infeasible utterances. S_max >= 2*max(target_lengths)+1
 * (<= 1024) is the scratch pitch; ws: st5_ctc_ws_floats(T, B, S_max) floats (row log-sum-exps, emission terms, alpha
 * and beta lattices). Three launches: row pass, the two recursions side by side in one CTA per utterance, gradient rows. */
int64_t st5_ctc_ws_floats(int32_t T, int32_t B, int32_t S_max);
int st5_ctc_loss(const float* logits, int64_t ld_t, int64_t ld_b, const int64_t* targets, const int64_t* tgt_offsets,
                 const int64_t* input_lengths, const int64_t* target_lengths, float* nll, float* grad, float* ws,
                 int32_t T, int32_t B, int32_t V, int32_t S_max, int32_t blank, int32_t zero_infinity, void* stream);

/* ------------------------------------------------------------------------------------------------- TTS criterion
 * The reductions of speecht5/criterions/text_to_speech_loss.py and their gradients (SURVEY section 8a row 17).
 * st5_tts_loss_fwd: Tacotron2Loss with use_masking (:217-345). after / before [B, L, D] fp32 contiguous, logits [B, L],
 * ys: element (b, l, c) at b*y_bs + l*D + c (the target tensor may be longer than L), labels: (b, l) at b*lab_bs + l,
 * olens int64 [B] (frames; the valid region of utterance b is l < olens[b] - olens[b] % r, and for r > 1 the stop label
 * of its last valid frame counts as 1, :161-166). out[0..2] = l1, l2, bce (means over valid frames, l1 / l2 also over D);
 * sums: scratch of st5_tts_loss_ws_floats(B, L) floats that st5_tts_loss_bwd reads back (sums[3] = number of valid
 * frames; the rest holds per-CTA partials, added in a fixed order: same inputs, same bits).
 * st5_tts_loss_bwd (gradient of text_to_speech_loss.py:288-330): g[3] = upstream gradients of (l1, l2, bce) in device memory; writes d_after, d_before [B, L, D] and
 * d_logits [B, L] everywhere (zeros outside the masks). */
int64_t st5_tts_loss_ws_floats(int32_t B, int32_t L);
int64_t st5_guided_attn_ws_floats(int32_t n_layers, int32_t B, int32_t heads, int32_t T_out);
int st5_tts_loss_fwd(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                     const float* labels, int64_t lab_bs, const int64_t* olens, int32_t B, int32_t L, int32_t D,
                     int32_t r, float pos_weight, float* sums, float* out, void* stream);
int st5_tts_loss_bwd(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                     const float* labels, int64_t lab_bs, const int64_t* olens, const float* sums, const float* g,
                     int32_t B, int32_t L, int32_t D, int32_t r, float pos_weight, float* d_after, float* d_before,
                     float* d_logits, void* stream);
/* GuidedMultiHeadAttentionLoss (text_to_speech_loss.py:370-427) over the first `heads` heads of n_layers (<= 8) returned cross-attention
 * probability tensors att[i] = [B, H, T_out, p_ld] fp32: out[0] = alpha * sum_valid W * A / (sum_b il_b * ol_b * heads *
 * n_layers), W = 1 - exp(-(t_in / il - t_out / ol)^2 / (2 sigma^2)), ol = olens[b] / r, il = ilens[b]. gsum: scratch of
 * st5_guided_attn_ws_floats(n_layers, B, heads, T_out) floats (fixed-order partial sums)
 * read back by the backward, which writes datt[i] (same layout) = g[0] * d out / d att on heads < `heads`; the other
 * heads are cleared only with zero_rest != 0 (st5_attn_fused_bwd with ext_heads never reads them). */
int st5_guided_attn_fwd(const float* const* att, int32_t n_layers, int32_t B, int32_t H, int32_t heads, int32_t T_out,
                        int32_t T_in, int64_t p_ld, const int64_t* ilens, const int64_t* olens, int32_t r, float sigma,
                        float alpha, float* gsum, float* out, void* stream);
int st5_guided_attn_bwd(float* const* datt, int32_t n_layers, int32_t B, int32_t H, int32_t heads, int32_t T_out,
                        int32_t T_in, int64_t p_ld, const int64_t* ilens, const int64_t* olens, int32_t r, float sigma,
                        float alpha, const float* gsum, const float* g, int32_t zero_rest, void* stream);

/* ------------------------------------------------------------------------------------------------- beam search
 * Joint CTC/attention beam search (speecht5/sequence_generator.py:273-284, :370-418). All values fp32; the sentinel is
 * the reference's finite logzero = -1e10. x: CTC log-probabilities, element (b, t, v) at b*ld_b + t*ld_t + v
 * (ld_t >= V); t_valid [B] int64: valid frames T_b of each utterance (rows t >= T_b are never read). T <= 1500,
 * K <= 256; outside these limits the call fails (code -2) without a launch.
 *
 * st5_ctc_prefix_init replaces CTCPrefixScore.initial_state (espnet ctc_prefix_score.py, numpy on the host): r [B, T, 2]
 * with r[b, t, 0] = logzero and r[b, t, 1] = sum_{tau <= t} x[b, tau, blank] for t < T_b (logzero beyond). */
int st5_ctc_prefix_init(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* t_valid, float* r, int32_t B,
                        int32_t T, int32_t V, int32_t blank, void* stream);
/* st5_ctc_prefix_score replaces the per-hypothesis CTCPrefixScore.__call__ loop of sequence_generator.py:379-391 (one
 * host call per hypothesis, each looping over every frame): H hypotheses x K candidate labels in one launch, a CTA per
 * hypothesis, a thread per candidate. Per hypothesis h: utt[h] (its utterance), r_prev [H, T, 2] (its state), last[h]
 * (its last label), out_len[h] (prefix length without the leading eos); candidates cs [H, K] int64. Writes
 * log_psi [H, K] and the candidate states r [H, T, 2, K] (frame-major, candidates innermost). Semantics of the
 * reference scorer: phi = r_prev_b where the candidate repeats the last label; the recursion starts at frame
 * max(out_len, 1); an eos candidate gets logaddexp(r_prev_n, r_prev_b) at frame T_b - 1, a blank candidate logzero;
 * out_len >= T_b leaves the recursion empty; rows the reference leaves uninitialised are logzero. */
int st5_ctc_prefix_score(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* utt, const float* r_prev,
                         const int64_t* last, const int64_t* out_len, const int64_t* cs, const int64_t* t_valid,
                         float* log_psi, float* r, int32_t H, int32_t T, int32_t K, int32_t V, int32_t blank,
                         int32_t eos, void* stream);
/* st5_beam_gather_rows replaces the per-layer index_select of the decoder's incremental state on a beam reorder
 * (sequence_generator.py:358, reorder_incremental_state): for every layer l < n_layers (<= 32) and hypothesis h < H,
 * copies the first n_rows * row_bytes bytes of src[l] + parent[h] * src_bs to dst[l] + h * dst_bs. src / dst: host
 * arrays of device pointers (two distinct buffer sets: no in-place reorder). row_bytes, src_bs, dst_bs and every
 * pointer 16-byte aligned. Only the rows already written are copied, not the whole max_len span. */
int st5_beam_gather_rows(const void* const* src, void* const* dst, const int64_t* parent, int32_t n_layers, int32_t H,
                         int32_t n_rows, int64_t row_bytes, int64_t src_bs, int64_t dst_bs, void* stream);

/* ------------------------------------------------------------------------------------------------- optimizer
 * Replaces fairseq/optim/adam.py + fp16_optimizer.py:106-218 on a flat fp32 parameter buffer: one pass applies the
 * gradient scale (grad_mul x clip coefficient max_norm / (norm + 1e-6) capped at 1: fairseq/utils.py clip_grad_norm_,
 * fairseq/trainer.py:796-826), Adam as fairseq/optim/adam.py:Adam.step writes it (denominator sqrt(v) + eps, step size
 * lr * sqrt(1 - b2^t) / (1 - b1^t), weight decay p -= wd * lr * p) and refreshes the bf16 shadow copy the GEMMs read.
 * st5_sumsq accumulates sum(x^2) (the squared gradient norm) into *out. lr_dev / step_dev: device-resident schedule
 * state so that a captured CUDA graph stays valid across updates. */
int st5_sumsq(const float* x, int64_t n, float* out /* 1 float, accumulated */, void* stream);
int st5_adam_step(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int64_t step, const float* grad_norm_sq, float max_norm,
                  float grad_mul, const float* lr_dev /* optional device lr */,
                  const int64_t* step_dev /* optional device step counter */, void* stream);

#ifdef __cplusplus
}
#endif
#endif
