// C-ABI entry points (include/speecht5_b200.h). Pure argument marshalling; kernels live in the other .cu files.
#include "../../include/speecht5_b200.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace st5 {
static thread_local char g_err[512] = "";
int set_error(int code, const char* where) {
  if (code == 0) return 0;
  if (code > 0) {
    const char* s = cudaGetErrorString((cudaError_t)code);
    if (code == (int)cudaErrorMemoryAllocation)
      snprintf(g_err, sizeof(g_err), "%s: CUDA out of memory (%s)", where, s);
    else
      snprintf(g_err, sizeof(g_err), "%s: CUDA error %d (%s)", where, code, s);
    cudaGetLastError();
  } else {
    snprintf(g_err, sizeof(g_err), "%s: invalid argument (code %d)", where, code);
  }
  return code;
}
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("ST5_PDL");
    return e == nullptr || atoi(e) != 0;
  }();
  return on;
}
}  // namespace st5

using namespace st5;

extern "C" {

int st5_version(void) { return 100; }
const char* st5_last_error(void) { return g_err; }

int st5_device_ok(void) {
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess) return set_error(-1, "st5_device_ok");
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return set_error(-1, "st5_device_ok");
  if (prop.major != 10) return set_error(-2, "st5_device_ok: library is built for sm_100a only");
  return 0;
}

int st5_gemm_bf16(const st5_gemm_args* a, void* stream) {
  GemmDesc g;
  g.M = a->M; g.N = a->N; g.K = a->K; g.nb1 = a->nb1; g.nb2 = a->nb2;
  g.A = a->a; g.a_mn = a->a_mn; g.a_ld = a->a_ld; g.a_bs1 = a->a_bs1; g.a_bs2 = a->a_bs2;
  g.B = a->b; g.b_mn = a->b_mn; g.b_ld = a->b_ld; g.b_bs1 = a->b_bs1; g.b_bs2 = a->b_bs2;
  g.C = a->c; g.c_fp32 = a->c_fp32; g.c_ld = a->c_ld; g.c_bs1 = a->c_bs1; g.c_bs2 = a->c_bs2;
  g.C_pre = a->c_pre; g.bias = a->bias; g.bias2 = a->bias2; g.bias2_rows = a->bias2_rows;
  g.residual = a->residual; g.act = a->act; g.alpha = a->alpha; g.accumulate = a->accumulate;
  g.drop_p = a->drop_p; g.drop_seed = a->drop_seed; g.drop_offset = a->drop_offset;
  g.ag_pre = a->actgrad_pre; g.ag_act = a->actgrad_act;
  return set_error(gemm_launch(g, (cudaStream_t)stream), "st5_gemm_bf16");
}

int st5_cast_bf16(const float* src, int64_t src_ld, void* hi, void* lo, int64_t dst_ld, int64_t rows, int64_t cols,
                  void* stream) {
  return set_error(cast_bf16_launch(src, src_ld, hi, lo, dst_ld, rows, cols, (cudaStream_t)stream), "st5_cast_bf16");
}

int st5_posenc_fwd(const int64_t* tokens, const float* emb, const void* x, const float* pe, const float* alpha,
                   void* y, int dtype, int64_t B, int64_t T, int64_t C, float drop_p, uint64_t seed, uint64_t offset,
                   void* stream) {
  return set_error(posenc_fwd_launch(tokens, emb, x, pe, alpha, y, dtype, B, T, C, drop_p, seed, offset,
                                     (cudaStream_t)stream),
                   "st5_posenc_fwd");
}
int st5_posenc_bwd(const void* dy, const int64_t* tokens, int64_t padding_idx, const float* pe, void* dx, float* demb,
                   float* dalpha, int dtype, int64_t B, int64_t T, int64_t C, float drop_p, uint64_t seed,
                   uint64_t offset, void* stream) {
  return set_error(posenc_bwd_launch(dy, tokens, padding_idx, pe, dx, demb, dalpha, dtype, B, T, C, drop_p, seed,
                                     offset, (cudaStream_t)stream),
                   "st5_posenc_bwd");
}

int st5_ln_fwd(const void* x, const void* residual, const float* gamma, const float* beta, void* y, void* s_out,
               float* mean, float* rstd, int dtype, int64_t rows, int64_t C, float eps, float drop_p, uint64_t seed,
               uint64_t offset, void* stream) {
  return set_error(ln_fwd_launch(x, residual, nullptr, gamma, beta, y, nullptr, s_out, mean, rstd, dtype, rows, C, eps,
                                 drop_p, seed, offset, (cudaStream_t)stream),
                   "st5_ln_fwd");
}
int st5_ln_fwd_stream(const void* x, const void* residual, const float* residual_f32, const float* gamma,
                      const float* beta, void* y, float* y_f32, void* s_out, float* mean, float* rstd, int dtype,
                      int64_t rows, int64_t C, float eps, float drop_p, uint64_t seed, uint64_t offset, void* stream) {
  return set_error(ln_fwd_launch(x, residual, residual_f32, gamma, beta, y, y_f32, s_out, mean, rstd, dtype, rows, C,
                                 eps, drop_p, seed, offset, (cudaStream_t)stream),
                   "st5_ln_fwd_stream");
}
int64_t st5_ln_bwd_blocks(int64_t rows) { return ln_bwd_blocks(rows); }
int st5_ln_bwd(const void* dy, const void* s, const float* mean, const float* rstd, const float* gamma, void* ds,
               void* dx, float* dgamma, float* dbeta, float* dxsum, int dtype, int64_t rows, int64_t C, float drop_p,
               uint64_t seed, uint64_t offset, void* stream) {
  return set_error(ln_bwd_launch(dy, s, mean, rstd, gamma, ds, dx, dgamma, dbeta, dxsum, dtype, rows, C, drop_p,
                                 seed, offset, (cudaStream_t)stream),
                   "st5_ln_bwd");
}

int st5_lrelu_pad(const void* x, void* out, int64_t B, int64_t T, int64_t C, int64_t n_in, int32_t d, int32_t ph,
                  int32_t pad, float slope, void* stream) {
  return set_error(lrelu_pad_launch(x, out, B, T, C, n_in, d, ph, pad, slope, (cudaStream_t)stream), "st5_lrelu_pad");
}

int st5_dropout(const void* x, void* y, int dtype, int64_t n, float drop_p, uint64_t seed, uint64_t offset,
                void* stream) {
  return set_error(dropout_launch(x, y, dtype, n, drop_p, seed, offset, (cudaStream_t)stream), "st5_dropout");
}
int st5_act_bwd(const void* dy, const void* pre, void* dpre, int dtype, int act, int64_t n, float drop_p, uint64_t seed,
                uint64_t offset, void* stream) {
  return set_error(act_bwd_launch(dy, pre, dpre, dtype, act, n, drop_p, seed, offset, (cudaStream_t)stream),
                   "st5_act_bwd");
}
int st5_colsum(const void* x, int64_t ld, float* out, int dtype, int64_t rows, int64_t cols, int64_t group_rows,
               int accumulate, void* stream) {
  return set_error(colsum_launch(x, ld, out, dtype, rows, cols, group_rows, accumulate, (cudaStream_t)stream),
                   "st5_colsum");
}

int st5_attn_fwd(const st5_attn_args* a, void* stream) {
  return set_error(attn_fwd_launch(*a, (cudaStream_t)stream), "st5_attn_fwd");
}
int st5_attn_bwd(const st5_attn_args* a, void* stream) {
  return set_error(attn_bwd_launch(*a, (cudaStream_t)stream), "st5_attn_bwd");
}

int st5_bn_fwd(const void* x, int64_t x_ld, const float* gamma, const float* beta, float* running_mean,
               float* running_var, float* save_mean, float* save_rstd, void* y, int64_t y_ld, void* y_pre, int dtype,
               int64_t rows, int64_t C, int training, float momentum, float eps, int act, float drop_p, uint64_t seed,
               uint64_t offset, float* scratch, void* stream) {
  return set_error(bn_fwd_launch(x, x_ld, gamma, beta, running_mean, running_var, save_mean, save_rstd, y, y_ld, y_pre,
                                 dtype, rows, C, training, momentum, eps, act, drop_p, seed, offset, scratch,
                                 (cudaStream_t)stream),
                   "st5_bn_fwd");
}
int st5_bn_bwd(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, const void* y_pre, const float* gamma,
               const float* save_mean, const float* save_rstd, void* dx, int64_t dx_ld, float* dgamma, float* dbeta,
               int dtype, int64_t rows, int64_t C, int act, float drop_p, uint64_t seed, uint64_t offset,
               float* scratch, void* stream) {
  return set_error(bn_bwd_launch(dy, dy_ld, x, x_ld, y_pre, gamma, save_mean, save_rstd, dx, dx_ld, dgamma, dbeta,
                                 dtype, rows, C, act, drop_p, seed, offset, scratch, (cudaStream_t)stream),
                   "st5_bn_bwd");
}

int64_t st5_conv0_ln_ws_floats(int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride) {
  return conv0_ln_ws_floats(B, n_samples, C, K, stride);
}
int st5_conv0_ln_gelu_fwd(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                          float* mean, float* rstd, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride,
                          float eps, int act, void* stream) {
  return set_error(conv0_ln_fwd_launch(wave, w, gamma, beta, y, dtype, mean, rstd, B, n_samples, C, K, stride, eps, act,
                                       (cudaStream_t)stream),
                   "st5_conv0_ln_gelu_fwd");
}
int st5_conv0_ln_gelu_bwd(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                          const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws,
                          int dtype, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride, int act,
                          void* stream) {
  return set_error(conv0_ln_bwd_launch(dy, wave, w, gamma, beta, mean, rstd, dw, dgamma, dbeta, ws, dtype, B, n_samples,
                                       C, K, stride, act, (cudaStream_t)stream),
                   "st5_conv0_ln_gelu_bwd");
}
int st5_act_fwd(const void* x, void* y, int dtype, int act, int64_t n, void* stream) {
  return set_error(act_fwd_launch(x, y, dtype, act, n, (cudaStream_t)stream), "st5_act_fwd");
}

int64_t st5_conv0_ws_floats(int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride) {
  return conv0_ws_floats(B, n_samples, C, K, stride);
}
int st5_conv0_gn_gelu_fwd(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                          float* mean, float* rstd, float* ws, int32_t B, int64_t n_samples, int32_t C, int32_t K,
                          int32_t stride, float eps, int act, void* stream) {
  return set_error(conv0_fwd_launch(wave, w, gamma, beta, y, dtype, mean, rstd, ws, B, n_samples, C, K, stride, eps, act,
                                    (cudaStream_t)stream),
                   "st5_conv0_gn_gelu_fwd");
}
int st5_conv0_gn_gelu_bwd(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                          const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws,
                          int dtype, int32_t B, int64_t n_samples, int32_t C, int32_t K, int32_t stride, int act,
                          void* stream) {
  return set_error(conv0_bwd_launch(dy, wave, w, gamma, beta, mean, rstd, dw, dgamma, dbeta, ws, dtype, B, n_samples, C,
                                    K, stride, act, (cudaStream_t)stream),
                   "st5_conv0_gn_gelu_bwd");
}

int64_t st5_tts_loss_ws_floats(int32_t B, int32_t L) { return 4 + 4 * tts_loss_blocks(B, L); }
int64_t st5_guided_attn_ws_floats(int32_t n_layers, int32_t B, int32_t heads, int32_t T_out) {
  return 2 + guided_attn_blocks(n_layers, B, heads, T_out);
}
int st5_tts_loss_fwd(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                     const float* labels, int64_t lab_bs, const int64_t* olens, int32_t B, int32_t L, int32_t D,
                     int32_t r, float pos_weight, float* sums, float* out, void* stream) {
  return set_error(tts_loss_fwd_launch(after, before, logits, ys, y_bs, labels, lab_bs, olens, B, L, D, r, pos_weight, sums,
                                       out, (cudaStream_t)stream),
                   "st5_tts_loss_fwd");
}
int st5_tts_loss_bwd(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                     const float* labels, int64_t lab_bs, const int64_t* olens, const float* sums, const float* g,
                     int32_t B, int32_t L, int32_t D, int32_t r, float pos_weight, float* d_after, float* d_before,
                     float* d_logits, void* stream) {
  return set_error(tts_loss_bwd_launch(after, before, logits, ys, y_bs, labels, lab_bs, olens, sums, g, B, L, D, r,
                                       pos_weight, d_after, d_before, d_logits, (cudaStream_t)stream),
                   "st5_tts_loss_bwd");
}
int st5_guided_attn_fwd(const float* const* att, int32_t n_layers, int32_t B, int32_t H, int32_t heads, int32_t T_out,
                        int32_t T_in, int64_t p_ld, const int64_t* ilens, const int64_t* olens, int32_t r, float sigma,
                        float alpha, float* gsum, float* out, void* stream) {
  return set_error(guided_attn_fwd_launch(att, n_layers, B, H, heads, T_out, T_in, p_ld, ilens, olens, r, sigma, alpha,
                                          gsum, out, (cudaStream_t)stream),
                   "st5_guided_attn_fwd");
}
int st5_guided_attn_bwd(float* const* datt, int32_t n_layers, int32_t B, int32_t H, int32_t heads, int32_t T_out,
                        int32_t T_in, int64_t p_ld, const int64_t* ilens, const int64_t* olens, int32_t r, float sigma,
                        float alpha, const float* gsum, const float* g, int32_t zero_rest, void* stream) {
  return set_error(guided_attn_bwd_launch(datt, n_layers, B, H, heads, T_out, T_in, p_ld, ilens, olens, r, sigma, alpha,
                                          gsum, g, zero_rest, (cudaStream_t)stream),
                   "st5_guided_attn_bwd");
}

int64_t st5_ctc_ws_floats(int32_t T, int32_t B, int32_t S_max) { return ctc_ws_floats(T, B, S_max); }
int st5_ctc_loss(const float* logits, int64_t ld_t, int64_t ld_b, const int64_t* targets, const int64_t* tgt_offsets,
                 const int64_t* input_lengths, const int64_t* target_lengths, float* nll, float* grad, float* ws,
                 int32_t T, int32_t B, int32_t V, int32_t S_max, int32_t blank, int32_t zero_infinity, void* stream) {
  return set_error(ctc_loss_launch(logits, ld_t, ld_b, targets, tgt_offsets, input_lengths, target_lengths, nll, grad,
                                   ws, T, B, V, S_max, blank, zero_infinity, (cudaStream_t)stream),
                   "st5_ctc_loss");
}

int st5_ctc_prefix_init(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* t_valid, float* r, int32_t B,
                        int32_t T, int32_t V, int32_t blank, void* stream) {
  return set_error(ctc_prefix_init_launch(x, ld_b, ld_t, t_valid, r, B, T, V, blank, (cudaStream_t)stream),
                   "st5_ctc_prefix_init");
}
int st5_ctc_prefix_score(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* utt, const float* r_prev,
                         const int64_t* last, const int64_t* out_len, const int64_t* cs, const int64_t* t_valid,
                         float* log_psi, float* r, int32_t H, int32_t T, int32_t K, int32_t V, int32_t blank,
                         int32_t eos, void* stream) {
  return set_error(ctc_prefix_score_launch(x, ld_b, ld_t, utt, r_prev, last, out_len, cs, t_valid, log_psi, r, H, T, K,
                                           V, blank, eos, (cudaStream_t)stream),
                   "st5_ctc_prefix_score");
}
int st5_beam_gather_rows(const void* const* src, void* const* dst, const int64_t* parent, int32_t n_layers, int32_t H,
                         int32_t n_rows, int64_t row_bytes, int64_t src_bs, int64_t dst_bs, void* stream) {
  return set_error(beam_gather_rows_launch(src, dst, parent, n_layers, H, n_rows, row_bytes, src_bs, dst_bs,
                                           (cudaStream_t)stream),
                   "st5_beam_gather_rows");
}

int st5_sumsq(const float* x, int64_t n, float* out, void* stream) {
  return set_error(sumsq_launch(x, n, out, (cudaStream_t)stream), "st5_sumsq");
}
int st5_adam_step(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int64_t step, const float* grad_norm_sq, float max_norm,
                  float grad_mul, const float* lr_dev, const int64_t* step_dev, void* stream) {
  return set_error(adam_launch(p, g, m, v, p_bf16, n, lr, beta1, beta2, eps, weight_decay, step, grad_norm_sq, max_norm,
                               grad_mul, lr_dev, step_dev, (cudaStream_t)stream),
                   "st5_adam_step");
}

}  // extern "C"
