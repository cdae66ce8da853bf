// Launcher declarations for the non-GEMM kernels (definitions in elementwise.cu, norm.cu, attention.cu, optim.cu).
#pragma once
#include "../../include/speecht5_b200.h"
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace st5 {

// activation storage accessors
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16(v); }

// Programmatic dependent launch. A kernel launched through launch_pdl() may begin while the grid before it on the stream
// is still draining: its CTAs are scheduled as that grid's CTAs exit, so block scheduling, shared-memory carve-out and
// any per-CTA prologue overlap the tail. pdl_sync() must run before the first global-memory access: it waits until the
// preceding grid has completed and its writes are visible, then lets the grid behind this one start the same way.
// (Both instructions are no-ops in a launch without the attribute. ST5_PDL=0 turns the attribute off everywhere.)
__device__ __forceinline__ void pdl_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  int na = 0;
  if (pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    na = 1;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Phi(x) = 0.5 (1 + erf(x / sqrt 2)) and exp(-x^2 / 2) from ONE exponential (Abramowitz-Stegun 7.1.26, |err| < 1.5e-7):
// the GELU of the reference (fairseq/modules/gelu.py:24 -> F.gelu, exact erf form) and its derivative share it.
// MUFU approximations without the denormal fix-up code nvcc wraps around __expf / __fdividef / exp2f (7 extra
// instructions per call in an epilogue that runs once per output element). Arguments here are never subnormal
// (rcp: >= 1) or underflow harmlessly to zero (ex2 of a large negative number).
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gauss_cdf(float x, float& ex) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  const float t = fast_rcp(fmaf(0.3275911f, z, 1.f));
  ex = fast_ex2(-1.4426950408889634f * z * z);
  const float poly = t * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 1.061405429f, -1.453152027f), 1.421413741f), -0.284496736f),
                              0.254829592f);
  const float erf_abs = fmaf(-poly, ex, 1.f);
  return 0.5f * (1.f + copysignf(erf_abs, x));
}
__device__ __forceinline__ float gelu_fwd(float x) {
  float ex;
  return x * gauss_cdf(x, ex);
}
// Throughput-mode GELU (bf16 activations): the tanh form 0.5 x (1 + tanh(sqrt(2/pi)(x + 0.044715 x^3))) on the MUFU
// tanh unit -- 7 instructions instead of 16. |gelu_tanh - gelu_erf| <= 4.8e-4 absolute (< half a bf16 ulp for every
// |y| > 0.13, and vanishing like x^5 near 0); the parity mode (fp32 activations) always uses the exact erf form above.
__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float gelu_tanh_fwd(float x) {
  const float t = fast_tanh(x * fmaf(0.0356774081f, x * x, 0.7978845608f));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float x2 = x * x;
  const float t = fast_tanh(x * fmaf(0.0356774081f, x2, 0.7978845608f));
  const float du = fmaf(0.1070322243f, x2, 0.7978845608f);
  return fmaf(0.5f * x * fmaf(-t, t, 1.f), du, fmaf(0.5f, t, 0.5f));
}
__device__ __forceinline__ float act_grad(float x, int act) {
  if (act == 4) return gelu_tanh_grad(x);
  if (act == 1) return x > 0.f ? 1.f : 0.f;
  if (act == 2) {
    float ex;
    const float cdf = gauss_cdf(x, ex);
    return fmaf(x * 0.39894228040143267794f, ex, cdf);
  }
  if (act == 3) {
    const float t = tanhf(x);
    return 1.f - t * t;
  }
  return 1.f;
}
__host__ __device__ __forceinline__ uint32_t drop_threshold(float p) {
  const float t = p * 65536.f;
  return p <= 0.f ? 0u : (t >= 65535.f ? 65535u : (uint32_t)t);
}

int cast_bf16_launch(const float* src, int64_t src_ld, void* hi, void* lo, int64_t dst_ld, int64_t rows, int64_t cols,
                     cudaStream_t s);
int posenc_fwd_launch(const int64_t* tokens, const float* emb, const void* x, const float* pe, const float* alpha,
                      void* y, int dtype, int64_t B, int64_t T, int64_t C, float drop_p, uint64_t seed, uint64_t offset,
                      cudaStream_t s);
int posenc_bwd_launch(const void* dy, const int64_t* tokens, int64_t padding_idx, const float* pe, void* dx,
                      float* demb, float* dalpha, int dtype, int64_t B, int64_t T, int64_t C, float drop_p,
                      uint64_t seed, uint64_t offset, cudaStream_t s);
int ln_fwd_launch(const void* x, const void* residual, const float* residual_f32, const float* gamma, const float* beta,
                  void* y, float* y_f32, void* s_out, float* mean, float* rstd, int dtype, int64_t rows, int64_t C,
                  float eps, float drop_p, uint64_t seed, uint64_t offset, cudaStream_t s);
int64_t ln_bwd_blocks(int64_t rows);
int ln_bwd_launch(const void* dy, const void* s_in, const float* mean, const float* rstd, const float* gamma, void* ds,
                  void* dx, float* dgamma, float* dbeta, float* dxsum, int dtype, int64_t rows, int64_t C,
                  float drop_p, uint64_t seed, uint64_t offset, cudaStream_t s);
int lrelu_pad_launch(const void* x, void* out, int64_t B, int64_t T, int64_t C, int64_t n_in, int d, int ph, int pad,
                     float slope, cudaStream_t s);
int dropout_launch(const void* x, void* y, int dtype, int64_t n, float drop_p, uint64_t seed, uint64_t offset,
                   cudaStream_t s);
int act_bwd_launch(const void* dy, const void* pre, void* dpre, int dtype, int act, int64_t n, float drop_p,
                   uint64_t seed, uint64_t offset, cudaStream_t s);
int colsum_launch(const void* x, int64_t ld, float* out, int dtype, int64_t rows, int64_t cols, int64_t group_rows,
                  int accumulate, cudaStream_t s);
int attn_fwd_launch(const st5_attn_args& a, cudaStream_t s);
int attn_bwd_launch(const st5_attn_args& a, cudaStream_t s);
int bn_fwd_launch(const void* x, int64_t x_ld, const float* gamma, const float* beta, float* running_mean,
                  float* running_var, float* save_mean, float* save_rstd, void* y, int64_t y_ld, void* y_pre, int dtype,
                  int64_t rows, int64_t C, int training, float momentum, float eps, int act, float drop_p,
                  uint64_t seed, uint64_t offset, float* scratch, cudaStream_t s);
int bn_bwd_launch(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, const void* y_pre, const float* gamma,
                  const float* save_mean, const float* save_rstd, void* dx, int64_t dx_ld, float* dgamma, float* dbeta,
                  int dtype, int64_t rows, int64_t C, int act, float drop_p, uint64_t seed, uint64_t offset,
                  float* scratch, cudaStream_t s);
int64_t conv0_ws_floats(int32_t B, int64_t n, int32_t C, int32_t K, int32_t S);
int conv0_fwd_launch(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                     float* mean, float* rstd, float* ws, int32_t B, int64_t n, int32_t C, int32_t K, int32_t S,
                     float eps, int act, cudaStream_t s);
int conv0_bwd_launch(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                     const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws, int dtype,
                     int32_t B, int64_t n, int32_t C, int32_t K, int32_t S, int act, cudaStream_t s);
int64_t conv0_ln_ws_floats(int32_t B, int64_t n, int32_t C, int32_t K, int32_t S);
int conv0_ln_fwd_launch(const float* wave, const float* w, const float* gamma, const float* beta, void* y, int dtype,
                        float* mean, float* rstd, int32_t B, int64_t n, int32_t C, int32_t K, int32_t S, float eps,
                        int act, cudaStream_t s);
int conv0_ln_bwd_launch(const void* dy, const float* wave, const float* w, const float* gamma, const float* beta,
                        const float* mean, const float* rstd, float* dw, float* dgamma, float* dbeta, float* ws,
                        int dtype, int32_t B, int64_t n, int32_t C, int32_t K, int32_t S, int act, cudaStream_t s);
int act_fwd_launch(const void* x, void* y, int dtype, int act, int64_t n, cudaStream_t s);
int64_t tts_loss_blocks(int B, int L);
int64_t guided_attn_blocks(int n_layers, int B, int heads, int T_out);
int tts_loss_fwd_launch(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                        const float* labels, int64_t lab_bs, const int64_t* olens, int B, int L, int D, int r,
                        float pos_weight, float* sums, float* out, cudaStream_t s);
int tts_loss_bwd_launch(const float* after, const float* before, const float* logits, const float* ys, int64_t y_bs,
                        const float* labels, int64_t lab_bs, const int64_t* olens, const float* sums, const float* g,
                        int B, int L, int D, int r, float pos_weight, float* d_after, float* d_before, float* d_logits,
                        cudaStream_t s);
int guided_attn_fwd_launch(const float* const* att, int n_layers, int B, int H, int heads, int T_out, int T_in,
                           int64_t p_ld, const int64_t* ilens, const int64_t* olens, int r, float sigma, float alpha,
                           float* gsum, float* out, cudaStream_t s);
int guided_attn_bwd_launch(float* const* datt, int n_layers, int B, int H, int heads, int T_out, int T_in, int64_t p_ld,
                           const int64_t* ilens, const int64_t* olens, int r, float sigma, float alpha,
                           const float* gsum, const float* g, int zero_rest, cudaStream_t s);
int64_t ctc_ws_floats(int32_t T, int32_t B, int32_t S_max);
int ctc_loss_launch(const float* logits, int64_t ld_t, int64_t ld_b, const int64_t* targets, const int64_t* tgt_offsets,
                    const int64_t* input_lengths, const int64_t* target_lengths, float* nll, float* grad, float* ws,
                    int32_t T, int32_t B, int32_t V, int32_t S_max, int32_t blank, int32_t zero_infinity,
                    cudaStream_t s);
int ctc_prefix_init_launch(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* t_valid, float* r, int32_t B,
                           int32_t T, int32_t V, int32_t blank, cudaStream_t s);
int ctc_prefix_score_launch(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* utt, const float* r_prev,
                            const int64_t* last, const int64_t* out_len, const int64_t* cs, const int64_t* t_valid,
                            float* log_psi, float* r_out, int32_t H, int32_t T, int32_t K, int32_t V, int32_t blank,
                            int32_t eos, cudaStream_t s);
int beam_gather_rows_launch(const void* const* src, void* const* dst, const int64_t* parent, int32_t L, int32_t H,
                            int32_t n_rows, int64_t row_bytes, int64_t src_bs, int64_t dst_bs, cudaStream_t s);
int sumsq_launch(const float* x, int64_t n, float* out, cudaStream_t s);
int adam_launch(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n, float lr, float beta1,
                float beta2, float eps, float weight_decay, int64_t step, const float* grad_norm_sq, float max_norm,
                float grad_mul, const float* lr_dev, const int64_t* step_dev, cudaStream_t s);

}  // namespace st5
