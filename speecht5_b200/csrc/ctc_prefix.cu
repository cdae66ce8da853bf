// CTC prefix scoring for joint CTC/attention beam search (reference: speecht5/sequence_generator.py:273-284 builds the
// scorer, :370-418 calls it once per hypothesis per step; the scorer is espnet's CTCPrefixScore, numpy on the host,
// Algorithm 2 of Watanabe et al., "Hybrid CTC/attention architecture for end-to-end speech recognition"), and the
// key/value-cache row gather the beam reorder needs.
//   1 ctc_prefix_init_kernel   (thread per utterance)  r_n = logzero, r_b[t] = sum_{tau <= t} x[tau, blank] over the
//                              utterance's T_b valid frames (sequential fp32 sum, the reference's order)
//   2 ctc_prefix_score_kernel  (CTA per hypothesis, thread per candidate label)  the forward recursion of every
//                              candidate c of hypothesis h over frames t = max(out_len, 1) .. T_b - 1:
//                                r_n[t](hc) = lae(r_n[t-1](hc), phi[t-1]) + x[t, c]
//                                r_b[t](hc) = lae(r_n[t-1](hc), r_b[t-1](hc)) + x[t, blank]
//                                psi        = lae(psi, phi[t-1] + x[t, c])
//                              phi = lae(r_prev_n, r_prev_b), or r_prev_b where c repeats the last label. The chains are
//                              independent; the frames are staged CHUNK at a time in shared memory (the candidate's
//                              column, the blank column and phi of the chunk), so the recursion itself reads only smem.
//   3 beam_gather_rows_kernel  rows [0, n) of every layer's [H, max_len, 2C] key/value cache, by parent index, into a
//                              second buffer set (16-byte vectors, grid over (row chunk, hypothesis, layer)).
// The sentinel is the reference's finite logzero = -1e10, not -inf: CTC-infeasible candidates (a prefix longer than the
// frame count) keep finite scores there and the ranking depends on them. lae() is numpy's float32 logaddexp.
#include "kernels.cuh"

namespace st5 {

constexpr float CTC_LOGZERO = -1e10f;
constexpr int CTCP_CHUNK = 32;     // frames staged per pass (32 x 256 candidates = 32 KB of smem)
constexpr int CTCP_MAX_T = 1500;   // 30 s of audio at the 20 ms encoder frame rate
constexpr int CTCP_MAX_K = 256;
constexpr int GATHER_MAX_LAYERS = 32;

// numpy's npy_logaddexpf: equal arguments (infinities of one sign included) give x + ln 2
__device__ __forceinline__ float lae(float x, float y) {
  if (x == y) return x + 0.693147180559945309f;
  const float d = x - y;
  return d > 0.f ? x + log1pf(expf(-d)) : y + log1pf(expf(d));
}

__global__ void ctc_prefix_init_kernel(const float* __restrict__ x, int64_t ld_b, int64_t ld_t,
                                       const int64_t* __restrict__ t_valid, float* __restrict__ r, int B, int T,
                                       int blank) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int Tb = (int)min((int64_t)T, t_valid[b]);
  const float* xb = x + (int64_t)b * ld_b + blank;
  float* rb = r + (int64_t)b * T * 2;
  float acc = 0.f;
  for (int t = 0; t < T; ++t) {
    float vb = CTC_LOGZERO;
    if (t < Tb) {
      acc = t == 0 ? xb[0] : acc + xb[(int64_t)t * ld_t];
      vb = acc;
    }
    rb[2 * t] = CTC_LOGZERO;
    rb[2 * t + 1] = vb;
  }
}

// r_out layout [H][T][2][K]: at a fixed frame the K candidates of a hypothesis write adjacent words (coalesced).
__global__ void __launch_bounds__(CTCP_MAX_K)
    ctc_prefix_score_kernel(const float* __restrict__ x, int64_t ld_b, int64_t ld_t, const int64_t* __restrict__ utt,
                            const float* __restrict__ r_prev, const int64_t* __restrict__ last,
                            const int64_t* __restrict__ out_len, const int64_t* __restrict__ cs,
                            const int64_t* __restrict__ t_valid, float* __restrict__ log_psi, float* __restrict__ r_out,
                            int T, int K, int blank, int eos) {
  __shared__ float xs_sh[CTCP_CHUNK][CTCP_MAX_K];
  __shared__ float xb_sh[CTCP_CHUNK];
  __shared__ float phi_sh[CTCP_CHUNK];   // lae(r_prev_n, r_prev_b) of frame t - 1
  __shared__ float rpb_sh[CTCP_CHUNK];   // r_prev_b of frame t - 1
  const int h = blockIdx.x;
  const int k = threadIdx.x;
  const bool on = k < K;
  const int64_t u = utt[h];
  const int Tb = (int)min((int64_t)T, t_valid[u]);
  const int64_t L = out_len[h];
  const int64_t lastl = last[h];
  const int c = on ? (int)cs[(int64_t)h * K + k] : blank;
  const bool repeat = L > 0 && c == lastl;
  const float* xu = x + u * ld_b;
  const float* rp = r_prev + (int64_t)h * T * 2;
  float* ro = r_out + (int64_t)h * T * 2 * K + k;
  const int64_t fstride = 2 * (int64_t)K;

  // rows below the start: logzero, except row 0 of the empty prefix (r_n[0] = x[0, c])
  const int start = (int)max(min(L, (int64_t)T + 1), (int64_t)1);
  float rn = CTC_LOGZERO, rb = CTC_LOGZERO, psi = CTC_LOGZERO;
  if (L == 0 && Tb > 0) rn = psi = xu[c];
  if (on) {
    const int lo_end = min(start, T);
    for (int t = 0; t < lo_end; ++t) {
      const bool row0 = t == 0 && L == 0 && Tb > 0;
      ro[t * fstride] = row0 ? rn : CTC_LOGZERO;
      ro[t * fstride + K] = CTC_LOGZERO;
    }
  }
  // the recursion over [start, Tb)
  for (int t0 = start; t0 < Tb; t0 += CTCP_CHUNK) {
    const int n = min(CTCP_CHUNK, Tb - t0);
    __syncthreads();  // (the previous chunk's reads are done)
    if (on)
      for (int i = 0; i < n; ++i) xs_sh[i][k] = xu[(int64_t)(t0 + i) * ld_t + c];
    for (int i = k; i < n; i += blockDim.x) {
      const int t = t0 + i;
      xb_sh[i] = xu[(int64_t)t * ld_t + blank];
      const float pn = rp[2 * (t - 1)], pb = rp[2 * (t - 1) + 1];
      phi_sh[i] = lae(pn, pb);
      rpb_sh[i] = pb;
    }
    __syncthreads();
    if (on) {
      for (int i = 0; i < n; ++i) {
        const float phi = repeat ? rpb_sh[i] : phi_sh[i];
        const float xc = xs_sh[i][k];
        const float rn_new = lae(rn, phi) + xc;
        const float rb_new = lae(rn, rb) + xb_sh[i];
        psi = lae(psi, phi + xc);
        rn = rn_new;
        rb = rb_new;
        const int64_t o = (int64_t)(t0 + i) * fstride;
        ro[o] = rn;
        ro[o + K] = rb;
      }
    }
  }
  if (!on) return;
  for (int t = max(start, Tb); t < T; ++t) {  // frames past the utterance: unused, defined
    ro[t * fstride] = CTC_LOGZERO;
    ro[t * fstride + K] = CTC_LOGZERO;
  }
  if (c == eos) psi = Tb > 0 ? lae(rp[2 * (Tb - 1)], rp[2 * (Tb - 1) + 1]) : CTC_LOGZERO;
  if (c == blank) psi = CTC_LOGZERO;
  log_psi[(int64_t)h * K + k] = psi;
}

struct GatherPtrs {
  const char* src[GATHER_MAX_LAYERS];
  char* dst[GATHER_MAX_LAYERS];
};

__global__ void beam_gather_rows_kernel(GatherPtrs p, const int64_t* __restrict__ parent, int64_t vecs,
                                        int64_t src_bs, int64_t dst_bs) {
  const int h = blockIdx.y, l = blockIdx.z;
  const int4* s = reinterpret_cast<const int4*>(p.src[l] + parent[h] * src_bs);
  int4* d = reinterpret_cast<int4*>(p.dst[l] + (int64_t)h * dst_bs);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += (int64_t)gridDim.x * blockDim.x)
    d[i] = s[i];
}

int ctc_prefix_init_launch(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* t_valid, float* r, int32_t B,
                           int32_t T, int32_t V, int32_t blank, cudaStream_t st) {
  if (B <= 0 || T <= 0 || T > CTCP_MAX_T || V <= 0 || blank < 0 || blank >= V || ld_t < V) return -2;
  ctc_prefix_init_kernel<<<(B + 127) / 128, 128, 0, st>>>(x, ld_b, ld_t, t_valid, r, B, T, blank);
  return (int)cudaGetLastError();
}

int ctc_prefix_score_launch(const float* x, int64_t ld_b, int64_t ld_t, const int64_t* utt, const float* r_prev,
                            const int64_t* last, const int64_t* out_len, const int64_t* cs, const int64_t* t_valid,
                            float* log_psi, float* r_out, int32_t H, int32_t T, int32_t K, int32_t V, int32_t blank,
                            int32_t eos, cudaStream_t st) {
  if (H <= 0 || T <= 0 || T > CTCP_MAX_T || K <= 0 || K > CTCP_MAX_K || V <= 0 || blank < 0 || blank >= V || eos < 0 ||
      eos >= V || ld_t < V)
    return -2;
  const int threads = (K + 31) / 32 * 32;
  ctc_prefix_score_kernel<<<H, threads, 0, st>>>(x, ld_b, ld_t, utt, r_prev, last, out_len, cs, t_valid, log_psi, r_out,
                                                  T, K, blank, eos);
  return (int)cudaGetLastError();
}

int beam_gather_rows_launch(const void* const* src, void* const* dst, const int64_t* parent, int32_t L, int32_t H,
                            int32_t n_rows, int64_t row_bytes, int64_t src_bs, int64_t dst_bs, cudaStream_t st) {
  if (L <= 0 || L > GATHER_MAX_LAYERS || H <= 0 || n_rows < 0 || row_bytes <= 0 || row_bytes % 16 || src_bs % 16 ||
      dst_bs % 16 || (int64_t)n_rows * row_bytes > src_bs || (int64_t)n_rows * row_bytes > dst_bs)
    return -2;
  if (n_rows == 0) return 0;
  GatherPtrs p;
  for (int l = 0; l < L; ++l) {
    if (((uintptr_t)src[l] | (uintptr_t)dst[l]) % 16) return -3;
    p.src[l] = static_cast<const char*>(src[l]);
    p.dst[l] = static_cast<char*>(dst[l]);
  }
  const int64_t vecs = (int64_t)n_rows * row_bytes / 16;
  const int threads = 256;
  const int64_t blocks = min((vecs + threads - 1) / threads, (int64_t)64);
  beam_gather_rows_kernel<<<dim3((unsigned)blocks, H, L), threads, 0, st>>>(p, parent, vecs, src_bs, dst_bs);
  return (int)cudaGetLastError();
}

}  // namespace st5
