// Video question answering head (TVQA / How2QA): HeroForVideoQA.get_modularized_video of the
// reference (model/videoQA.py:36-59) on the packed output of the query-fused temporal stack.
//
//   x[v, q, t]  = y[frame_tok[v, q, t]]            (0 where frame_tok == -1: padded frame)
//   s_se / s_qa = w_se . x / w_qa . x, mask_logits (score where valid, exactly -1e4 elsewhere)
//   a_se        = softmax over the Nq candidates q   (per question v and frame t)
//   a_qa        = softmax over the frames t          (per question v and candidate q)
//   P_se[v, t]  = sum_q a_se x                       P_qa[v, q] = sum_t a_qa x
//
// Two launches each way: per-row dot products (a warp per (v, q, t) row), then the softmaxes and
// the weighted sums (a CTA per output row forward, a CTA per (v, q) backward). HBM / latency bound
// and tiny next to the encoder; the point is launch count and no host round trip.
#include "common.h"
#include "ptx.cuh"

namespace hero {

constexpr float kQaMaskFill = -1e4f;   // mask_logits (model/modeling_utils.py:42-43)
constexpr int QA_MAX_T = 1024;         // frames per clip (shared-memory softmax over t)
constexpr int QA_MAX_NQ = 64;          // answer candidates per question

// Sum / max over a 256-thread CTA (8 warps).
template <bool is_max>
__device__ __forceinline__ float qa_block_reduce(float v, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float u = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, u) : v + u;
  }
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) r = is_max ? fmaxf(r, red[w]) : r + red[w];
  return r;
}

// One warp per (v, q, t) row: a = u . x, b = w . x. The forward passes the two pool weights (one
// vector each), the backward dP_se (u_per_t: row [v, t]) and dP_qa (w_per_q: row [v, q]). Rows
// without a frame get `fill`.
__global__ void __launch_bounds__(256)
videoqa_dots_kernel(const float* __restrict__ y, const int32_t* __restrict__ frame_tok, int nq,
                    int T, long long rows, int h, const float* __restrict__ u, int u_per_t,
                    const float* __restrict__ w, int w_per_q, float fill, float* __restrict__ out_a,
                    float* __restrict__ out_b) {
  pdl_wait();
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int tok = frame_tok[r];
  if (tok < 0) {
    if (lane == 0) out_a[r] = out_b[r] = fill;
    return;
  }
  const long long t = r % T, vq = r / T, v = vq / nq;
  const float* ur = u + (u_per_t ? (v * T + t) * h : 0);
  const float* wr = w + (w_per_q ? vq * h : 0);
  const float* x = y + (long long)tok * h;
  float a = 0.f, b = 0.f;
  for (int c = lane * 4; c < h; c += 128) {
    const float4 xv = *reinterpret_cast<const float4*>(x + c);
    const float4 uv = *reinterpret_cast<const float4*>(ur + c);
    const float4 wv = *reinterpret_cast<const float4*>(wr + c);
    a += xv.x * uv.x + xv.y * uv.y + xv.z * uv.z + xv.w * uv.w;
    b += xv.x * wv.x + xv.y * wv.y + xv.z * wv.z + xv.w * wv.w;
  }
  a = warp_sum(a);
  b = warp_sum(b);
  if (lane == 0) {
    out_a[r] = a;
    out_b[r] = b;
  }
}

// Forward pooling. CTAs [0, Nv*T): P_se[v, t] with the softmax over q of s_se[v, :, t]; CTAs
// [Nv*T, Nv*T + Nv*Nq): P_qa[v, q] with the softmax over t of s_qa[v, q, :]. The probabilities are
// written for the backward (a_se, a_qa: [Nv, Nq, T]).
__global__ void __launch_bounds__(256)
videoqa_pool_fwd_kernel(const float* __restrict__ y, const int32_t* __restrict__ frame_tok,
                        const float* __restrict__ s_se, const float* __restrict__ s_qa, int nv,
                        int nq, int T, int h, float* __restrict__ p_se, float* __restrict__ p_qa,
                        float* __restrict__ a_se, float* __restrict__ a_qa) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float s_p[QA_MAX_T];
  __shared__ int s_tok[QA_MAX_T];
  __shared__ float red[8];
  const int n_se = nv * T;
  if ((int)blockIdx.x < n_se) {
    const int v = blockIdx.x / T, t = blockIdx.x % T;
    // softmax over the nq (<= 64) candidates, computed redundantly by every thread
    const float* sv = s_se + (long long)v * nq * T + t;
    float m = -INFINITY;
    for (int q = 0; q < nq; ++q) m = fmaxf(m, sv[(long long)q * T]);
    float sum = 0.f;
    for (int q = 0; q < nq; ++q) sum += __expf(sv[(long long)q * T] - m);
    if (threadIdx.x < nq) {
      const int q = threadIdx.x;
      const long long i = ((long long)v * nq + q) * T + t;
      s_p[q] = __expf(sv[(long long)q * T] - m) / sum;
      s_tok[q] = frame_tok[i];
      a_se[i] = s_p[q];
    }
    __syncthreads();
    float* out = p_se + ((long long)v * T + t) * h;
    for (int c = threadIdx.x; c < h; c += blockDim.x) {
      float acc = 0.f;
      for (int q = 0; q < nq; ++q)
        if (s_tok[q] >= 0) acc = fmaf(s_p[q], y[(long long)s_tok[q] * h + c], acc);
      out[c] = acc;
    }
    return;
  }
  const long long vq = (int)blockIdx.x - n_se;
  const float* s = s_qa + vq * T;
  float m = -INFINITY;
  for (int t = threadIdx.x; t < T; t += blockDim.x) m = fmaxf(m, s[t]);
  m = qa_block_reduce<true>(m, red);
  float sum = 0.f;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const float e = __expf(s[t] - m);
    s_p[t] = e;
    s_tok[t] = frame_tok[vq * T + t];
    sum += e;
  }
  sum = qa_block_reduce<false>(sum, red);
  const float inv = 1.0f / sum;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    s_p[t] *= inv;
    a_qa[vq * T + t] = s_p[t];
  }
  __syncthreads();
  float* out = p_qa + vq * h;
  for (int c = threadIdx.x; c < h; c += blockDim.x) {
    float acc = 0.f;
    for (int t = 0; t < T; ++t)
      if (s_tok[t] >= 0) acc = fmaf(s_p[t], y[(long long)s_tok[t] * h + c], acc);
    out[c] = acc;
  }
}

// Backward, one CTA per (v, q): with dA_se = dP_se[v, t] . x and dA_qa = dP_qa[v, q] . x
//   g_se[t] = a_se (dA_se - sum_q' a_se dA_se)   g_qa[t] = a_qa (dA_qa - sum_t' a_qa dA_qa)
// (both 0 at padded frames: mask_logits multiplies the score by the mask), then per valid frame
//   dx = a_se dP_se[v, t] + a_qa dP_qa[v, q] + g_se w_se + g_qa w_qa   -> dy[frame_tok]
// and dw_se += sum_t g_se x, dw_qa += sum_t g_qa x (fp32 atomics, one per column and CTA).
__global__ void __launch_bounds__(256)
videoqa_pool_bwd_kernel(const float* __restrict__ y, const int32_t* __restrict__ frame_tok,
                        const float* __restrict__ a_se, const float* __restrict__ a_qa,
                        const float* __restrict__ da_se, const float* __restrict__ da_qa,
                        const float* __restrict__ dp_se, const float* __restrict__ dp_qa,
                        const float* __restrict__ w_se, const float* __restrict__ w_qa, int nq,
                        int T, int h, float* __restrict__ dy, float* __restrict__ dw_se,
                        float* __restrict__ dw_qa) {
  pdl_wait();
  pdl_launch_dependents();
  __shared__ float s_ase[QA_MAX_T], s_aqa[QA_MAX_T], s_gse[QA_MAX_T], s_gqa[QA_MAX_T];
  __shared__ int s_tok[QA_MAX_T];
  __shared__ float red[8];
  const long long vq = blockIdx.x;
  const long long v = vq / nq;
  const long long base = vq * T;
  float dot = 0.f;
  for (int t = threadIdx.x; t < T; t += blockDim.x) dot += a_qa[base + t] * da_qa[base + t];
  dot = qa_block_reduce<false>(dot, red);
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const int tok = frame_tok[base + t];
    const float ase = a_se[base + t], aqa = a_qa[base + t];
    float gse = 0.f, gqa = 0.f;
    if (tok >= 0) {
      float sse = 0.f;             // sum over the candidates of this question at frame t
      for (int q = 0; q < nq; ++q) {
        const long long i = (v * nq + q) * T + t;
        sse += a_se[i] * da_se[i];
      }
      gse = ase * (da_se[base + t] - sse);
      gqa = aqa * (da_qa[base + t] - dot);
    }
    s_tok[t] = tok;
    s_ase[t] = ase;
    s_aqa[t] = aqa;
    s_gse[t] = gse;
    s_gqa[t] = gqa;
  }
  __syncthreads();
  const float* dpq = dp_qa + vq * h;
  for (int c = threadIdx.x; c < h; c += blockDim.x) {
    const float wse = w_se[c], wqa = w_qa[c], dq = dpq[c];
    float acc_se = 0.f, acc_qa = 0.f;
    for (int t = 0; t < T; ++t) {
      const int tok = s_tok[t];
      if (tok < 0) continue;
      const long long row = (long long)tok * h + c;
      const float xv = y[row];
      acc_se = fmaf(s_gse[t], xv, acc_se);
      acc_qa = fmaf(s_gqa[t], xv, acc_qa);
      dy[row] = s_ase[t] * dp_se[(v * T + t) * h + c] + s_aqa[t] * dq + s_gse[t] * wse +
                s_gqa[t] * wqa;
    }
    atomicAdd(dw_se + c, acc_se);
    atomicAdd(dw_qa + c, acc_qa);
  }
}

}  // namespace hero

using namespace hero;

extern "C" int hero_videoqa_pool_fwd(const float* y, const int32_t* frame_tok, const float* w_se,
                                     const float* w_qa, int32_t nv, int32_t nq, int32_t t,
                                     int32_t h, float* s_se, float* s_qa, float* a_se, float* a_qa,
                                     float* p_se, float* p_qa, void* stream) {
  HERO_REQUIRE(y && frame_tok && w_se && w_qa && s_se && s_qa && a_se && a_qa && p_se && p_qa,
               "videoqa_pool_fwd: null pointer");
  HERO_REQUIRE(nq >= 1 && nq <= QA_MAX_NQ && t >= 1 && t <= QA_MAX_T && h > 0 && h % 4 == 0,
               "videoqa_pool_fwd: unsupported shape (nq %d, t %d, h %d)", nq, t, h);
  if (nv <= 0) return HERO_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long rows = (long long)nv * nq * t;
  HERO_CUDA_CHECK(launch_pdl(videoqa_dots_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0,
                             st, y, frame_tok, nq, t, rows, h, w_se, 0, w_qa, 0, kQaMaskFill,
                             s_se, s_qa));
  HERO_CUDA_CHECK(launch_pdl(videoqa_pool_fwd_kernel,
                             dim3((unsigned)((long long)nv * t + (long long)nv * nq)), dim3(256), 0,
                             st, y, frame_tok, s_se, s_qa, nv, nq, t, h, p_se, p_qa, a_se, a_qa));
  return HERO_OK;
}

extern "C" int hero_videoqa_pool_bwd(const float* y, const int32_t* frame_tok, const float* w_se,
                                     const float* w_qa, const float* a_se, const float* a_qa,
                                     const float* dp_se, const float* dp_qa, int32_t nv,
                                     int32_t nq, int32_t t, int32_t h, float* da_se, float* da_qa,
                                     float* dy, float* dw_se, float* dw_qa, void* stream) {
  HERO_REQUIRE(y && frame_tok && w_se && w_qa && a_se && a_qa && dp_se && dp_qa && da_se && da_qa &&
                   dy && dw_se && dw_qa,
               "videoqa_pool_bwd: null pointer");
  HERO_REQUIRE(nq >= 1 && nq <= QA_MAX_NQ && t >= 1 && t <= QA_MAX_T && h > 0 && h % 4 == 0,
               "videoqa_pool_bwd: unsupported shape (nq %d, t %d, h %d)", nq, t, h);
  if (nv <= 0) return HERO_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long rows = (long long)nv * nq * t;
  HERO_CUDA_CHECK(launch_pdl(videoqa_dots_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0,
                             st, y, frame_tok, nq, t, rows, h, dp_se, 1, dp_qa, 1, 0.0f, da_se,
                             da_qa));
  HERO_CUDA_CHECK(launch_pdl(videoqa_pool_bwd_kernel, dim3((unsigned)((long long)nv * nq)),
                             dim3(256), 0, st, y, frame_tok, a_se, a_qa, da_se, da_qa, dp_se,
                             dp_qa, w_se, w_qa, nq, t, h, dy, dw_se, dw_qa));
  return HERO_OK;
}
