// Flat-buffer fused AdamW and sum-of-squares (global-norm clipping), HBM-bound.
// Arithmetic follows the reference's optim/adamw.py:80-104: bias-corrected step size computed on
// the host, eps added to sqrt(v) (not inside), decoupled weight decay applied AFTER the Adam
// update on the already-updated parameter with the un-corrected lr.
#include "common.h"
#include "ptx.cuh"

namespace hero {

// 16-byte vector accesses on all seven streams (p, g, m, v read; p, m, v + bf16 written: 30 B per
// parameter). `clip` (device scalar: sum of squares of ALL gradients) folds global-norm clipping
// into the update without a host round trip.
__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
             float* __restrict__ v, __nv_bfloat16* __restrict__ p_bf16, long long n, float step_size,
             float beta1, float beta2, float eps, float lr_wd, float grad_scale,
             const float* __restrict__ clip, float clip_max_norm) {
  if (clip != nullptr) {
    const float norm = sqrtf(__ldg(clip));
    grad_scale *= fminf(1.0f, clip_max_norm / (norm + 1e-6f));
  }
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const float ob1 = 1.0f - beta1, ob2 = 1.0f - beta2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(g) + i);
    float4 m4 = reinterpret_cast<float4*>(m)[i];
    float4 v4 = reinterpret_cast<float4*>(v)[i];
    float4 p4 = reinterpret_cast<float4*>(p)[i];
    const float gr[4] = {g4.x * grad_scale, g4.y * grad_scale, g4.z * grad_scale, g4.w * grad_scale};
    float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
    float pp[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mm[j] = beta1 * mm[j] + ob1 * gr[j];
      vv[j] = beta2 * vv[j] + ob2 * gr[j] * gr[j];
      pp[j] = pp[j] - step_size * (mm[j] / (sqrtf(vv[j]) + eps));
      if (lr_wd > 0.0f) pp[j] = pp[j] - lr_wd * pp[j];
    }
    reinterpret_cast<float4*>(m)[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
    reinterpret_cast<float4*>(v)[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    reinterpret_cast<float4*>(p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
    if (p_bf16 != nullptr) {
      uint2 u;
      u.x = pack_bf16x2(pp[0], pp[1]);
      u.y = pack_bf16x2(pp[2], pp[3]);
      reinterpret_cast<uint2*>(p_bf16)[i] = u;
    }
  }
  // tail (n not a multiple of 4)
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gr = g[i] * grad_scale;
    const float mi = beta1 * m[i] + ob1 * gr;
    const float vi = beta2 * v[i] + ob2 * gr * gr;
    float pi = p[i] - step_size * (mi / (sqrtf(vi) + eps));
    if (lr_wd > 0.0f) pi = pi - lr_wd * pi;
    m[i] = mi;
    v[i] = vi;
    p[i] = pi;
    if (p_bf16 != nullptr) p_bf16[i] = __float2bfloat16(pi);
  }
}

__global__ void __launch_bounds__(256)
sumsq_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  float s = 0.f;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(x) + i);
    s = fmaf(t.x, t.x, s); s = fmaf(t.y, t.y, s); s = fmaf(t.z, t.z, s); s = fmaf(t.w, t.w, s);
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float t = x[i];
    s = fmaf(t, t, s);
  }
  s = warp_sum(s);
  __shared__ float sm[8];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 8) {
    float t = sm[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(0xffu, t, o);
    if (threadIdx.x == 0) atomicAdd(out, t);
  }
}

// Finish of the fused LM-head cross entropy: combine the (max, sum exp) partials of a row.
__global__ void __launch_bounds__(128)
ce_finish_kernel(const float2* __restrict__ part, long long ld, int n_slabs,
                 const float* __restrict__ lab, int m, float* __restrict__ loss,
                 float* __restrict__ lse) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  float mx = -INFINITY;
  for (int t = 0; t < n_slabs; ++t) mx = fmaxf(mx, part[(long long)t * ld + r].x);   // coalesced in r
  float s = 0.f;
  for (int t = 0; t < n_slabs; ++t) {
    const float2 p = part[(long long)t * ld + r];
    s += p.y * __expf(p.x - mx);
  }
  const float l = mx + __logf(s);
  lse[r] = l;
  loss[r] = l - lab[r];
}

}  // namespace hero

using namespace hero;

extern "C" int hero_adamw_step(float* p, const float* g, float* m, float* v, void* p_bf16,
                               int64_t n, float step_size, float beta1, float beta2, float eps,
                               float lr_wd, float grad_scale, const float* clip_sumsq,
                               float clip_max_norm, void* stream) {
  HERO_REQUIRE(p && g && m && v && n >= 0, "adamw: bad args");
  HERO_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) |
                 reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15u) == 0 &&
                   (reinterpret_cast<uintptr_t>(p_bf16) & 7u) == 0,
               "adamw: buffers must be 16-byte aligned (bf16 copy 8-byte)");
  if (n == 0) return HERO_OK;
  const int sms = sm_count();
  if (sms <= 0) return set_error(HERO_ERR_NO_DEVICE, "no CUDA device");
  long long blocks = (n / 4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > sms * 8LL) blocks = sms * 8LL;
  adamw_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, reinterpret_cast<__nv_bfloat16*>(p_bf16), n, step_size, beta1, beta2, eps, lr_wd,
      grad_scale, clip_sumsq, clip_max_norm);
  HERO_LAUNCH_CHECK();
  return HERO_OK;
}

extern "C" int hero_ce_finish(const void* ce_partial, int64_t ld_partial, int32_t n_slabs,
                              const float* label_logit, int32_t m, float* loss, float* lse,
                              void* stream) {
  HERO_REQUIRE(ce_partial && label_logit && loss && lse && n_slabs > 0 && ld_partial >= m,
               "ce_finish: bad args");
  if (m <= 0) return HERO_OK;
  ce_finish_kernel<<<(m + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float2*>(ce_partial), ld_partial, n_slabs, label_logit, m, loss, lse);
  HERO_LAUNCH_CHECK();
  return HERO_OK;
}

extern "C" int hero_sumsq_f32(const float* x, int64_t n, float* out, void* stream) {
  HERO_REQUIRE(x && out && n >= 0, "sumsq: bad args");
  if (n == 0) return HERO_OK;
  const int sms = sm_count();
  if (sms <= 0) return set_error(HERO_ERR_NO_DEVICE, "no CUDA device");
  HERO_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15u) == 0, "sumsq: x must be 16-byte aligned");
  long long blocks = (n / 4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > sms * 8LL) blocks = sms * 8LL;
  sumsq_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, n, out);
  HERO_LAUNCH_CHECK();
  return HERO_OK;
}
