// K6 - fused optimizer updates.  One pass over (p, g, m, v): 28 B/param for AdamW, the HBM-bound
// kernel of the step at the reference's batch sizes.  Replaces optimizer.step() of
// torch.optim.AdamW / Adam / SGD as built by engine/optimizer/optim.py:15-71 (the reference's
// `_foreach` path issues ~10 elementwise launches per step and re-reads every buffer).
//
// Also: the split-K reduction of the tensor-core dW partials is folded into the same pass, and the
// bf16 shadow of the weights (B operand of the next tcgen05 forward) is refreshed here, so neither
// costs an extra trip through HBM.
#include <cmath>
#include <cstdlib>

#include "common.cuh"
#include "optim.cuh"

namespace uml {

// g = sum_s parts[s*stride + i] (n_parts >= 1) + w2 * g2[i]
template <bool kVec>
__global__ void __launch_bounds__(256)
    adam_kernel(float* __restrict__ p, const float* __restrict__ parts, int n_parts, int64_t stride,
                const float* __restrict__ g2, float w2, float* __restrict__ m, float* __restrict__ v, int64_t n,
                AdamArgs a, __nv_bfloat16* __restrict__ shadow, float* __restrict__ g_out) {
  const int64_t tid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t nthreads = static_cast<int64_t>(gridDim.x) * blockDim.x;
  if (kVec) {
    const int64_t nv = n >> 2;
    for (int64_t i = tid; i < nv; i += nthreads) {
      float4 g = reinterpret_cast<const float4*>(parts)[i];
      for (int s = 1; s < n_parts; ++s) {
        const float4 q = reinterpret_cast<const float4*>(parts + s * stride)[i];
        g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
      }
      if (g2) {
        const float4 q = reinterpret_cast<const float4*>(g2)[i];
        g.x = fmaf(w2, q.x, g.x); g.y = fmaf(w2, q.y, g.y); g.z = fmaf(w2, q.z, g.z); g.w = fmaf(w2, q.w, g.w);
      }
      float4 w = reinterpret_cast<float4*>(p)[i];
      float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
      w.x = adam_one(a, w.x, g.x, mm.x, vv.x);
      w.y = adam_one(a, w.y, g.y, mm.y, vv.y);
      w.z = adam_one(a, w.z, g.z, mm.z, vv.z);
      w.w = adam_one(a, w.w, g.w, mm.w, vv.w);
      reinterpret_cast<float4*>(p)[i] = w;
      reinterpret_cast<float4*>(m)[i] = mm;
      reinterpret_cast<float4*>(v)[i] = vv;
      if (shadow) reinterpret_cast<uint2*>(shadow)[i] = pack_bf16x4(w);
      if (g_out) reinterpret_cast<float4*>(g_out)[i] = g;
    }
  } else {
    for (int64_t i = tid; i < n; i += nthreads) {
      float g = parts[i];
      for (int s = 1; s < n_parts; ++s) g += parts[s * stride + i];
      if (g2) g = fmaf(w2, g2[i], g);
      float mm = m[i], vv = v[i];
      const float w = adam_one(a, p[i], g, mm, vv);
      p[i] = w;
      m[i] = mm;
      v[i] = vv;
      if (shadow) shadow[i] = __float2bfloat16_rn(w);
      if (g_out) g_out[i] = g;
    }
  }
}

__global__ void __launch_bounds__(256)
    sgd_kernel(float* __restrict__ p, const float* __restrict__ g1, const float* __restrict__ g2, float w2,
               float* __restrict__ buf, int64_t n, float lr, float momentum, float wd, int first,
               __nv_bfloat16* __restrict__ shadow) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float g = g1[i];
    if (g2) g = fmaf(w2, g2[i], g);
    const float w = p[i];
    g = fmaf(wd, w, g);
    const float b = first ? g : fmaf(momentum, buf[i], g);
    buf[i] = b;
    const float nw = w - lr * b;
    p[i] = nw;
    if (shadow) shadow[i] = __float2bfloat16_rn(nw);
  }
}

__global__ void __launch_bounds__(256)
    sum_partials_kernel(const float* __restrict__ parts, int n_parts, int64_t stride, int64_t n4,
                        float* __restrict__ out) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 g = reinterpret_cast<const float4*>(parts)[i];
    for (int s = 1; s < n_parts; ++s) {
      const float4 q = reinterpret_cast<const float4*>(parts + s * stride)[i];
      g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
    }
    reinterpret_cast<float4*>(out)[i] = g;
  }
}

static int launch_adam(float* p, const float* parts, int n_parts, int64_t stride, const float* g2, float w2, float* m,
                       float* v, int64_t n, const AdamArgs& a, uint16_t* shadow, float* g_out, cudaStream_t st) {
  if (n == 0) return 0;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  const bool vec = (n % 4 == 0) && (stride % 4 == 0) && al16(p) && al16(parts) && al16(m) && al16(v) &&
                   (!g2 || al16(g2)) && (!shadow || (reinterpret_cast<uintptr_t>(shadow) & 7u) == 0) &&
                   (!g_out || al16(g_out));
  const int64_t work = vec ? n / 4 : n;
  // a multiple of the SM count; 8 CTAs of 256 threads keep 64 warps resident per SM
  static int ctas_per_sm = 0;
  if (ctas_per_sm == 0) {
    const char* e = getenv("UML_ADAM_CTAS_PER_SM");
    ctas_per_sm = e && atoi(e) > 0 ? atoi(e) : 8;
  }
  const int grid = static_cast<int>(std::min<int64_t>((work + 255) / 256, static_cast<int64_t>(sm_count()) * ctas_per_sm));
  __nv_bfloat16* sh = reinterpret_cast<__nv_bfloat16*>(shadow);
  if (vec)
    UML_CUDA(launch_kernel(adam_kernel<true>, dim3(grid), dim3(256), 0, st, 1, p, parts, n_parts, stride, g2, w2, m, v, n,
                           a, sh, g_out));
  else
    UML_CUDA(launch_kernel(adam_kernel<false>, dim3(grid), dim3(256), 0, st, 1, p, parts, n_parts, stride, g2, w2, m, v, n,
                           a, sh, g_out));
  return 0;
}

}  // namespace uml

extern "C" {

int uml_adamw_step(float* p, const float* g, const float* g2, float g2_weight, float* m, float* v, int64_t n,
                   double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                   int32_t decoupled, uint16_t* p_bf16, void* stream) {
  using namespace uml;
  UML_REQUIRE(p && g && m && v && n >= 0 && step >= 1, "adamw_step: bad arguments");
  return launch_adam(p, g, 1, 0, g2, g2_weight, m, v, n, make_adam(lr, beta1, beta2, eps, weight_decay, step, decoupled),
                     p_bf16, nullptr, as_stream(stream));
}

int uml_adamw_step_partials(float* p, const float* partials, int32_t n_splits, int64_t split_stride, float* m, float* v,
                            int64_t n, double lr, double beta1, double beta2, double eps, double weight_decay,
                            int64_t step, int32_t decoupled, uint16_t* p_bf16, float* g_out, void* stream) {
  using namespace uml;
  UML_REQUIRE(p && partials && m && v && n >= 0 && step >= 1 && n_splits >= 1 && split_stride >= n,
              "adamw_step_partials: bad arguments");
  return launch_adam(p, partials, n_splits, split_stride, nullptr, 0.f, m, v, n,
                     make_adam(lr, beta1, beta2, eps, weight_decay, step, decoupled), p_bf16, g_out, as_stream(stream));
}

int uml_sum_partials(const float* partials, int32_t n_splits, int64_t split_stride, int64_t n, float* out,
                     void* stream) {
  using namespace uml;
  UML_REQUIRE(partials && out && n_splits >= 1 && n >= 0 && split_stride >= n, "sum_partials: bad arguments");
  UML_REQUIRE(n % 4 == 0 && split_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(partials) & 15u) == 0 &&
                  (reinterpret_cast<uintptr_t>(out) & 15u) == 0,
              "sum_partials: buffers must be 16B aligned and n a multiple of 4");
  if (n == 0) return 0;
  const int64_t n4 = n / 4;
  const int grid = static_cast<int>(std::min<int64_t>((n4 + 255) / 256, static_cast<int64_t>(sm_count()) * 8));
  sum_partials_kernel<<<grid, 256, 0, as_stream(stream)>>>(partials, n_splits, split_stride, n4, out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int uml_sgd_step(float* p, const float* g, const float* g2, float g2_weight, float* buf, int64_t n, double lr,
                 double momentum, double weight_decay, int64_t step, uint16_t* p_bf16, void* stream) {
  using namespace uml;
  UML_REQUIRE(p && g && buf && n >= 0 && step >= 1, "sgd_step: bad arguments");
  if (n == 0) return 0;
  const int grid = static_cast<int>(std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(sm_count()) * 8));
  sgd_kernel<<<grid, 256, 0, as_stream(stream)>>>(p, g, g2, g2_weight, buf, n, static_cast<float>(lr),
                                                  static_cast<float>(momentum), static_cast<float>(weight_decay),
                                                  step <= 1, reinterpret_cast<__nv_bfloat16*>(p_bf16));
  UML_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
