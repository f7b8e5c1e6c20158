// Fused optimizer step for the generator's parameter list (SURVEY.md section 8f, rank 1): GradScaler unscale + non-finite
// skip + Adam (torch.optim.Adam semantics, L2 weight decay) + the reference's EMA rule
//   ema <- (1 - d) * ema + d * p        (ESRGAN/train_rrdbnet.py:182, AveragedModel avg_fn; first update copies p)
// in ONE multi-tensor launch.  HBM-bound: 5 fp32 reads + 4 fp32 writes per parameter (36 B).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace b200sr {

struct OptTensor {       // one parameter tensor
  float* p;
  const float* g;         // nullptr: a frozen parameter (no gradient) -- no Adam update, the EMA still averages it
  float* m;
  float* v;
  float* ema;            // may be nullptr
  long long numel;
  long long block0;      // first 1024-element block of this tensor in the launch
};

struct AdamEmaHyper {
  float lr, beta1, beta2, eps, weight_decay;
  float ema_decay;                     // d above
  int ema_copy;                        // 1: first EMA update (copy)
  const float* grad_scale;             // device scalar or nullptr: gradients are divided by it
  const float* found_inf;              // device scalar or nullptr: > 0 -> Adam is skipped (GradScaler), the EMA still updates
  const float* step;                   // device scalar: number of Adam steps taken so far (this launch computes step + 1)
  const int* block_tensor;             // block -> tensor index
};

constexpr int kOptBlock = 256;
constexpr int kOptElemsPerBlock = 1024;

__global__ void __launch_bounds__(kOptBlock) fused_adam_ema_kernel(const OptTensor* __restrict__ tensors, int n_tensors,
                                                                   const AdamEmaHyper h) {
  const bool skip = h.found_inf && *h.found_inf > 0.f;
  const long long b = blockIdx.x;
  const OptTensor t = tensors[h.block_tensor[b]];
  const bool no_adam = skip || !t.g;
  if (no_adam && !t.ema) return;
  const float tstep = *h.step + 1.f;
  const float bias_corr1 = 1.f - powf(h.beta1, tstep);
  const float bias_corr2_sqrt = sqrtf(1.f - powf(h.beta2, tstep));
  const float inv_scale = h.grad_scale ? 1.f / *h.grad_scale : 1.f;
  const long long base = (b - t.block0) * kOptElemsPerBlock;
  const float step_size = h.lr / bias_corr1;
  auto upd = [&](float& p, float g, float& m, float& v, float& e) {
    if (!no_adam) {
      g *= inv_scale;
      if (h.weight_decay != 0.f) g = fmaf(h.weight_decay, p, g);
      m = fmaf(h.beta1, m, (1.f - h.beta1) * g);
      v = fmaf(h.beta2, v, (1.f - h.beta2) * g * g);
      p = p - step_size * (m / (sqrtf(v) / bias_corr2_sqrt + h.eps));
    }
    e = h.ema_copy ? p : fmaf(h.ema_decay, p, (1.f - h.ema_decay) * e);
  };
  const long long i0 = base + 4LL * threadIdx.x;  // 256 threads x 4 consecutive elements = one 1024-element block
  const bool vec = ((reinterpret_cast<uintptr_t>(t.p) | reinterpret_cast<uintptr_t>(t.g) | reinterpret_cast<uintptr_t>(t.m) |
                     reinterpret_cast<uintptr_t>(t.v) | reinterpret_cast<uintptr_t>(t.ema)) & 15) == 0;
  if (vec && i0 + 3 < t.numel) {
    float4 p = *reinterpret_cast<const float4*>(t.p + i0);
    const float4 g = t.g ? *reinterpret_cast<const float4*>(t.g + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 m = *reinterpret_cast<const float4*>(t.m + i0);
    float4 v = *reinterpret_cast<const float4*>(t.v + i0);
    float4 e = t.ema ? *reinterpret_cast<const float4*>(t.ema + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
    upd(p.x, g.x, m.x, v.x, e.x); upd(p.y, g.y, m.y, v.y, e.y); upd(p.z, g.z, m.z, v.z, e.z); upd(p.w, g.w, m.w, v.w, e.w);
    *reinterpret_cast<float4*>(t.p + i0) = p;
    *reinterpret_cast<float4*>(t.m + i0) = m;
    *reinterpret_cast<float4*>(t.v + i0) = v;
    if (t.ema) *reinterpret_cast<float4*>(t.ema + i0) = e;
  } else {
    for (long long i = i0; i < i0 + 4 && i < t.numel; ++i) {
      float p = t.p[i], m = t.m[i], v = t.v[i], e = t.ema ? t.ema[i] : 0.f;
      upd(p, t.g ? t.g[i] : 0.f, m, v, e);
      t.p[i] = p; t.m[i] = m; t.v[i] = v;
      if (t.ema) t.ema[i] = e;
    }
  }
}

// step += 1 unless the step was skipped (runs after the update kernel on the same stream)
__global__ void adam_step_advance_kernel(float* step, const float* found_inf) {
  if (!(found_inf && *found_inf > 0.f)) *step += 1.f;
}

}  // namespace b200sr
