// Helpers of the VGG19 feature path (SURVEY.md section 8f rank 3: the perceptual "content" loss, ESRGAN/model.py:246-292,
// BSRGAN/model.py:501-554).  The sixteen 3x3 convs run on conv3x3_chain_kernel; these HBM-bound kernels do the rest:
// input normalisation + hi/lo split, 2x2 max-pool forward / backward on NHWC bf16, and the L1 feature loss and its gradient.
#pragma once
#include "ptx.cuh"

namespace b200sr {

struct VggNorm { float mean[4]; float std[4]; };

// x: [N, 3, H, W] fp32 (element strides) -> [N*H*W, 64] bf16 = [hi(3) | lo(3) | hi(3) | 0...] of (x - mean) / std
// (transforms.Normalize, ESRGAN/model.py:275,283-284; the first conv's weights are packed [w_hi | w_hi | w_lo])
__global__ void vgg_ingest_kernel(const float* __restrict__ x, long long sn, long long sc, long long sh, long long sw, int N, int H, int W,
                                  const VggNorm nm, __nv_bfloat16* __restrict__ out) {
  const long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (pix >= static_cast<long long>(N) * H * W) return;
  const int xw = static_cast<int>(pix % W);
  const int yh = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  float hi[3], lo[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = (x[n * sn + c * sc + yh * sh + xw * sw] - nm.mean[c]) / nm.std[c];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[c] = __bfloat162float(h);
    lo[c] = v - hi[c];
  }
  uint4* o = reinterpret_cast<uint4*>(out + pix * 64);
  o[0] = make_uint4(pack_bf16x2(hi[0], hi[1]), pack_bf16x2(hi[2], lo[0]), pack_bf16x2(lo[1], lo[2]), pack_bf16x2(hi[0], hi[1]));
  o[1] = make_uint4(pack_bf16x2(hi[2], 0.f), 0u, 0u, 0u);
#pragma unroll
  for (int k = 2; k < 8; ++k) o[k] = make_uint4(0u, 0u, 0u, 0u);
}

__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b) {
  __nv_bfloat162 x = *reinterpret_cast<__nv_bfloat162*>(&a), y = *reinterpret_cast<__nv_bfloat162*>(&b);
  __nv_bfloat162 m = __hmax2(x, y);
  return *reinterpret_cast<uint32_t*>(&m);
}

// in: [N, H, W, C] bf16 -> out: [N, H/2, W/2, C] (MaxPool2d(2, 2), floor); one thread per output pixel and 8 channels
__global__ void vgg_maxpool_kernel(const __nv_bfloat16* __restrict__ in, __nv_bfloat16* __restrict__ out, int N, int H, int W, int C) {
  const int c8 = C >> 3;
  const int Ho = H >> 1, Wo = W >> 1;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(N) * Ho * Wo * c8) return;
  const int cc = static_cast<int>(i % c8);
  const long long op = i / c8;
  const int xo = static_cast<int>(op % Wo), yo = static_cast<int>((op / Wo) % Ho), n = static_cast<int>(op / (static_cast<long long>(Wo) * Ho));
  const uint4* p00 = reinterpret_cast<const uint4*>(in + ((static_cast<long long>(n) * H + 2 * yo) * W + 2 * xo) * C) + cc;
  const uint4 a = p00[0], b = p00[c8], c = p00[static_cast<long long>(W) * c8], d = p00[static_cast<long long>(W) * c8 + c8];
  uint4 m;
  m.x = bf16x2_max(bf16x2_max(a.x, b.x), bf16x2_max(c.x, d.x));
  m.y = bf16x2_max(bf16x2_max(a.y, b.y), bf16x2_max(c.y, d.y));
  m.z = bf16x2_max(bf16x2_max(a.z, b.z), bf16x2_max(c.z, d.z));
  m.w = bf16x2_max(bf16x2_max(a.w, b.w), bf16x2_max(c.w, d.w));
  reinterpret_cast<uint4*>(out + op * C)[cc] = m;
}

// Backward of ReLU -> MaxPool2d(2, 2): act [N, H, W, C] = the pooled layer's input (post-ReLU), gout [N, H/2, W/2, C] the gradient of
// the pooled output; gin [N, H, W, C] = gradient w.r.t. the conv output BEFORE the ReLU: the window's first maximum (row-major, as
// torch's max_pool2d backward) receives gout if its activation is positive (ReLU'), everything else 0.  Rows / columns the floor
// pooling drops (odd H / W) get 0.  One thread per pooled pixel and channel pair.
__global__ void vgg_maxpool_relu_bwd_kernel(const __nv_bfloat16* __restrict__ act, const __nv_bfloat16* __restrict__ gout,
                                            __nv_bfloat16* __restrict__ gin, int N, int H, int W, int C) {
  const int c2 = C >> 1;
  const int Ho = (H + 1) >> 1, Wo = (W + 1) >> 1;  // covers the dropped last row / column too
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(N) * Ho * Wo * c2) return;
  const int cc = static_cast<int>(i % c2);
  const long long op = i / c2;
  const int xo = static_cast<int>(op % Wo), yo = static_cast<int>((op / Wo) % Ho), n = static_cast<int>(op / (static_cast<long long>(Wo) * Ho));
  const bool full = (2 * yo + 1 < H) && (2 * xo + 1 < W);
  float g0 = 0.f, g1 = 0.f;
  if (full) {
    const float2 g = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(gout + ((static_cast<long long>(n) * (H >> 1) + yo) * (W >> 1) + xo) * C)[cc]);
    g0 = g.x; g1 = g.y;
  }
  float2 a[4];
  long long idx[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int y = 2 * yo + (k >> 1), x = 2 * xo + (k & 1);
    idx[k] = -1;
    a[k] = make_float2(-1.f, -1.f);
    if (y < H && x < W) {
      idx[k] = ((static_cast<long long>(n) * H + y) * W + x) * C;
      a[k] = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(act + idx[k])[cc]);
    }
  }
  int w0 = 0, w1 = 0;
#pragma unroll
  for (int k = 1; k < 4; ++k) {
    if (a[k].x > a[w0].x) w0 = k;
    if (a[k].y > a[w1].y) w1 = k;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (idx[k] < 0) continue;
    const float o0 = (full && k == w0 && a[k].x > 0.f) ? g0 : 0.f;
    const float o1 = (full && k == w1 && a[k].y > 0.f) ? g1 : 0.f;
    reinterpret_cast<uint32_t*>(gin + idx[k])[cc] = pack_bf16x2(o0, o1);
  }
}

constexpr int kVggL1MaxBlocks = 8 * 148;  // grid cap of vgg_l1_pair_sum_kernel (a constant: the grid depends on the shape only)

// sum over the first `half` elements of |f[i] - f[i + half]| (fp32 features of the sr images followed by those of the gt images).
// kDet: out[blockIdx.x] = this block's partial sum (ordered_sum_kernel adds them) instead of an atomicAdd into out[0]
template <bool kDet>
__global__ void __launch_bounds__(256) vgg_l1_pair_sum_kernel(const float* __restrict__ f, long long half, double* __restrict__ out) {
  __shared__ double red[8];
  double acc = 0.0;
  for (long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < half; i += static_cast<long long>(gridDim.x) * blockDim.x * 4) {
    const float4 a = *reinterpret_cast<const float4*>(f + i), b = *reinterpret_cast<const float4*>(f + half + i);
    acc += static_cast<double>(fabsf(a.x - b.x)) + static_cast<double>(fabsf(a.y - b.y)) + static_cast<double>(fabsf(a.z - b.z)) +
           static_cast<double>(fabsf(a.w - b.w));
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    double s = red[threadIdx.x];
    for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffu, s, o);
    if (threadIdx.x == 0) {
      if constexpr (kDet) out[blockIdx.x] = s;
      else atomicAdd(out, s);
    }
  }
}

// g[i] = bf16(sign(f[i] - f[i + half]) * scale[0] / half): gradient of mean |f_sr - f_gt| w.r.t. f_sr times the upstream gradient.
// g is the gradient w.r.t. the conv's PRE-activation output.  post_relu: f holds max(pre, 0) (a feature node before the last conv),
// so the ReLU derivative [f_sr > 0] -- equal to [pre > 0], f being fmaxf(pre, 0) in fp32 -- multiplies the sign.
__global__ void vgg_l1_grad_kernel(const float* __restrict__ f, long long half, const float* __restrict__ scale, int post_relu,
                                   __nv_bfloat16* __restrict__ g) {
  const long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= half) return;
  const float s = scale[0] / static_cast<float>(half);
  const float4 a = *reinterpret_cast<const float4*>(f + i), b = *reinterpret_cast<const float4*>(f + half + i);
  auto sg = [&](float fs, float fg) {
    if (post_relu && !(fs > 0.f)) return 0.f;
    const float d = fs - fg;
    return d > 0.f ? s : (d < 0.f ? -s : 0.f);
  };
  uint2 o;
  o.x = pack_bf16x2(sg(a.x, b.x), sg(a.y, b.y));
  o.y = pack_bf16x2(sg(a.z, b.z), sg(a.w, b.w));
  *reinterpret_cast<uint2*>(g + i) = o;
}

}  // namespace b200sr
