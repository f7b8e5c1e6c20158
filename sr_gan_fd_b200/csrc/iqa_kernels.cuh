// Next to the path (SURVEY.md section 8f rank 4): the evaluation epilogue the reference runs on every validated frame --
// PSNR / SSIM on the Y channel (ESRGAN/image_quality_assessment.py:361-541, via imgproc.rgb_to_ycbcr_torch :409-434) and the
// fp32 NCHW -> uint8 HWC image conversion (ESRGAN/imgproc.py:160-183).  The reference spends ~25 elementwise / grouped-conv
// launches with fp64 full-frame temporaries per metric; here each metric is ONE pass over the two images: crop, RGB -> Y
// (fp32, as the reference's fp32 matmul), then fp64 arithmetic as in the reference.  HBM-bound: 24 B read per pixel.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace b200sr {

struct IqaParams {
  const float* raw;  // [N, 3, H, W] RGB in [0, 1]
  const float* dst;
  int N, H, W, crop;
  double win[11];    // 1-D gaussian (the 2-D window is its outer product)
  double* psnr_sum;  // [N] sum over the cropped frame of (255 Yr - 255 Yd)^2
  double* ssim_sum;  // [N] sum of the SSIM map (valid 11 x 11 windows of the cropped frame)
};

__device__ __forceinline__ float iqa_y(const float* img, long long plane, long long i) {
  // imgproc.py:423-432: matmul([R G B], [65.481 128.553 24.966]) + 16, then / 255 -- all in fp32
  const float y = img[i] * 65.481f + img[i + plane] * 128.553f + img[i + 2 * plane] * 24.966f + 16.0f;
  return y / 255.0f;
}

__device__ __forceinline__ double iqa_block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = (threadIdx.y * blockDim.x + threadIdx.x) >> 5, lane = (threadIdx.y * blockDim.x + threadIdx.x) & 31;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (warp == 0) {
    const int nw = (blockDim.x * blockDim.y + 31) >> 5;
    s = lane < nw ? red[lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  }
  return s;  // valid in thread 0
}

// grid (blocks, N), block (256, 1).  kDet: psnr_sum is a [blocks][N] partial-sum matrix (ordered_sum_kernel adds the rows)
template <bool kDet>
__global__ void __launch_bounds__(256) iqa_psnr_y_kernel(const IqaParams p) {
  __shared__ double red[8];
  const int n = blockIdx.y;
  const int hc = p.H - 2 * p.crop, wc = p.W - 2 * p.crop;
  const long long plane = static_cast<long long>(p.H) * p.W;
  const float* r = p.raw + static_cast<long long>(n) * 3 * plane;
  const float* d = p.dst + static_cast<long long>(n) * 3 * plane;
  double acc = 0.0;
  const long long total = static_cast<long long>(hc) * wc;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int y = static_cast<int>(i / wc), x = static_cast<int>(i - static_cast<long long>(y) * wc);
    const long long idx = static_cast<long long>(y + p.crop) * p.W + (x + p.crop);
    const double e = static_cast<double>(iqa_y(r, plane, idx)) * 255.0 - static_cast<double>(iqa_y(d, plane, idx)) * 255.0;
    acc += e * e;
  }
  const double s = iqa_block_sum(acc, red);
  if (threadIdx.x == 0) {
    if constexpr (kDet) p.psnr_sum[static_cast<long long>(blockIdx.x) * p.N + n] = s;
    else atomicAdd(p.psnr_sum + n, s);
  }
}

// grid (ceil(Wo / 16), ceil(Ho / 16), N), block (16, 16); Wo = W - 2 crop - 10.  kDet: ssim_sum is a [blocks][N] partial-sum
// matrix, block = blockIdx.y * gridDim.x + blockIdx.x
template <bool kDet>
__global__ void __launch_bounds__(256) iqa_ssim_y_kernel(const IqaParams p) {
  __shared__ double yr[26][26], yd[26][26];
  __shared__ double hq[5][26][16];
  __shared__ double red[8];
  const int n = blockIdx.z;
  const int hc = p.H - 2 * p.crop, wc = p.W - 2 * p.crop;
  const int ho = hc - 10, wo = wc - 10;
  const int ox = blockIdx.x * 16, oy = blockIdx.y * 16;
  const long long plane = static_cast<long long>(p.H) * p.W;
  const float* r = p.raw + static_cast<long long>(n) * 3 * plane;
  const float* d = p.dst + static_cast<long long>(n) * 3 * plane;
  const int t = threadIdx.y * 16 + threadIdx.x;
  for (int i = t; i < 26 * 26; i += 256) {
    const int ly = i / 26, lx = i - ly * 26;
    const int y = oy + ly, x = ox + lx;  // cropped-frame coordinates
    double a = 0.0, b = 0.0;
    if (y < hc && x < wc) {
      const long long idx = static_cast<long long>(y + p.crop) * p.W + (x + p.crop);
      a = static_cast<double>(iqa_y(r, plane, idx)) * 255.0;
      b = static_cast<double>(iqa_y(d, plane, idx)) * 255.0;
    }
    yr[ly][lx] = a; yd[ly][lx] = b;
  }
  __syncthreads();
  for (int i = t; i < 26 * 16; i += 256) {  // horizontal pass
    const int ly = i >> 4, lx = i & 15;
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const double w = p.win[k], a = yr[ly][lx + k], b = yd[ly][lx + k];
      s0 += w * a; s1 += w * b; s2 += w * (a * a); s3 += w * (b * b); s4 += w * (a * b);
    }
    hq[0][ly][lx] = s0; hq[1][ly][lx] = s1; hq[2][ly][lx] = s2; hq[3][ly][lx] = s3; hq[4][ly][lx] = s4;
  }
  __syncthreads();
  double val = 0.0;
  if (ox + threadIdx.x < wo && oy + threadIdx.y < ho) {  // vertical pass + SSIM map value
    double m_r = 0, m_d = 0, e_rr = 0, e_dd = 0, e_rd = 0;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const double w = p.win[k];
      m_r += w * hq[0][threadIdx.y + k][threadIdx.x]; m_d += w * hq[1][threadIdx.y + k][threadIdx.x];
      e_rr += w * hq[2][threadIdx.y + k][threadIdx.x]; e_dd += w * hq[3][threadIdx.y + k][threadIdx.x];
      e_rd += w * hq[4][threadIdx.y + k][threadIdx.x];
    }
    const double c1 = (0.01 * 255.0) * (0.01 * 255.0), c2 = (0.03 * 255.0) * (0.03 * 255.0);
    const double v_r = e_rr - m_r * m_r, v_d = e_dd - m_d * m_d, cov = e_rd - m_r * m_d;
    val = ((2 * m_r * m_d + c1) * (2 * cov + c2)) / ((m_r * m_r + m_d * m_d + c1) * (v_r + v_d + c2));
  }
  const double s = iqa_block_sum(val, red);
  if (t == 0) {
    if constexpr (kDet) p.ssim_sum[(static_cast<long long>(blockIdx.y) * gridDim.x + blockIdx.x) * p.N + n] = s;
    else atomicAdd(p.ssim_sum + n, s);
  }
}

// x: [C, H, W] fp32 (C <= 4) -> out [H, W, C] uint8 = trunc(clamp(255 x, 0, 255)); half: round to fp16 and multiply in fp16 first
__global__ void tensor_to_image_u8_kernel(const float* __restrict__ x, int C, int H, int W, int range_norm, int half, uint8_t* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long plane = static_cast<long long>(H) * W;
  if (i >= plane) return;
  for (int c = 0; c < C; ++c) {
    float v = x[c * plane + i];
    if (range_norm) v = (v + 1.0f) / 2.0f;
    if (half) v = __half2float(__hmul(__float2half(v), __float2half(255.0f)));
    else v = v * 255.0f;
    v = fminf(fmaxf(v, 0.f), 255.f);
    out[i * C + c] = static_cast<uint8_t>(v);  // numpy astype("uint8") truncates
  }
}

}  // namespace b200sr
