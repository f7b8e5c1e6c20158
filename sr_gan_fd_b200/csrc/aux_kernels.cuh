// Bandwidth-bound helper kernels around the tcgen05 convs: weight re-packing (fp32 OIHW master -> bf16 K-major
// tap-major tiles, incl. the dgrad transpose/flip, the hi/lo split and the nearest-upsample phase folding),
// input/output layout conversion, bias gradients, and the fold of phase weight-gradients back to 3x3.
#pragma once
#include "ptx.cuh"

namespace b200sr {

// ------------------------------------------------------------------------------------------------ weight packing
enum PackMode : int {
  kPackFwd = 0,      // elem(n, k, ty, tx) = W[o_off + n][i_off + k][ty][tx]
  kPackDgrad = 1,    // elem(n, k, ty, tx) = W[o_off + k][i_off + n][2-ty][2-tx]
  kPackUpFwd = 2,    // n = phase*64 + co: sum of the taps of W[co][k] that fold onto LR tap (ty,tx) for that phase
  kPackUpDgrad = 3,  // k = phase*64 + co, n = ci: transposed + flipped version of kPackUpFwd
  // 4x4 stride-2 pad-1 conv (U-Net discriminator, BSRGAN/model.py:103-114) as a 3x3 conv over the pixel-unshuffled input
  // (channel (py*2+px)*I + c of the half-resolution lattice): kernel position (ky, kx) = (2 ty + py - 1, 2 tx + px - 1)
  kPackDownFwd = 4,   // elem(n, k = phase*I + c, ty, tx) = W[n][c][ky][kx] (0 where ky / kx fall outside 0..3); W is [O][I][4][4]
  kPackDownDgrad = 5  // elem(n = phase*I + c, k = co, ty, tx) = kPackDownFwd elem(co, n, 2-ty, 2-tx)
};

struct PackSeg {
  int n0, nlen;   // packed output-column range [n0, n0 + nlen) served by this segment (nlen = 0: all columns)
  int k0, klen;   // packed K-channel range [k0, k0 + klen) served by this segment
  int w_index;    // index into the parameter pointer table
  int O, I;       // source tensor dims (OIHW)
  int o_off, i_off;
  int part;       // 0: bf16(w)   1: bf16(w - bf16(w))   (hi / lo split)
};

struct PackOp {
  int row0;        // first packed row
  int n_total;     // output columns of the conv (= n_cols * column groups)
  int n_cols;      // columns per column group (rows per tap tile)
  int n_valid;     // output columns >= n_valid are zero
  int num_chunks;  // 64-channel K chunks
  int mode;
  int nseg;
  int k32;         // 1: a single K chunk of 32 channels, packed as 64-byte rows under the 64B swizzle (half the bytes of a padded 128-byte row)
  int f16;         // 1: packed as fp16 (U-Net discriminator plans in the reference's autocast format) instead of bf16
  int down_c;      // > 0 (modes kPackDownFwd / kPackDownDgrad): channels of one unshuffle phase; only the FOUR non-zero tap tiles of every
                   // (chunk, column group) are packed, rows [chunk][column group][tap 0..3][n] (see ConvParams::down_mode)
  PackSeg seg[5];
};

// nearest-x2 upsample followed by a 3x3 conv == four phase convs on the LOW-RES grid.  For output phase a (0/1)
// and low-res tap t (0,1,2 <-> offset -1,0,+1) the contributing original taps d are [lo, hi):
//   a = 0: t=0 <- {0}, t=1 <- {1,2}, t=2 <- {}        a = 1: t=0 <- {}, t=1 <- {0,1}, t=2 <- {2}
__host__ __device__ inline void up_phase_taps(int a, int t, int& lo, int& hi) {
  if (a == 0) { lo = (t == 0) ? 0 : (t == 1 ? 1 : 0); hi = (t == 0) ? 1 : (t == 1 ? 3 : 0); }
  else        { lo = (t == 0) ? 0 : (t == 1 ? 0 : 2); hi = (t == 0) ? 0 : (t == 1 ? 2 : 3); }
}

__device__ __forceinline__ float pack_fetch(const PackOp& op, const float* const* params, int n_in, int k, int ty, int tx) {
  if (n_in >= op.n_valid) return 0.f;
  for (int s = 0; s < op.nseg; ++s) {
    const PackSeg& sg = op.seg[s];
    int n = n_in;
    const int kl = k - sg.k0;
    if (kl < 0 || kl >= sg.klen) continue;
    if (sg.nlen > 0) {
      if (n < sg.n0 || n >= sg.n0 + sg.nlen) continue;
      n -= sg.n0;
    }
    const float* w = params[sg.w_index];
    float v = 0.f;
    if (op.mode == kPackFwd) {
      v = w[((static_cast<long long>(sg.o_off + n) * sg.I + sg.i_off + kl) * 3 + ty) * 3 + tx];
    } else if (op.mode == kPackDgrad) {
      v = w[((static_cast<long long>(sg.o_off + kl) * sg.I + sg.i_off + n) * 3 + (2 - ty)) * 3 + (2 - tx)];
    } else if (op.mode == kPackDownFwd || op.mode == kPackDownDgrad) {
      int co, cu, ry, rx;
      if (op.mode == kPackDownFwd) { co = n; cu = kl; ry = ty; rx = tx; }
      else                         { co = kl; cu = n; ry = 2 - ty; rx = 2 - tx; }
      const int phase = cu / sg.I, c = cu - phase * sg.I;
      const int ky = 2 * ry + (phase >> 1) - 1, kx = 2 * rx + (phase & 1) - 1;
      if (phase < 4 && ky >= 0 && ky < 4 && kx >= 0 && kx < 4)
        v = w[((static_cast<long long>(sg.o_off + co) * sg.I + sg.i_off + c) * 4 + ky) * 4 + kx];
    } else {
      int phase, co, ci, ry, rx;
      if (op.mode == kPackUpFwd) { phase = n >> 6; co = n & 63; ci = kl; ry = ty; rx = tx; }
      else                       { phase = kl >> 6; co = kl & 63; ci = n; ry = 2 - ty; rx = 2 - tx; }
      int ylo, yhi, xlo, xhi;
      up_phase_taps(phase >> 1, ry, ylo, yhi);
      up_phase_taps(phase & 1, rx, xlo, xhi);
      const float* wp = w + (static_cast<long long>(sg.o_off + co) * sg.I + sg.i_off + ci) * 9;
      for (int dy = ylo; dy < yhi; ++dy)
        for (int dx = xlo; dx < xhi; ++dx) v += wp[dy * 3 + dx];
    }
    if (sg.part == 1) v = v - (op.f16 ? __half2float(__float2half_rn(v)) : __bfloat162float(__float2bfloat16_rn(v)));
    return v;
  }
  return 0.f;
}

// One thread per packed element.  Row layout inside an op: [chunk][column group][dx][dy][n in group], 64 K-channels
// (128 B) per row.  The rows are stored PRE-SWIZZLED: 16-byte chunk j of a row lands at position j ^ (n & 7), i.e. the
// image is byte-for-byte what a 128B-swizzled TMA load would have produced in shared memory, so the kernels fetch a
// whole chunk's nine tap tiles with ONE linear bulk copy (cp.async.bulk) instead of nine tensor-map boxes.
__global__ void pack_weights_kernel(const PackOp* __restrict__ ops, int num_ops, const float* const* __restrict__ params,
                                    __nv_bfloat16* __restrict__ packed, long long total_rows) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long row = idx >> 6;
  const int kk = static_cast<int>(idx & 63);
  if (row >= total_rows) return;
  int lo = 0, hi = num_ops - 1;  // last op with row0 <= row
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (ops[mid].row0 <= row) lo = mid; else hi = mid - 1;
  }
  const PackOp& op = ops[lo];
  if (op.k32) {
    // two 64-byte rows per 128-byte unit; 16-byte chunk j of row n lands at position j ^ ((n >> 1) & 3) (64B swizzle on address bits 7-8)
    const int r2 = static_cast<int>(row - op.row0) * 2 + (kk >> 5);
    const int kc = kk & 31;
    const int ng2 = r2 % op.n_cols, t2 = r2 / op.n_cols;
    const int cgs2 = op.n_total / op.n_cols;
    const int dy2 = t2 % 3, dx2 = (t2 / 3) % 3, cg2 = (t2 / 9) % cgs2, c2 = t2 / (9 * cgs2);
    const float v2 = (c2 < op.num_chunks) ? pack_fetch(op, params, cg2 * op.n_cols + ng2, c2 * 64 + kc, dy2, dx2) : 0.f;
    packed[op.row0 * 64LL + static_cast<long long>(r2) * 32 + (((kc >> 3) ^ ((ng2 >> 1) & 3)) * 8) + (kc & 7)] = __float2bfloat16_rn(v2);
    return;
  }
  const int r = static_cast<int>(row - op.row0);
  const int ng = r % op.n_cols;          // row inside the tap tile
  const int t = r / op.n_cols;           // ((chunk*CG + cg)*3 + dx)*3 + dy
  const int cgs = op.n_total / op.n_cols;
  int dy, dx, cg, c;
  if (op.down_c > 0) {
    // four tap tiles per (chunk, column group): tile i = (row i >> 1, column i & 1) of the 2 x 2 non-zero block, which starts at
    // row / column 1 (selector 0) or 0 (selector 1); selector = phase bits (forward) or their complement (data gradient)
    const int i = t % 4;
    cg = (t / 4) % cgs; c = t / (4 * cgs);
    const int phase = (op.mode == kPackDownFwd) ? (c * 64) / op.down_c : (cg * op.n_cols) / op.down_c;
    const int sel = (op.mode == kPackDownFwd) ? phase : (phase ^ 3);
    dy = ((sel >> 1) ? 0 : 1) + (i >> 1);
    dx = ((sel & 1) ? 0 : 1) + (i & 1);
  } else {
    dy = t % 3; dx = (t / 3) % 3; cg = (t / 9) % cgs; c = t / (9 * cgs);
  }
  const int n = cg * op.n_cols + ng;
  float v = (c < op.num_chunks) ? pack_fetch(op, params, n, c * 64 + kk, dy, dx) : 0.f;
  const int chunk16 = (kk >> 3) ^ (ng & 7);
  if (op.f16) reinterpret_cast<__half*>(packed)[row * 64 + chunk16 * 8 + (kk & 7)] = __float2half_rn(v);
  else packed[row * 64 + chunk16 * 8 + (kk & 7)] = __float2bfloat16_rn(v);
}

// biases: flat fp32 copy (bias_index < 0 -> zeros)
struct BiasOp { int off; int n; int b_index; int n_valid; int rep; };  // rep: repeat period (phase convs reuse 64 biases)
__global__ void pack_bias_kernel(const BiasOp* __restrict__ ops, int num_ops, const float* const* __restrict__ params,
                                 float* __restrict__ out) {
  const int o = blockIdx.x;
  if (o >= num_ops) return;
  const BiasOp op = ops[o];
  for (int i = threadIdx.x; i < op.n; i += blockDim.x) {
    const int j = op.rep > 0 ? (i % op.rep) : i;
    out[op.off + i] = (op.b_index >= 0 && j < op.n_valid) ? params[op.b_index][j] : 0.f;
  }
}

// -------------------------------------------------------------------------------------------- input conversion
// x: [N, C, H, W] (any strides, fp32/fp16/bf16) -> [N*H*W, 64*chunks] bf16 with channels [hi(C) | lo(C) | hi(C) | 0..]
// (the conv1 weights are packed as [w_hi | w_hi | w_lo], giving ~fp32-accurate products from bf16 MMAs).
template <typename T>
__global__ void ingest_input_kernel(const T* __restrict__ x, long long sn, long long sc, long long sh, long long sw,
                                    int N, int C, int H, int W, __nv_bfloat16* __restrict__ out, int out_stride) {
  const long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(N) * H * W;
  if (pix >= total) return;
  const int xw = static_cast<int>(pix % W);
  const int yh = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  __nv_bfloat16* o = out + pix * out_stride;
  for (int c = 0; c < C; ++c) {
    const float v = static_cast<float>(x[n * sn + c * sc + yh * sh + xw * sw]);
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    o[c] = h;
    o[C + c] = l;
    o[2 * C + c] = h;
  }
  for (int c = 3 * C; c < out_stride; ++c) o[c] = __float2bfloat16_rn(0.f);
}

// dy: [N, C, H, W] fp32 contiguous (gradient of the generator output) -> [N*H*W, 64] bf16, channels >= C zero.  kMasked (clamped
// plans): multiplied by the clamp pass-through mask recorded in the forward; otherwise (unclamped plans) mask is unused.
template <bool kMasked>
__global__ void ingest_grad_kernel(const float* __restrict__ dy, const unsigned char* __restrict__ mask, int N, int C,
                                   int H, int W, __nv_bfloat16* __restrict__ out, int out_stride) {
  const long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long plane = static_cast<long long>(H) * W;
  const long long total = static_cast<long long>(N) * plane;
  if (pix >= total) return;
  const long long n = pix / plane;
  const long long r = pix - n * plane;
  float v[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) {
    v[c] = 0.f;
    if (c < C) {
      const long long i = (n * C + c) * plane + r;
      v[c] = (!kMasked || mask[i]) ? dy[i] : 0.f;
    }
  }
  // 16 channels = 32 bytes per pixel: two 16-byte stores (out_stride is a multiple of 8 channels)
  uint4* o = reinterpret_cast<uint4*>(out + pix * out_stride);
  o[0] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  o[1] = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
}

// ------------------------------------------------------------------------------------------------ bias gradients
// db[c] += sum over pixels of g[pixel][c0 + c] for c in [0, ncols).  g is bf16 (or fp16) [P][stride]; ncols, c0 and stride are
// multiples of 8 and g is 16-byte aligned.  Each thread owns EIGHT consecutive channels of a pixel row (one 16-byte load, four of
// them in flight); pixel lanes are reduced through shared memory, one atomicAdd per channel and block.  The launch uses at most two
// blocks per SM: those final atomics all hit the SAME few addresses and cost ~45 ns each once a thousand blocks queue up on one.
// kDet (deterministic plans): seg[0].out is a [gridDim.x][ncols] partial-sum matrix instead; every block stores its row and
// ordered_sum_kernel adds the rows in block order.
struct BiasGradSeg { int col_begin, col_end; float* out; int n_valid; };
struct BiasGradParams { const __nv_bfloat16* g; long long P; int stride; int c0; int ncols; int nseg; BiasGradSeg seg[5]; int f16; };
constexpr int kBiasGradThreads = 256;

template <bool kDet>
__global__ void __launch_bounds__(kBiasGradThreads) bias_grad_vec_kernel(const BiasGradParams p) {
  __shared__ float red[8 * kBiasGradThreads];
  const int L = p.ncols >> 3;                 // 8-channel lanes per pixel row
  const int PL = kBiasGradThreads / L;        // pixel lanes per block
  const int cl = threadIdx.x % L;
  const int pl = threadIdx.x / L;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  const bool hf = p.f16 != 0;
  auto add8 = [&](const uint4& w) {
    const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (hf) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&ww[j]));
        acc[2 * j] += f.x; acc[2 * j + 1] += f.y;
      } else {
        acc[2 * j] += __uint_as_float(ww[j] << 16); acc[2 * j + 1] += __uint_as_float(ww[j] & 0xFFFF0000u);
      }
    }
  };
  if (pl < PL) {
    const uint4* base = reinterpret_cast<const uint4*>(p.g + p.c0) + cl;
    const long long step = static_cast<long long>(gridDim.x) * PL;
    const long long sp = p.stride >> 3;
    long long px = static_cast<long long>(blockIdx.x) * PL + pl;
    for (; px + 3 * step < p.P; px += 4 * step) {
      const uint4 v0 = __ldg(base + px * sp);
      const uint4 v1 = __ldg(base + (px + step) * sp);
      const uint4 v2 = __ldg(base + (px + 2 * step) * sp);
      const uint4 v3 = __ldg(base + (px + 3 * step) * sp);
      add8(v0); add8(v1); add8(v2); add8(v3);
    }
    for (; px < p.P; px += step) add8(__ldg(base + px * sp));
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) red[k * kBiasGradThreads + threadIdx.x] = acc[k];
  __syncthreads();
  if (pl == 0) {
    for (int i = 1; i < PL; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += red[k * kBiasGradThreads + i * L + cl];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = 8 * cl + k;
      if constexpr (kDet) {
        p.seg[0].out[static_cast<long long>(blockIdx.x) * p.ncols + c] = acc[k];
      } else {
        for (int sgi = 0; sgi < p.nseg; ++sgi) {
          const BiasGradSeg& sg = p.seg[sgi];
          if (c >= sg.col_begin && c < sg.col_end && (c - sg.col_begin) < sg.n_valid) atomicAdd(sg.out + (c - sg.col_begin), acc[k]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------ ordered sums (deterministic plans)
// Every per-split / per-block partial a deterministic plan's reductions leave behind is summed here, in index order, so the
// result does not depend on which CTA finished first.  One job, over a box of elements (i0 < n0, i1 < n1, i2 < n2, i3 < n3):
//   dst[i0 + i1 d1 + i2 d2 + i3 d3] = sum over s < S, in order, of src[s * stride + i0 + i1 s1 + i2 s2 + i3 s3]
// The weight-gradient jobs are boxes of [tap][co/4][ci][4] staging tensors (src: the compact copies of a pixel split); bias,
// VGG and IQA partials are rows (n0 only).
template <typename T>
struct SumJob {
  T* dst;
  const T* src;
  long long stride;  // between the S partials of an element
  int S, n0, n1, n2, n3;
  long long d1, d2, d3, s1, s2, s3;
};
constexpr int kMaxSumJobs = 24;
template <typename T>
struct SumJobs {
  int n;
  int block0[kMaxSumJobs + 1];  // blocks of job j: [block0[j], block0[j + 1])
  SumJob<T> job[kMaxSumJobs];
};

template <typename T>
__global__ void __launch_bounds__(256) ordered_sum_kernel(const __grid_constant__ SumJobs<T> J) {
  int j = 0;
  while (j + 1 < J.n && static_cast<int>(blockIdx.x) >= J.block0[j + 1]) ++j;
  const SumJob<T>& b = J.job[j];
  const unsigned total = static_cast<unsigned>(b.n0) * b.n1 * b.n2 * b.n3;
  const unsigned step = static_cast<unsigned>(J.block0[j + 1] - J.block0[j]) * blockDim.x;
  for (unsigned e = (blockIdx.x - J.block0[j]) * blockDim.x + threadIdx.x; e < total; e += step) {
    unsigned r = e;
    const unsigned i0 = r % b.n0; r /= b.n0;
    const unsigned i1 = r % b.n1; r /= b.n1;
    const unsigned i2 = r % b.n2, i3 = r / b.n2;
    const long long o = i0 + i1 * b.s1 + i2 * b.s2 + i3 * b.s3;
    T acc = b.src[o];
    for (int s = 1; s < b.S; ++s) acc += b.src[o + s * b.stride];
    b.dst[i0 + i1 * b.d1 + i2 * b.d2 + i3 * b.d3] = acc;
  }
}

// ------------------------------------------------------------ unpack staged weight gradients to the OIHW flat buffer
// src: [tap][co_pad/4][ci][4] fp32 staging tensor written by wgrad3x3_kernel;  dst: [co][ci][3][3] (state_dict layout).
// fold = 1: src holds the four low-res phase kernels of an upsample conv ([tap][ci][4*64]) and they are folded back
// onto the 3x3 taps of the original weight (see up_phase_taps).
struct UnpackOp { long long src_off; long long dst_off; int co, ci, co_pad, fold; int block0; int nblocks; };

__global__ void __launch_bounds__(256) unpack_wgrad_kernel(const UnpackOp* __restrict__ ops, int op_begin, int op_end,
                                                           const float* __restrict__ staging, float* __restrict__ grads) {
  // find the op this block works on (ops of one launch have consecutive block ranges starting at ops[op_begin].block0)
  const int b = blockIdx.x + ops[op_begin].block0;
  int lo = op_begin, hi = op_end - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (ops[mid].block0 <= b) lo = mid; else hi = mid - 1;
  }
  const UnpackOp op = ops[lo];
  // one block = 32 co x 32 ci tile, all 9 taps, staged through smem so both sides are coalesced
  __shared__ float tile[9][32][33];
  const int tiles_co = (op.co + 31) / 32;
  const int tb = b - op.block0;
  const int co0 = (tb % tiles_co) * 32, ci0 = (tb / tiles_co) * 32;
  const float* src = staging + op.src_off;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  if (!op.fold) {
    // staging layout [tap][co/4][ci][4]: one 16-byte load per thread and tap, consecutive threads -> consecutive ci (coalesced)
    const int ci = ci0 + tx, cq = (co0 >> 2) + ty;  // ty = 0..7: the tile's eight co quads
    for (int tap = 0; tap < 9; ++tap) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ci < op.ci && 4 * cq < op.co_pad)
        v = *reinterpret_cast<const float4*>(src + ((static_cast<long long>(tap) * (op.co_pad >> 2) + cq) * op.ci + ci) * 4);
      tile[tap][tx][4 * ty] = v.x; tile[tap][tx][4 * ty + 1] = v.y; tile[tap][tx][4 * ty + 2] = v.z; tile[tap][tx][4 * ty + 3] = v.w;
    }
  } else
  for (int tap = 0; tap < 9; ++tap) {
    for (int r = ty; r < 32; r += 8) {
      const int ci = ci0 + tx, co = co0 + r;  // consecutive threads -> consecutive ci (16-byte stride in the staging layout)
      float v = 0.f;
      if (ci < op.ci && co < op.co) {
        {
          const int dy = tap / 3, dx = tap % 3;
          for (int ph = 0; ph < 4; ++ph) {
            int ry = -1, rx = -1;
            for (int t = 0; t < 3; ++t) {
              int l, h;
              up_phase_taps(ph >> 1, t, l, h);
              if (dy >= l && dy < h) ry = t;
              up_phase_taps(ph & 1, t, l, h);
              if (dx >= l && dx < h) rx = t;
            }
            const int cc = ph * 64 + co;
            v += src[((static_cast<long long>(ry * 3 + rx) * (op.co_pad >> 2) + (cc >> 2)) * op.ci + ci) * 4 + (cc & 3)];
          }
        }
      }
      tile[tap][tx][r] = v;  // [ci][co]
    }
  }
  __syncthreads();
  float* dst = grads + op.dst_off;
  // write: for each co row of the tile, 32 ci x 9 taps contiguous floats
  for (int cr = ty; cr < 32; cr += 8) {
    const int co = co0 + cr;
    if (co >= op.co) continue;
    for (int e = tx; e < 32 * 9; e += 32) {
      const int ci = ci0 + e / 9, tap = e % 9;
      if (ci < op.ci) dst[(static_cast<long long>(co) * op.ci + ci) * 9 + tap] = tile[tap][e / 9][cr];
    }
  }
}

// out_bf16[pixel][64] = bf16(a + b) where a, b are fp32 carriers in the tile-blocked layout of the conv epilogues
// ([tile][half][16-byte chunk][pixel-in-half][4]); tiles are 8 x 32 pixels, halves 8 x 16.
__global__ void add_carriers_to_bf16_kernel(const float* __restrict__ a, const float* __restrict__ b, __nv_bfloat16* __restrict__ out,
                                            int N, int H, int W, int tiles_x, int tiles_y) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;  // ((tile*2+half)*16 + chunk)*128 + m
  const long long total = static_cast<long long>(N) * tiles_x * tiles_y * 2 * 16 * 128;
  if (idx >= total) return;
  const int m = static_cast<int>(idx & 127);
  const int chunk = static_cast<int>((idx >> 7) & 15);
  const int half = static_cast<int>((idx >> 11) & 1);
  const long long tile = idx >> 12;
  const int tpi = tiles_x * tiles_y;
  const int n = static_cast<int>(tile / tpi);
  const int t2 = static_cast<int>(tile - static_cast<long long>(n) * tpi);
  const int ty = t2 / tiles_x;
  const int x = (t2 - ty * tiles_x) * 8 + (m & 7);
  const int y = ty * 32 + half * 16 + (m >> 3);
  if (x >= W || y >= H) return;
  const float4 va = *reinterpret_cast<const float4*>(a + idx * 4);
  const float4 vb = *reinterpret_cast<const float4*>(b + idx * 4);
  __nv_bfloat16* o = out + ((static_cast<long long>(n) * H + y) * W + x) * 64 + chunk * 4;
  uint2 pk;
  pk.x = pack_bf16x2(va.x + vb.x, va.y + vb.y);
  pk.y = pack_bf16x2(va.z + vb.z, va.w + vb.w);
  *reinterpret_cast<uint2*>(o) = pk;
}

// ------------------------------------------------------------------------------------------------ trunk plans: both ends
// One thread per slot (tile, half, pixel m) of the tile-blocked carrier layout above, so that consecutive threads touch consecutive
// 16-byte carrier chunks (and, for NCHW tensors, consecutive x); padded slots outside the image are skipped -- the conv epilogues
// never read them.  Launch: one 256-thread block per 8 x 32 tile.
__device__ __forceinline__ bool trunk_slot(int N, int H, int W, int tiles_x, int tiles_y, long long& slot, int& n, int& y, int& x) {
  slot = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;  // (tile * 2 + half) * 128 + m
  const int m = static_cast<int>(slot & 127), half = static_cast<int>((slot >> 7) & 1);
  const long long tile = slot >> 8;
  const int tpi = tiles_x * tiles_y;
  n = static_cast<int>(tile / tpi);
  const int t2 = static_cast<int>(tile - static_cast<long long>(n) * tpi);
  const int ty = t2 / tiles_x;
  x = (t2 - ty * tiles_x) * 8 + (m & 7);
  y = ty * 32 + half * 16 + (m >> 3);
  return n < N && x < W && y < H;
}

// x: [N, 64, H, W], any strides, fp32 / fp16 / bf16 -> carrier (fp32, exact) and shadow[pixel][shadow_stride] channels [0, 64) =
// bf16(scale * x).  With scale 1 this is what conv1's epilogue leaves for the trunk (T0 / TR and D0), with scale 0.04 what conv2's
// data-gradient epilogue leaves (GR and dY5 of the last dense block).
template <typename T>
__global__ void __launch_bounds__(256) trunk_ingest_kernel(const T* __restrict__ x, long long sn, long long sc, long long sh, long long sw,
                                                           int N, int H, int W, int tiles_x, int tiles_y, float scale,
                                                           float* __restrict__ carrier, __nv_bfloat16* __restrict__ shadow, int shadow_stride) {
  long long slot;
  int n, y, xx;
  if (!trunk_slot(N, H, W, tiles_x, tiles_y, slot, n, y, xx)) return;
  const T* src = x + n * sn + y * sh + xx * sw;
  float4* cp = reinterpret_cast<float4*>(carrier) + (slot >> 7) * 16 * 128 + (slot & 127);
  uint4* sp = reinterpret_cast<uint4*>(shadow + ((static_cast<long long>(n) * H + y) * W + xx) * shadow_stride);
#pragma unroll
  for (int c8 = 0; c8 < 8; ++c8) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = static_cast<float>(src[(8 * c8 + k) * sc]);
    cp[(2 * c8) * 128] = make_float4(v[0], v[1], v[2], v[3]);
    cp[(2 * c8 + 1) * 128] = make_float4(v[4], v[5], v[6], v[7]);
    sp[c8] = make_uint4(pack_bf16x2(scale * v[0], scale * v[1]), pack_bf16x2(scale * v[2], scale * v[3]),
                        pack_bf16x2(scale * v[4], scale * v[5]), pack_bf16x2(scale * v[6], scale * v[7]));
  }
}

// carrier (fp32 tile-blocked) -> out [N, 64, H, W] fp32 contiguous: the trunk output y, or the trunk-input gradient dx
__global__ void __launch_bounds__(256) trunk_export_kernel(const float* __restrict__ carrier, float* __restrict__ out, int N, int H, int W,
                                                           int tiles_x, int tiles_y) {
  long long slot;
  int n, y, x;
  if (!trunk_slot(N, H, W, tiles_x, tiles_y, slot, n, y, x)) return;
  const float4* cp = reinterpret_cast<const float4*>(carrier) + (slot >> 7) * 16 * 128 + (slot & 127);
  const long long plane = static_cast<long long>(H) * W;
  float* o = out + static_cast<long long>(n) * 64 * plane + static_cast<long long>(y) * W + x;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const float4 v = cp[q * 128];
    o[(4 * q) * plane] = v.x; o[(4 * q + 1) * plane] = v.y; o[(4 * q + 2) * plane] = v.z; o[(4 * q + 3) * plane] = v.w;
  }
}

}  // namespace b200sr
