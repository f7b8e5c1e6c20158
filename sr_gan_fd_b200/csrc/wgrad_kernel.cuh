// Weight-gradient of the 3x3 convs as a tcgen05 GEMM whose reduction dimension is the PIXEL axis:
//
//   dW[tap][ci][co] = sum_{pixel} X[pixel + tap, ci] * dY[pixel, co]
//
// Both operands are NHWC bf16 tiles (rows = pixels, 64 channels = 128 B per row) brought in by TMA with the 128B
// swizzle, i.e. exactly the UMMA "MN-major" canonical layout (the GEMM K index walks smem rows).  One CTA owns one
// horizontal tap dx and a slice of the pixel tiles (split-K over pixels across CTAs); the three vertical taps are
// three accumulators fed from the same haloed X tile at +0/+1024/+2048 bytes.  M = 128 input channels (two 64-ch
// TMA boxes), N = up to 160 output-gradient channels -- for a dense block that is the concatenation
// [dY5|dY4|dY3|dY2|dY1] of all consumers of the input slice, so the X tile is read once for all five convs
// ("re-associated by input slice").  The accumulators (3 x N <= 480 TMEM columns) live in TMEM for the whole
// pixel loop and are flushed once with 16-byte vector reductions (red.global.add.v4.f32) into a [tap][co/4][ci][4]
// fp32 staging tensor; a small unpack kernel transposes that to the OIHW gradient layout per gradient bucket.
// kDet (deterministic plans): the flush stores instead, into one copy per pixel split of the part of the staging tensor the segment
// writes (the host hands the kernel a segment that describes that compact [tap][co/4][ci][4] copy: `out` is the slab, split s at
// s * 9 * co_pad * ci_total floats), and ordered_sum_kernel adds the copies in split order.
//
// One launch carries a BATCH of up to five such problems over the same two tensor maps (the five problems of a dense
// block), with the CTAs dealt out in proportion to each problem's cost so the whole dense block is one balanced wave.
//
// The two 64-row M blocks of a problem are described independently (WgradMBlock): each is X channels [c0, c0 + 64) at
// its own horizontal tap, an all-ones block, or idle.  A CTA that needs only 64 input channels therefore fills its
// other half with useful rows -- the same channels at another tap, or ones whose products are the bias gradients
// (column sums of dY) -- instead of multiplying rows that are never flushed (every tcgen05 MMA costs the same for
// M = 64 real rows as for 128).
#pragma once
#include "conv_kernel.cuh"

namespace b200sr {

constexpr int kWgTileH = 16;                         // wgrad K-tile: 8 x 16 pixels
constexpr int kWgXRows = kWgTileH + 2;
constexpr int kWgXBytes = kWgXRows * kTileW * 128;   // 18432 B per 64-channel haloed X tile
constexpr int kWgBBytes = kWgTileH * kTileW * 128;   // 16384 B per 64-channel dY tile
constexpr int kWgThreads = 192;
constexpr int kWgMaxSeg = 6;
constexpr int kWgMaxProblems = 5;

struct WgradSegment {
  int col_begin, col_end;  // accumulator columns of this conv's output channels (multiples of 16)
  float* out;              // gradient staging tensor, [tap][co_pad/4][ci_total][4] fp32: the 32 lanes (= input channels) of a
                           // warp reduce into 512 contiguous bytes per instruction (4 L1 wavefronts instead of 32)
  int ci_total;            // input channels of that conv
  int ci0;                 // conv input channel of accumulator row 0
  int co_pad;              // output channels rounded up to a multiple of 4
  int blk_mask;            // M blocks whose rows this segment flushes (bit b = block b; 0 = both)
};

enum : int { kWgBlkIdle = 0, kWgBlkX = 1, kWgBlkOnes = 2 };
// One 64-row half of the UMMA's M = 128, at stage offset b * kWgXBytes (the A descriptor's LBO).
//   kWgBlkX:    haloed X tile of channels [c0, c0 + 64) at horizontal tap dx; rows map to (tap, channel) in the flush.
//   kWgBlkOnes: bf16 1.0 (written once per ring stage, never loaded): every row and every vertical-tap accumulator holds the column
//               sums of dY, so ONE row of ONE accumulator is flushed -- the bias gradients of the problem's columns.
//   kWgBlkIdle: block 1 only: nothing loaded (the MMA reads whatever follows in the stage, finite data), nothing flushed.
struct WgradMBlock {
  int kind;
  int c0;
  int dx;  // 0..2, or -1: the CTA's own tap (the problem's dx_mask deals one tap per CTA).  Either both X blocks use -1 or neither.
};

struct WgradParams {
  WgradMBlock blk[2];
  int b_c0;      // first dY channel (accumulator column 0)
  int n_cols;    // UMMA N (multiple of 16, <= 160)
  int n_blocks;  // ceil(n_cols / 64) dY boxes per tile
  int splits;    // pixel-tile splits of this problem (CTAs = splits * wgrad_ntap)
  int num_seg;
  int dx_mask, dy_mask;  // horizontal taps that get a CTA / vertical taps that get an accumulator (0 = all three).  The 4x4 stride-2
                         // convs of the U-Net discriminator, computed as 3x3 convs over the pixel-unshuffled input, only have a
                         // 2 x 2 block of non-zero taps per unshuffle phase: the others are neither computed nor flushed
  WgradSegment seg[kWgMaxSeg];
};

struct WgradBatch {
  int N, H, W;
  int tiles_x, tiles_y, num_tiles;
  int num_problems;
  int a_f16, b_f16;  // 1: X (a) / dY (b) tiles are fp16 instead of bf16 (discriminator plans: both; the generator's fp16 tail activations: a)
  int cta_begin[kWgMaxProblems + 1];
  WgradParams prob[kWgMaxProblems];
};

// ring-stage footprint (an all-ones block keeps its slot) and the bytes TMA brings in per stage
__host__ __device__ inline int wgrad_stage_bytes(const WgradParams& p) {
  return (p.blk[1].kind == kWgBlkIdle ? 1 : 2) * kWgXBytes + p.n_blocks * kWgBBytes;
}
__host__ __device__ inline int wgrad_load_bytes(const WgradParams& p) {
  return ((p.blk[0].kind == kWgBlkX) + (p.blk[1].kind == kWgBlkX)) * kWgXBytes + p.n_blocks * kWgBBytes;
}
// CTAs per pixel split: one per horizontal tap of dx_mask when the X blocks follow the CTA's tap, else one
__host__ __device__ inline int wgrad_ntap(const WgradParams& p) {
  if (p.blk[0].dx >= 0) return 1;
  const int m = p.dx_mask ? p.dx_mask : 7;
  return (m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1);
}
// plain A operand: X channels [a_c0, a_c0 + 64 * a_blocks) at the CTA's tap (a_blocks = 1: block 1 idle)
__host__ inline void wgrad_set_a(WgradParams& p, int a_c0, int a_blocks) {
  p.blk[0].kind = kWgBlkX; p.blk[0].c0 = a_c0; p.blk[0].dx = -1;
  p.blk[1].kind = a_blocks == 2 ? kWgBlkX : kWgBlkIdle; p.blk[1].c0 = a_c0 + 64; p.blk[1].dx = -1;
}
constexpr int kWgSmemBytes = 227 * 1024;

template <bool kDet>
__global__ void __launch_bounds__(kWgThreads, 1)
wgrad3x3_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY,
                const __grid_constant__ WgradBatch batch) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kRing = kWgSmemBytes - 1024 - 1024;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kRing);
  uint64_t* full = bars;
  uint64_t* empty = bars + 4;
  uint64_t* done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // which problem / tap / split does this CTA own
  int pj = 0;
  while (pj + 1 < batch.num_problems && static_cast<int>(blockIdx.x) >= batch.cta_begin[pj + 1]) ++pj;
  const WgradParams& p = batch.prob[pj];
  const int local = blockIdx.x - batch.cta_begin[pj];
  const int dxm = p.dx_mask ? p.dx_mask : 7, dym = p.dy_mask ? p.dy_mask : 7;
  const int ntap = wgrad_ntap(p);
  int dxi = 1;  // horizontal tap owned by this CTA: the (local % ntap)-th set bit of the mask
  if (p.blk[0].dx < 0) {
    int k = local % ntap;
    dxi = 0;
    while (!((dxm >> dxi) & 1) || k-- > 0) ++dxi;
  }
  const int split = local / ntap;
  const int stage_bytes = wgrad_stage_bytes(p);
  int S = kRing / stage_bytes;
  if (S > 4) S = 4;
  const int b_off = stage_bytes - p.n_blocks * kWgBBytes;
  const int bdx0 = p.blk[0].dx >= 0 ? p.blk[0].dx : dxi, bdx1 = p.blk[1].dx >= 0 ? p.blk[1].dx : dxi;
  const bool ones_blk = p.blk[1].kind == kWgBlkOnes;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmX);
    prefetch_tensormap(&tmDY);
    for (int s = 0; s < 4; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_imm<512>(tmem_slot);
  if (ones_blk) {
    // all-ones M block 1: its slot of every ring stage, written once (the producer never loads into it)
    constexpr int kVec = kWgXBytes / 16;
    const uint32_t one2 = batch.a_f16 ? 0x3C003C00u : 0x3F803F80u;
    for (int i = threadIdx.x; i < S * kVec; i += kWgThreads) {
      const int s = i / kVec;
      *reinterpret_cast<uint4*>(smem + s * stage_bytes + kWgXBytes + (i - s * kVec) * 16) = make_uint4(one2, one2, one2, one2);
    }
    fence_proxy_async_smem();
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = batch.tiles_x * batch.tiles_y;
  const bool has_work = split < batch.num_tiles;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int tile = split; tile < batch.num_tiles; tile += p.splits) {
      const int n = tile / tiles_per_img;
      const int t2 = tile - n * tiles_per_img;
      const int ty = t2 / batch.tiles_x;
      const int x0 = (t2 - ty * batch.tiles_x) * kTileW;
      const int y0 = ty * kWgTileH;
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one_sync()) {
        uint8_t* st = smem + s * stage_bytes;
        mbar_arrive_expect_tx(&full[s], wgrad_load_bytes(p));
        if (p.blk[0].kind == kWgBlkX) tma_load_4d(st, &tmX, &full[s], p.blk[0].c0, x0 + bdx0 - 1, y0 - 1, n);
        if (p.blk[1].kind == kWgBlkX) tma_load_4d(st + kWgXBytes, &tmX, &full[s], p.blk[1].c0, x0 + bdx1 - 1, y0 - 1, n);
        for (int j = 0; j < p.n_blocks; ++j)
          tma_load_4d(st + b_off + j * kWgBBytes, &tmDY, &full[s], p.b_c0 + 64 * j, x0, y0, n);
      }
      __syncwarp();
      if (++s == S) { s = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_ab(128, p.n_cols, 1, 1, batch.a_f16 != 0, batch.b_f16 != 0);  // both operands MN-major
    constexpr uint32_t kHi = smem_desc_hi(1024);
    int s = 0;
    uint32_t ph = 0;
    uint32_t acc = 0;
    for (int tile = split; tile < batch.num_tiles; tile += p.splits) {
      mbar_wait(&full[s], ph);
      tcgen05_fence_after();
      if (elect_one_sync()) {
        const uint32_t a0 = smem_u32(smem + s * stage_bytes);
        const uint32_t b_lo = smem_desc_lo(a0 + b_off, kWgBBytes);  // LBO = stride between 64-ch N blocks
        const uint32_t a_lo = smem_desc_lo(a0, kWgXBytes);          // LBO = stride between the two 64-ch M blocks
#pragma unroll
        for (int dyi = 0; dyi < 3; ++dyi) {
          if (!((dym >> dyi) & 1)) continue;
#pragma unroll
          for (int ks = 0; ks < kWgTileH / 2; ++ks)  // 16 pixels (two 8-pixel patch rows) per UMMA
            umma_bf16_ss_lohi(tmem_base + dyi * p.n_cols, a_lo + dyi * 64 + ks * 128, b_lo + ks * 128, kHi, idesc,
                              (ks == 0) ? acc : 1u);
        }
        umma_commit(&empty[s]);
      }
      __syncwarp();
      acc = 1;
      if (++s == S) { s = 0; ph ^= 1; }
    }
    if (elect_one_sync()) umma_commit(done);
    __syncwarp();
  } else if (has_work && p.blk[(warp & 3) >> 1].kind != kWgBlkIdle) {
    // epilogue: flush the accumulators with 16-byte fp32 vector reductions into [tap][ci][co] staging tensors.  Warps 2 + q
    // hold accumulator rows 32q .. 32q + 31: rows 0..63 are M block 0, rows 64..127 block 1.
    const int q = warp & 3;
    const int b = q >> 1;
    const bool ones = p.blk[b].kind == kWgBlkOnes;
    // conv input channel = sg.ci0 + m: m counts X channels from block 0's first one (ones block: row 0 of the block)
    const int m = (ones ? 0 : p.blk[b].c0 - p.blk[0].c0) + (q & 1) * 32 + lane;
    const int bdx = b ? bdx1 : bdx0;
    const int nacc = ones ? 1 : 3;  // the vertical-tap accumulators of a ones block all hold the same column sums
    mbar_wait(done, 0);
    tcgen05_fence_after();
    for (int dyi = 0; dyi < nacc; ++dyi) {
      if (!ones && !((dym >> dyi) & 1)) continue;
      const int tap = ones ? 0 : dyi * 3 + bdx;
      for (int c0 = 0; c0 < p.n_cols; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + dyi * p.n_cols + c0, r);
        tmem_ld_wait();
        int sgi = 0;
        while (sgi < p.num_seg - 1 && (c0 >= p.seg[sgi].col_end || (p.seg[sgi].blk_mask && !((p.seg[sgi].blk_mask >> b) & 1)))) ++sgi;
        const WgradSegment& sg = p.seg[sgi];
        const int co = c0 - sg.col_begin;
        const int ci = sg.ci0 + m;
        if (c0 >= sg.col_begin && c0 < sg.col_end && ci < sg.ci_total && (!sg.blk_mask || ((sg.blk_mask >> b) & 1))) {
          float* dst = sg.out + ((static_cast<long long>(tap) * (sg.co_pad >> 2) + (co >> 2)) * sg.ci_total + ci) * 4;
          if constexpr (kDet) dst += static_cast<long long>(split) * 9 * sg.co_pad * sg.ci_total;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (co + 4 * j < sg.co_pad) {
              if constexpr (kDet)
                *reinterpret_cast<float4*>(dst + static_cast<long long>(j) * sg.ci_total * 4) =
                    make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
              else
                red_add_v4_f32(dst + static_cast<long long>(j) * sg.ci_total * 4, __uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                               __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
            }
        }
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_imm<512>(tmem_base);
  }
}

}  // namespace b200sr
