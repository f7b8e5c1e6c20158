// 3x3 / stride 1 / pad 1 convolution as an implicit GEMM on tcgen05 (sm_100a).  Used for every forward conv and
// every data-gradient conv of the RRDBNet generator (a dgrad is the same kernel over flipped/transposed weights).
//
//   D[pixel, cout] = sum_{tap, cin} X[pixel + tap, cin] * Wt[tap][cout][cin]        (fp32 accumulate in TMEM)
//
// Data layout: activations are NHWC bf16, possibly a channel range of a wider "dense" buffer (the dense block writes
// its growth channels into slices of one buffer, so no concat copy exists).  A work item = an 8-wide x 32-tall patch
// of one image = two M = 128 halves (one TMEM lane per pixel) that share every weight tile.  K is walked in chunks of
// 64 channels: per chunk ONE 4-D TMA box [64 ch, 10 px, 34 rows] (the patch plus a 1-pixel halo; out-of-image
// elements are zero-filled by TMA = the conv's zero padding) serves all nine taps -- the UMMA descriptor of tap
// (dy,dx) simply starts (dy*10+dx) rows = (dy*10+dx)*128 B into the tile with a 1280 B stride between 8-row groups.
// (Measured on B200, tools/probe_desc.cu: the 128B swizzle is applied on absolute shared-memory address bits, so
// start addresses that are not 1024-byte aligned and strides that are not multiples of 1024 read exactly the rows
// TMA wrote; the descriptor's base_offset field must stay 0.)  Weights are pre-packed per (chunk, dx, dy) as
// pre-swizzled [cout][64] K-major bf16 rows and stream through their own smem ring (10 granules of 12 KB), ONE 1-D bulk
// copy per stage of nine, three (one dx column) or one tap tile.
//
// Warp roles (352 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer, warp 10 = signaller,
// warps 2..5 / 6..9 = epilogue of the upper / lower 128-pixel half (TMEM -> registers -> fused bias / LeakyReLU /
// mask / residuals -> global).  Ordinary layers double buffer their accumulators in TMEM (epilogue of item i overlaps
// the MMAs of item i+1); the passes of a re-associated dense block keep their partial sums resident in the image
// group's accumulator slot from one layer to the next.
#pragma once
#include "ptx.cuh"


namespace b200sr {

constexpr int kTileW = 8;
constexpr int kTileH = 32;                              // a work item = 8 x 32 pixels = two M=128 halves sharing every weight tile
constexpr int kABoxRows = kTileH + 2;                   // 34 image rows incl. the vertical halo
constexpr int kABoxW = kTileW + 2;                      // 10 pixels incl. the horizontal halo
constexpr int kABytes = kABoxRows * kABoxW * 128;       // 43520 B: one haloed activation tile per 64-channel chunk
constexpr int kASlot = 44032;                           // A-ring slot (1024-byte multiple)
constexpr int kConvThreads = 352;  // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue of the upper 128-pixel half, warps 6-9 of the lower half

enum StoreMode : int {
  kStorePix = 0,        // same lattice position
  kStoreShuffle = 1,    // pixel-shuffle: column group (col / 64) = phase (a, b) -> pixel (2y+a, 2x+b), channel col % 64
  kStoreUnshuffle = 2,  // pixel-unshuffle: pixel (y, x) -> (y/2, x/2), channel ((y&1)*2 + (x&1)) * 64 + col
  kStoreFinal = 3,      // clamp to [0,1], NCHW fp32 image + clamp mask bytes (generator output head); epi.unclamped: no clamp, no mask
  kStoreNCHW = 4        // plain NCHW fp32 store of channels < n_valid to the per-launch output pointer (gradient w.r.t. the LR input)
};

struct ConvEpilogue {
  const float* bias;  // [n_total] or nullptr
  float alpha;        // v = alpha * (acc + bias)
  int act;            // 1: v = LeakyReLU_0.2(v)
  const __nv_bfloat16* mask;  // dgrad: v *= (m > 0 ? 1 : 0.2), m = saved forward activation at the same pixel
  int mask_stride;            // channels per pixel of the mask buffer
  int mask_coff;
  // fp32 residual carriers use a TILE-BLOCKED layout private to the epilogues: [tile][half][16-byte chunk][pixel-in-half]
  // [4 floats], so the 32 lanes (= 32 pixels) of a warp access 512 contiguous bytes per instruction (4 wavefronts, not 32)
  const float* r1;
  const float* r2;
  float beta1, beta2;
  int res_stride;
  float* out_f32;    // optional fp32 copy of v ([pixel][of_stride])
  float* out_f32_b;  // optional second fp32 copy
  int of_stride;
  __nv_bfloat16* out_bf16;  // optional bf16(delta * v) at channel ob_coff + col
  int ob_stride;
  int ob_coff;
  float delta;
  int split_off;  // > 0: also store a second 16-bit copy at channel ob_coff + split_off + col: lo = bf16(delta*v - hi) (bf16 layers) or
                  // bf16(delta*v) (fp16 layers: the bf16 twin the weight-gradient GEMM reads)
  int store_mode;
  unsigned char* clamp_mask;  // kStoreFinal, may be nullptr
  int n_valid;                // kStoreFinal: real output channels (<= 16)
  // VGG feature layers (sr_gan_fd_b200/vgg.py): act == 2 is ReLU, mask_relu makes the dgrad mask the ReLU derivative, and
  // feat_out receives alpha * (acc + bias) as plain fp32 NHWC rows ([pixel][feat_stride], column col) -- before the activation,
  // or after it when bit 1 of mask_relu is set
  int mask_relu;  // bit 0: dgrad mask is the ReLU derivative; bit 1: feat_out is stored after the activation
  int feat_stride;
  float* feat_out;
  // U-Net discriminator layers (sr_gan_fd_b200/discriminator.py; extended build only): a bf16 residual read at the DESTINATION
  // address of the bf16 store (after the pixel shuffle) and added BEFORE the activation-derivative mask -- the skip-connection
  // gradient joining the data gradient of a stride-2 conv -- and the channel count of one pixel-(un)shuffle phase (0 = 64)
  const __nv_bfloat16* res_bf16;
  int res_bf16_stride;
  int shuf_c;
  int f16;  // 1: this layer's 16-bit operands / outputs / residual are fp16 instead of bf16 (same tcgen05 kind::f16 instruction): the
            // generator's head / tail convs (one fp16 product instead of three split-bf16 ones) and the discriminator plans
  int unclamped;  // kStoreFinal only: store the conv output as it is, no clamp (unclamped generator plans; clamp_mask is nullptr).
                  // Occupies what was the struct's tail padding: sizeof(ConvParams) and the staging copy are unchanged
};

struct ConvParams {
  int N, H, W;  // pixel lattice the conv runs on
  int tiles_x, tiles_y, num_tiles;
  int num_chunks;   // K chunks of 64 channels
  int ksteps_last;  // 16-channel k-steps issued for the last chunk (1..4); other chunks use 4
  int a_c0;         // activation channel coordinate of chunk c: a_c0 + (c % a_wrap) * 64
  int a_wrap;
  int w_row0;   // first row of this conv in the packed weight matrix
  int n_cols;   // UMMA N handled by one work item (multiple of 16, <= 64 for ordinary layers, <= 192 for pass layers)
  int n_total;  // n_cols * col_groups
  int col_groups;  // work item w -> tile w / col_groups, column group w % col_groups
  int w_taps;      // taps fetched per weight bulk copy: 9 (a whole K chunk), 3 (one dx column) or 1
  // accumulator placement.  Ordinary layers: fresh accumulators, double buffered (acc_hold = 0).  Dense-block PASS layers
  // (acc_hold = 1): the block's 192 accumulator columns live in a fixed TMEM block across five consecutive entries; pass j
  // adds input slice j's contribution to columns [acc_col0, acc_col0 + n_cols) and its epilogue consumes the leading
  // epi_cols columns (the conv that just became complete).
  int halves;      // 128-pixel halves per work item: 2 (8 x 32 patch, ordinary layers) or 1 (8 x 16 unit, dense-block passes)
  int acc_col0;
  int acc_first;   // 1: the first MMA of an item overwrites the accumulators, 0: accumulate onto earlier passes
  int acc_hold;
  int epi_cols;
  int num_stages;
  int k32;         // weights of this (single-chunk, 32-channel) layer are packed as 64-byte rows (64B swizzle)
  // 4x4 stride-2 convs over the pixel-unshuffled input (U-Net discriminator; extended build only): of the nine taps only a 2 x 2
  // subset is non-zero for the channels of one unshuffle phase.  w_taps == 4: ONE weight stage per K chunk holding those four tap
  // tiles.  The phase is that of the K chunk (down_mode 1, forward: chunk / down_c64) or of the item's column group (down_mode 2,
  // data gradient: column group / down_c64); down_c64 = channels of one phase / 64.
  int down_mode;
  int down_c64;
  int mma_f16;     // 1: the layer's activation AND weight tiles are fp16 (instruction descriptor a / b format); epi.f16 is the STORE format
  int pad_[2];
  ConvEpilogue epi;
};

__host__ __device__ constexpr int conv_smem_bytes(int ctas_per_sm) { return ctas_per_sm == 1 ? 227 * 1024 : 112 * 1024; }
__host__ inline int conv_pick_stages(int n_cols) { return n_cols >= 128 ? 2 : 3; }  // A-ring depth (informational)

// tile-blocked carrier layout: float offset of (tile, half, pixel m, chunk 0); consecutive 16-byte chunks are 512 floats apart
constexpr int kCarrierChunkStride = 128 * 4;
__host__ __device__ inline long long carrier_base(int tile, int half, int m) {
  return ((static_cast<long long>(tile) * 2 + half) * 16 * 128 + m) * 4;
}
constexpr long long kCarrierBytesPerTile = 2LL * 16 * 128 * 16;  // 65536

__device__ __forceinline__ float lrelu02(float v) { return v > 0.f ? v : 0.2f * v; }

// Store 64 contiguous bytes per lane (h[16] -> row pointer `row`) so that each warp-wide store instruction covers
// whole 64-byte runs: the four lanes of a quad first transpose their 4 x 4 grid of 16-byte pieces with two rounds of
// shuffles, then instruction i writes piece (lane & 3) of the quad's i-th row.  A warp store touches 8 rows x 64 B
// instead of 32 rows x 16 B (4x fewer L1 wavefronts).  All 32 lanes must call this; `ok` guards the lane's own row.
__device__ __forceinline__ void store_rows_quad(uint32_t (&h)[16], void* row, bool ok, int lane) {
  const bool b0 = lane & 1, b1 = lane & 2;
#pragma unroll
  for (int c = 0; c < 4; c += 2) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t send = b0 ? h[4 * c + k] : h[4 * (c + 1) + k];
      const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 1);
      if (b0) h[4 * c + k] = recv; else h[4 * (c + 1) + k] = recv;
    }
  }
#pragma unroll
  for (int sidx = 0; sidx < 2; ++sidx) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t send = b1 ? h[4 * sidx + k] : h[4 * (sidx + 2) + k];
      const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 2);
      if (b1) h[4 * sidx + k] = recv; else h[4 * (sidx + 2) + k] = recv;
    }
  }
  const unsigned long long mine = reinterpret_cast<unsigned long long>(row);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int src = (lane & ~3) + i;
    const unsigned long long r = __shfl_sync(0xffffffffu, mine, src);
    const int rok = __shfl_sync(0xffffffffu, ok ? 1 : 0, src);
    if (rok) st_global_v4(reinterpret_cast<uint8_t*>(r) + (lane & 3) * 16, h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogue for one pixel and 32 (or 16) consecutive accumulator columns held in registers.
//   sbias : this layer's bias vector staged in shared memory (indexed by global column)
//   res   : beta1*r1 + beta2*r2 for these 32 columns, prefetched before the accumulator was ready (or nullptr)
//   maskw : 16 words = 32 bf16 saved activations for the LeakyReLU-derivative mask, prefetched (or nullptr)
// ---------------------------------------------------------------------------------------------------------------
struct HW { int H, W; bool nostore; };
// Part 1 (registers only): bias + scale, LeakyReLU, LeakyReLU-derivative mask, fp32 residuals.
template <int kVgg>
__device__ __forceinline__ void conv_epilogue_math(const ConvEpilogue& e, const float* sbias, const float (&res)[32], bool has_res,
                                                   const uint32_t (&maskw)[16], bool has_mask, int col0, int ncol, float (&v)[32],
                                                   float* feat_row = nullptr) {
  if (kVgg && !e.bias) {  // bias-free layer (its columns may exceed the staged bias slot): scale only
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] *= e.alpha;
  } else if (ncol == 32) {
    const float4* b4 = reinterpret_cast<const float4*>(sbias + col0);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 b = b4[q];
      v[4 * q] = e.alpha * (v[4 * q] + b.x); v[4 * q + 1] = e.alpha * (v[4 * q + 1] + b.y);
      v[4 * q + 2] = e.alpha * (v[4 * q + 2] + b.z); v[4 * q + 3] = e.alpha * (v[4 * q + 3] + b.w);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = e.alpha * (v[i] + sbias[col0 + i]);
  }
  if (kVgg && feat_row && !(e.mask_relu & 2)) {  // pre-activation feature map (VGG node that ends the graph), fp32
#pragma unroll
    for (int q = 0; q < 8; ++q) st_global_v4f(feat_row + 4 * q, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  }
  if (e.act == 1) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.2f * v[i]);  // LeakyReLU(0.2)
  } else if (kVgg && e.act == 2) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);          // ReLU
  }
  if (kVgg && feat_row && (e.mask_relu & 2)) {  // feature node followed by torchvision's IN-PLACE ReLU: what the reference reads is post-ReLU
#pragma unroll
    for (int q = 0; q < 8; ++q) st_global_v4f(feat_row + 4 * q, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  }
  const bool res_first = kVgg && e.res_bf16 != nullptr;  // skip-connection gradient: joins BEFORE the activation derivative
  if (res_first && has_res) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += res[i];
  }
  if (has_mask) {  // activation derivative from the saved forward activation (LeakyReLU 0.2, or ReLU)
    const float neg = (kVgg && (e.mask_relu & 1)) ? 0.f : 0.2f;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      // (extended build: a sign / magnitude test on the bit pattern, valid for bf16 and fp16 activations alike)
      v[2 * j] *= (kVgg ? pos16_lo(maskw[j]) : (bf16_lo_to_f32(maskw[j]) > 0.f)) ? 1.f : neg;
      v[2 * j + 1] *= (kVgg ? pos16_hi(maskw[j]) : (bf16_hi_to_f32(maskw[j]) > 0.f)) ? 1.f : neg;
    }
  }
  if (has_res && !res_first) {  // fp32 residuals (already combined)
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += res[i];
  }
}

// Destination of the bf16 store of global column col0 at lattice position (n, y, x): pixel index and channel, with the pixel
// (un)shuffle folded in.  kExt = 0 (generator build): a phase is always 64 channels wide.
template <int kExt>
__device__ __forceinline__ void conv_store_dest(const HW p, const ConvEpilogue& e, int n, int y, int x, int col0, long long& opix, int& ch) {
  const int sc = (kExt && e.shuf_c > 0) ? e.shuf_c : 64;
  if (e.store_mode == kStoreShuffle) {
    const int phase = kExt ? col0 / sc : (col0 >> 6);
    opix = (static_cast<long long>(n) * (2 * p.H) + (2 * y + (phase >> 1))) * (2 * p.W) + (2 * x + (phase & 1));
    ch = kExt ? col0 - phase * sc : (col0 & 63);
  } else if (e.store_mode == kStoreUnshuffle) {
    opix = (static_cast<long long>(n) * (p.H >> 1) + (y >> 1)) * (p.W >> 1) + (x >> 1);
    ch = (((y & 1) << 1) | (x & 1)) * sc + col0;
  } else {
    opix = (static_cast<long long>(n) * p.H + y) * p.W + x;
    ch = col0;
  }
}

// Part 2: stores.  Called by all 32 lanes of the warp (the bf16 store shuffles); `ok` = this lane's pixel exists and
// stores are enabled.
template <int kExt>
__device__ __forceinline__ void conv_epilogue_write(const HW p, const ConvEpilogue& e, float* y_dyn, long long cbase, int n, int y, int x,
                                                    int col0, float (&v)[32], bool ok, int lane) {
  if (__builtin_expect(e.store_mode == kStoreNCHW, 0)) {
    if (!ok) return;
    const long long plane = static_cast<long long>(p.H) * p.W;
    const long long base = static_cast<long long>(n) * e.n_valid * plane + static_cast<long long>(y) * p.W + x;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (col0 + i < e.n_valid) st_global_f32(y_dyn + base + (col0 + i) * plane, v[i]);
    return;
  }
  if (__builtin_expect(e.store_mode == kStoreFinal, 0)) {
    if (!ok) return;
    const long long plane = static_cast<long long>(p.H) * p.W;
    const long long base = static_cast<long long>(n) * e.n_valid * plane + static_cast<long long>(y) * p.W + x;
    const bool unclamped = e.unclamped;  // read once: the stores below are volatile asm, which would reload it per channel
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (i < e.n_valid) {
        float pre = v[i];
        float cl = unclamped ? pre : fminf(fmaxf(pre, 0.f), 1.f);
        st_global_f32(y_dyn + base + i * plane, cl);  // the generator output tensor is passed per launch, not baked into the layer list
        if (e.clamp_mask) st_global_u8(e.clamp_mask + base + i * plane, (pre >= 0.f && pre <= 1.f) ? 1u : 0u);
      }
    }
    return;
  }
  // 4. fp32 outputs (same lattice position)
  if (e.out_f32 && ok) {
    float* op = e.out_f32 + cbase + (col0 >> 2) * kCarrierChunkStride;
#pragma unroll
    for (int q = 0; q < 8; ++q) st_global_v4f(op + q * kCarrierChunkStride, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  }
  if (e.out_f32_b && ok) {
    float* op = e.out_f32_b + cbase + (col0 >> 2) * kCarrierChunkStride;
#pragma unroll
    for (int q = 0; q < 8; ++q) st_global_v4f(op + q * kCarrierChunkStride, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  }
  // 5. bf16 output (optionally hi/lo split), with the pixel (un)shuffle folded into the address
  if (e.out_bf16) {
    long long opix;
    int ch;
    conv_store_dest<kExt>(p, e, n, y, x, col0, opix, ch);
    __nv_bfloat16* ob = e.out_bf16 + opix * e.ob_stride + e.ob_coff + ch;
    uint32_t hi[16];
    if (__builtin_expect(e.f16 != 0, 0)) {  // (uniform branch: the generator's fp16 tail layers and the discriminator plans)
#pragma unroll
      for (int j = 0; j < 16; ++j) hi[j] = pack_f16x2(e.delta * v[2 * j], e.delta * v[2 * j + 1]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) hi[j] = pack_bf16x2(e.delta * v[2 * j], e.delta * v[2 * j + 1]);
    }
    uint32_t lo[16];
    if (__builtin_expect(e.split_off > 0, 0)) {
      if (e.f16) {  // fp16 primary copy: the second copy is the SAME value in bf16 (weight-gradient operand: its MMA partner, dY, is bf16)
#pragma unroll
        for (int j = 0; j < 16; ++j) lo[j] = pack_bf16x2(e.delta * v[2 * j], e.delta * v[2 * j + 1]);
      } else {      // bf16 primary copy: the second copy is the rounding residual (split-precision operand pair [hi | lo])
#pragma unroll
        for (int j = 0; j < 16; ++j)
          lo[j] = pack_bf16x2(e.delta * v[2 * j] - bf16_lo_to_f32(hi[j]), e.delta * v[2 * j + 1] - bf16_hi_to_f32(hi[j]));
      }
    }
    store_rows_quad(hi, ob, ok && !p.nostore, lane);
    if (__builtin_expect(e.split_off > 0, 0)) store_rows_quad(lo, ob + e.split_off, ok && !p.nostore, lane);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// One layer = one 3x3 conv over one pixel lattice.  A launch executes a CHAIN of ENTRIES: entry = (layer, image group).
// Persistent CTAs (one per SM, cooperative launch) walk the entry list; the three warp roles of a CTA run through
// it asynchronously from each other.  There is no grid-wide barrier: every entry has a completion counter that each
// CTA's epilogue bumps when its stores for that entry are done, and an entry's inputs are only read once the counter
// of the entry it depends on (the previous layer OF THE SAME IMAGE GROUP) shows all CTAs.  With two image groups the
// dependency / TMA / epilogue latency of one group hides behind the other group's tensor work.  The whole forward
// pass (351 convs) is ONE launch; pipeline state (smem rings, TMEM, mbarriers) is set up once.
// ---------------------------------------------------------------------------------------------------------------
struct alignas(128) LayerDesc {
  CUtensorMap tmA;  // activation tensor map of this layer (lives in global memory, read by TMA through a generic address)
  ConvParams p;
};
struct alignas(32) EntryDesc {
  int layer;             // index into the layer list handed to the kernel
  int tile_lo, tile_hi;  // pixel tiles of this entry (an image group of the layer)
  int dep;               // entry whose completion gates this entry's input reads (-1: inputs exist before the launch)
  int rot;               // CTA rotation: virtual CTA v = (blockIdx.x - rot) mod gridDim.x takes items v, v + gridDim.x, ...
  int slot;              // dense-block passes: which of the CTA's two resident accumulator blocks this image group uses
  int pad[2];            // pad[0] = 1: this entry announces itself PER IMAGE (counter 1 + image of the entry's range) instead of on the entry's
                         // one counter: every entry that depends on it maps the same tiles to the same CTAs, so a consumer only waits
                         // for the tiles of its OWN image (a conv reads nothing of another image)
};

// Compact per-layer / per-entry records for the TMA-producer and MMA-issuer warps, kept in CONSTANT memory: loads with a
// warp-uniform index go through the uniform datapath, so everything derived from them (TMEM addresses, instruction
// descriptors, loop bounds) stays in uniform registers and tcgen05.mma issues back to back without R2UR round trips.
// The host copies the slice of the chain being launched into these tables right before the launch (stream ordered).
constexpr int kMaxChainLayers = 768;
constexpr int kMaxChainEntries = 2048;
// layer record A: x = n_cols (9 bits) | chunks<<9 (5 bits) | ksteps_last<<14 | halves<<17 | w_taps<<19 | col_groups<<23
//                 y = acc_col0 | acc_first<<8 | acc_hold<<9 | has_epi<<10 | k32<<11 | down_mode<<12 | down_c64<<14 | mma_f16<<17      z = w_row0      w = a_c0
// layer record B: x = tiles_x | tiles_y<<16      y = a_wrap      z = bias byte offset in the packed buffer + 1 (0: none)      w = bias floats
// entry record  : x = layer (absolute) | slot<<20 | per_image_announce<<21      y = tile_lo      z = tile_hi      w = rot | (dep+1)<<16
__constant__ uint4 c_layer_rec[kMaxChainLayers * 2];
__constant__ uint4 c_entry_rec[kMaxChainEntries];
inline void make_layer_rec(const ConvParams& p, uint4 out[2], const void* packed_base) {
  out[0].x = static_cast<uint32_t>(p.n_cols) | (p.num_chunks << 9) | (p.ksteps_last << 14) | (p.halves << 17) | (p.w_taps << 19) | (p.col_groups << 23);
  out[0].y = static_cast<uint32_t>(p.acc_col0) | ((p.acc_first ? 1u : 0u) << 8) | ((p.acc_hold ? 1u : 0u) << 9) | ((p.epi_cols > 0 ? 1u : 0u) << 10) |
             ((p.k32 ? 1u : 0u) << 11) | (static_cast<uint32_t>(p.down_mode & 3) << 12) | (static_cast<uint32_t>(p.down_c64 & 7) << 14) |
             ((p.mma_f16 ? 1u : 0u) << 17);
  out[0].z = static_cast<uint32_t>(p.w_row0);
  out[0].w = static_cast<uint32_t>(p.a_c0);
  out[1].x = static_cast<uint32_t>(p.tiles_x) | (static_cast<uint32_t>(p.tiles_y) << 16);
  out[1].y = static_cast<uint32_t>(p.a_wrap);
  out[1].z = p.epi.bias ? static_cast<uint32_t>(reinterpret_cast<const char*>(p.epi.bias) - static_cast<const char*>(packed_base)) + 1u : 0u;
  out[1].w = static_cast<uint32_t>(p.acc_hold ? p.epi_cols : p.n_total);
}
inline uint4 make_entry_rec(const EntryDesc& e) {
  uint4 r;
  r.x = static_cast<uint32_t>(e.layer) | (static_cast<uint32_t>(e.slot & 1) << 20) | (static_cast<uint32_t>(e.pad[0] & 1) << 21);
  r.y = static_cast<uint32_t>(e.tile_lo);
  r.z = static_cast<uint32_t>(e.tile_hi);
  r.w = static_cast<uint32_t>(e.rot) | (static_cast<uint32_t>(e.dep + 1) << 16);
  return r;
}


constexpr int kWGranule = 12288;   // weight ring granule = one (chunk, dx) stage of a 32-column layer (3 taps x 32 x 128 B)
constexpr int kWGranules = 10;
constexpr int kNumASlots = 2;

// Software profiler (debug bit 64): cycles each warp role of every CTA spends in each kind of wait, summed over a launch.
//  [0] producer: dependency wait   [1] producer: A slot free   [2] producer: W granules free   [3] producer: total
//  [4] MMA: accumulator free       [5] MMA: A tile landed      [6] MMA: W stage landed         [7] MMA: total
//  [8] epilogue(warp 2): dependency wait + barriers   [9] epilogue: accumulator ready   [10] epilogue: total   [11] items
constexpr int kTlEntries = 256, kTlFirst = 300, kTlCtas = 4, kTlStride = 37;
__device__ unsigned long long g_conv_prof[160 * 12 + kTlCtas * kTlEntries * 16];
// debug bit 128: per-entry event timeline (globaltimer ns) of CTAs 0, 37, 74, 111 for entries [kTlFirst, kTlFirst + kTlEntries):
//  0 producer reaches the entry   1 producer: dependency seen done   2 MMA: accumulator free, entry's first item starts
//  3 MMA: first A tile landed     4 MMA: last MMA issued (tfull commit)   5 epilogue: accumulator ready
//  6 epilogue: stores issued      7 signaller: counter bumped    8 epilogue: entry start (after bar)   9 epilogue: dependency flag seen
//  10 epilogue: first TMEM load returned   11 signaller: epilogue warps arrived
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TL_MARK(ev)                                                                                                   \
  do {                                                                                                                \
    if (kInstr && tl && e >= kTlFirst && e < kTlFirst + kTlEntries)                                                    \
      g_conv_prof[160 * 12 + ((blockIdx.x / kTlStride) * kTlEntries + (e - kTlFirst)) * 16 + (ev)] = globaltimer_ns();   \
  } while (0)
#define PROF_T0(flag) const long long _t0 = (kInstr && (flag)) ? clock64() : 0
#define PROF_ADD(flag, slot) do { if (kInstr && (flag)) prof[slot] += clock64() - _t0; } while (0)

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Wait until every CTA has finished entry `dep` (one lane polls; bounded so a broken chain traps instead of hanging).
// Completion counters: kCtrStride words per entry -- word 0 counts the CTAs that finished their share of the entry (consumers whose
// tile -> CTA mapping differs wait for all of them), words 1 + i the finished tiles of image i of the entry's range (per-image announce).
constexpr int kCtrStride = 16;
__device__ __forceinline__ void wait_entry_done(const unsigned int* ctr, int dep, unsigned int need) {
  const long long t0 = clock64();
  while (ld_acquire_gpu(ctr) < need) {
    if (clock64() - t0 > 4000000000LL) {
      printf("b200sr: dependency wait timeout (block %d entry %d)\n", blockIdx.x, dep);
      __trap();
    }
  }
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }  // the 8 epilogue warps

// One weight stage worth of tcgen05.mma, fully unrolled with compile-time tap offsets so that consecutive MMAs differ
// only by immediates added to uniform registers.  TAPS = taps in the stage (9: whole 3x3, centre first; 3: the three
// dy of one dx column -- a_lo / b_base already point at that column; 1: a single tap), HALVES = 128-pixel halves of
// the work item (the second half reuses the weight tile), KSTEPS = 16-channel K steps of this chunk.
template <int TAPS, int HALVES, int KSTEPS>
__device__ __forceinline__ void issue_stage(uint32_t d_tmem, uint32_t a_lo, uint32_t b_base, uint32_t b_dy, uint32_t idesc, uint32_t first,
                                            uint32_t kHi /* weight descriptor hi word: 128-byte rows (SBO 1024) or 64-byte rows (SBO 512, 64B swizzle) */) {
  constexpr uint32_t kHiA = smem_desc_hi(kABoxW * 128);   // activations: 8 pixels of a patch row, rows 1280 B apart
  constexpr int ord[3] = {1, 0, 2};
#pragma unroll
  for (int tt = 0; tt < TAPS; ++tt) {
    const int dxi = (TAPS == 9) ? ord[tt / 3] : 0;   // TAPS 3 / 1: the caller folded dx (and dy) into a_lo
    const int dyi = (TAPS == 1) ? 0 : ord[tt % 3];
    const int tile_in_stage = (TAPS == 9) ? dxi * 3 + dyi : (TAPS == 3 ? dyi : 0);  // rows are packed [dx][dy][n]
    const uint32_t b_lo = b_base + tile_in_stage * b_dy;
    const uint32_t a_tap = a_lo + (dyi * kABoxW + dxi) * 8;  // tap (dy,dx) = the haloed tile shifted by dy*10+dx rows of 128 B
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
      const uint32_t acc = (tt == 0 && ks == 0) ? first : 1u;
      umma_bf16_ss_lohi2(d_tmem, a_tap + ks * 2, kHiA, b_lo + ks * 2, kHi, idesc, acc);
      if (HALVES == 2) umma_bf16_ss_lohi2(d_tmem + 128, a_tap + 16 * kABoxW * 8 + ks * 2, kHiA, b_lo + ks * 2, kHi, idesc, acc);
    }
  }
}

// All weight stages of one K chunk (TAPS taps per stage -> 9 / TAPS stages), fully specialised: per stage nothing but the
// barrier wait, the unrolled MMAs, one commit and the ring bookkeeping.  Executed by the whole MMA warp (uniform).
template <int TAPS, int HALVES, int KSTEPS>
__device__ __forceinline__ void issue_chunk(uint32_t d_tmem, uint32_t a_lo, uint32_t smemW_addr, uint32_t b_dy, uint32_t idesc, bool fresh,
                                            int g, int& gw, uint32_t& fW_bits, uint64_t* fullW, uint64_t* emptyW, bool no_mma, uint32_t b_hi) {
  constexpr int kStages = 9 / TAPS;
  constexpr int ord[3] = {1, 0, 2};
#pragma unroll
  for (int d = 0; d < kStages; ++d) {
    if (gw + g > kWGranules) gw = 0;
    // centre-first tap order: stage d of a 3-tap layer is the dx column {1,0,2}[d], of a 1-tap layer tap (dx,dy) = ({1,0,2}[d/3], {1,0,2}[d%3])
    const int dxi = (TAPS == 9) ? 0 : ord[(TAPS == 1) ? d / 3 : d];
    const int dyi = (TAPS == 1) ? ord[d % 3] : 0;
    const uint32_t a1 = a_lo + (dyi * kABoxW + dxi) * 8;
    const uint32_t b_base = ((smemW_addr + gw * kWGranule) >> 4 & 0x3FFFu) | (1u << 16);  // smem_desc_lo(addr, 16)
    mbar_wait(&fullW[gw], (fW_bits >> gw) & 1u);
    // (no tcgen05 fence here: the mbarrier wait orders the TMA writes before the MMAs that read them)
    if (elect_one_sync()) {
      if (!no_mma) issue_stage<TAPS, HALVES, KSTEPS>(d_tmem, a1, b_base, b_dy, idesc, (fresh && d == 0) ? 0u : 1u, b_hi);
      umma_commit(&emptyW[gw]);  // one commit per stage: frees its weight granules and (last stage of a chunk) the activation tile
    }
    __syncwarp();
    fW_bits ^= (1u << gw);
    gw += g;
  }
}

// The four non-zero taps of a stride-2 conv's K chunk / column group (see ConvParams::down_mode): rows {1,2} (SY = 0) or {0,1}
// (SY = 1) times columns {1,2} / {0,1} (SX) of the 3 x 3 neighbourhood; the stage holds the four tap tiles in that order.
template <int SY, int SX>
__device__ __forceinline__ void issue_stage_down(uint32_t d_tmem, uint32_t a_lo, uint32_t b_base, uint32_t b_dy, uint32_t idesc, uint32_t first, uint32_t kHi) {
  constexpr uint32_t kHiA = smem_desc_hi(kABoxW * 128);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int dyi = (SY ? 0 : 1) + (i >> 1), dxi = (SX ? 0 : 1) + (i & 1);
    const uint32_t b_lo = b_base + i * b_dy;
    const uint32_t a_tap = a_lo + (dyi * kABoxW + dxi) * 8;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t acc = (i == 0 && ks == 0) ? first : 1u;
      umma_bf16_ss_lohi2(d_tmem, a_tap + ks * 2, kHiA, b_lo + ks * 2, kHi, idesc, acc);
      umma_bf16_ss_lohi2(d_tmem + 128, a_tap + 16 * kABoxW * 8 + ks * 2, kHiA, b_lo + ks * 2, kHi, idesc, acc);
    }
  }
}
__device__ __forceinline__ void issue_chunk_down(int sel, uint32_t d_tmem, uint32_t a_lo, uint32_t smemW_addr, uint32_t b_dy, uint32_t idesc, bool fresh,
                                                 int g, int& gw, uint32_t& fW_bits, uint64_t* fullW, uint64_t* emptyW, uint32_t b_hi) {
  if (gw + g > kWGranules) gw = 0;
  const uint32_t b_base = ((smemW_addr + gw * kWGranule) >> 4 & 0x3FFFu) | (1u << 16);
  mbar_wait(&fullW[gw], (fW_bits >> gw) & 1u);
  if (elect_one_sync()) {
    const uint32_t first = fresh ? 0u : 1u;
    switch (sel) {
      case 0: issue_stage_down<0, 0>(d_tmem, a_lo, b_base, b_dy, idesc, first, b_hi); break;
      case 1: issue_stage_down<0, 1>(d_tmem, a_lo, b_base, b_dy, idesc, first, b_hi); break;
      case 2: issue_stage_down<1, 0>(d_tmem, a_lo, b_base, b_dy, idesc, first, b_hi); break;
      default: issue_stage_down<1, 1>(d_tmem, a_lo, b_base, b_dy, idesc, first, b_hi); break;
    }
    umma_commit(&emptyW[gw]);
  }
  __syncwarp();
  fW_bits ^= (1u << gw);
  gw += g;
}

// kInstr = 0: production build (no probes: every `debug` test folds away).  kInstr = 1: the same kernel with the timing
// switches, role profiler and per-entry timeline compiled in (used only while b200sr_debug_set() is non-zero).
// kVgg = 1: the build used by the VGG19 feature plans (ReLU, ReLU-derivative mask, fp32 feature store, bias vectors of up to 512
// columns); the generator's build (kVgg = 0) compiles none of it -- its epilogue sits on the dependency chain of every layer.
template <int kInstr, int kVgg>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_chain_kernel(const LayerDesc* __restrict__ layers, const EntryDesc* __restrict__ entries, int num_entries,
                     const uint8_t* __restrict__ packed_w, unsigned int* counters, float* y_dyn, int debug_arg, int layer0) {
  const int debug = kInstr ? debug_arg : 0;
  // `entries` points at the first entry of THIS chain; c_entry_rec[0..num_entries) / c_layer_rec[2 * (layer - layer0)] mirror it
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, still provably a shared-memory pointer
  // [ A ring: kNumASlots x 44032 | W ring: kWGranules x 12288 | barriers 512 B | flags | epilogue params 4 x 384 B | epilogue bias 4 x 1 KB ]
  uint8_t* smemW = smem + kNumASlots * kASlot;
  uint8_t* fixed = smemW + kWGranules * kWGranule;
  uint64_t* bars = reinterpret_cast<uint64_t*>(fixed);
  uint64_t* fullA = bars;        // [4]
  // (bars + 4 .. 7: spare; the activation slots are released through the weight-stage barriers)
  uint64_t* fullW = bars + 8;    // [10]
  uint64_t* emptyW = bars + 18;  // [10]
  uint64_t* tfull = bars + 28;   // [2]
  uint64_t* tempty = bars + 30;  // [2]
  uint64_t* sig = bars + 32;     // [2] epilogue warps -> signaller warp: "my stores for entry e are issued"
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(fixed + 512);
  volatile uint32_t* dep_flag = reinterpret_cast<volatile uint32_t*>(fixed + 516);  // producer -> epilogue: e + 1 once entry e's dependency is done
  volatile uint32_t* sig_done = reinterpret_cast<volatile uint32_t*>(fixed + 520);  // signaller -> epilogue: entries announced so far
  uint8_t* sp_base = fixed + 1024;                                  // 4 x 384 B
  float* sbias_base = reinterpret_cast<float*>(fixed + 3072);       // 4 x 1 KB (kVgg: 4 x 2 KB, up to 512 bias floats per layer)
  constexpr int kBiasSlot = kVgg ? 512 : 256;                       // floats
  constexpr int kFixedBytes = 3072 + 4 * kBiasSlot * 4;
  static_assert(sizeof(ConvParams) <= 384 && sizeof(ConvParams) % 16 == 0, "ConvParams must fit the 384-byte smem slot in 16-byte pieces");
  static_assert(kNumASlots * kASlot + kWGranules * kWGranule + kFixedBytes + 1024 <= conv_smem_bytes(1), "smem budget");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const unsigned int grid = gridDim.x;
  constexpr uint32_t kTmemCols = 512;
  constexpr int kAccStride = 256;  // TMEM columns between the two accumulator stages (each: two halves x <= 128 columns)

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < 4; ++s) mbar_init(&fullA[s], 1);
    for (int s = 0; s < kWGranules; ++s) { mbar_init(&fullW[s], 1); mbar_init(&emptyW[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 8); mbar_init(&sig[a], 8); }
    *dep_flag = 0;
    *sig_done = 0;
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_imm<kTmemCols>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool tl = (debug & 128) && (blockIdx.x % kTlStride == 0) && (blockIdx.x / kTlStride < kTlCtas) && (lane == 0);

  if (warp == 0) {
    // ================================================= TMA producer =================================================
    // (whole warp walks the loops so the index math stays warp-uniform; one elected lane issues)
    // Weight stages form one FIFO: the MMA warp commits ONCE per stage (to the barrier of the stage's first granule; a
    // tcgen05.commit costs about as much tensor-pipe time as 1.5 MMAs) and stages complete in issue order, so "granule
    // free" and "A slot free" both reduce to "stage number s has completed".  `confirmed` stages have been waited for.
    // All of the bookkeeping lives in (warp-uniform) registers: a FIFO of the outstanding stages (first granule and length,
    // 4 bits each, oldest in the low bits), a mask of the granules no unconfirmed stage occupies, and per activation slot
    // the number of the last stage that reads it.  This warp's own instruction path sits on the critical path whenever the
    // weight ring is too shallow for it to run ahead, so it must stay short.
    uint32_t cW_bits = 0;               // next phase parity to wait for, per stage barrier
    uint32_t issued = 0, confirmed = 0;
    uint64_t fifo_start = 0, fifo_len = 0;
    uint32_t free_mask = (1u << kWGranules) - 1u;
    uint32_t a_need[kNumASlots] = {0, 0};
    static_assert(kNumASlots == 2 && kWGranules <= 15, "producer bookkeeping is sized for 2 A slots and 4-bit granule indices");
    auto confirm_oldest = [&]() {
      const uint32_t j = static_cast<uint32_t>(fifo_start) & 15u, n = static_cast<uint32_t>(fifo_len) & 15u;
      mbar_wait(&emptyW[j], (cW_bits >> j) & 1u);
      cW_bits ^= (1u << j);
      free_mask |= ((1u << n) - 1u) << j;
      fifo_start >>= 4;
      fifo_len >>= 4;
      ++confirmed;
    };
    auto ensure_stage = [&](uint32_t seq_p1) { while (confirmed < seq_p1) confirm_oldest(); };
    int sa = 0, gw = 0;
    const bool pf = (debug & 64) != 0;
    long long prof[4] = {0, 0, 0, 0};
    const long long pstart = pf ? clock64() : 0;
    for (int e = 0; e < num_entries; ++e) {
      const uint4 er = c_entry_rec[e];
      const int li = static_cast<int>(er.x & 0xFFFFF);
      const int tile_lo = static_cast<int>(er.y), tile_hi = static_cast<int>(er.z);
      const int rot = static_cast<int>(er.w & 0xFFFF), dep = static_cast<int>(er.w >> 16) - 1;
      const uint4 la = c_layer_rec[(li - layer0) * 2], lb = c_layer_rec[(li - layer0) * 2 + 1];
      const int n_cols = la.x & 0x1FF, num_chunks = (la.x >> 9) & 0x1F, w_taps = (la.x >> 19) & 0xF, col_groups = (la.x >> 23) & 0x1F;
      constexpr int tile_h = kTileH;
      const int w_row0 = static_cast<int>(la.z), a_c0 = static_cast<int>(la.w), a_wrap = static_cast<int>(lb.y);
      const int tiles_x = static_cast<int>(lb.x & 0xFFFF), tiles_y = static_cast<int>(lb.x >> 16);
      constexpr int a_bytes = kABytes;
      const CUtensorMap* tmA = &layers[li].tmA;
      const int tiles_per_img = tiles_x * tiles_y;
      const int num_work = (tile_hi - tile_lo) * col_groups;
      const int k32 = static_cast<int>((la.y >> 11) & 1);    // 64-byte weight rows (32 channels)
      const int tap_rows = k32 ? (n_cols >> 1) : n_cols;     // 128-byte units of one tap tile
      const int wbytes = w_taps * tap_rows * 128;            // one weight stage = w_taps tap tiles, fetched by ONE bulk copy
      const int g = (wbytes + kWGranule - 1) / kWGranule;    // W granules per stage
      const int wsteps = (w_taps == 4) ? 1 : 9 / w_taps;     // stages per K chunk (1 or 3; stride-2 layers: one stage of four taps)
      const int taps_per_chunk = (w_taps == 4) ? 4 : 9;      // tap tiles packed per (chunk, column group)
      const int v = static_cast<int>((blockIdx.x + grid - static_cast<unsigned int>(rot)) % grid);
      TL_MARK(0);
      // The entry's inputs may only be read once the entry it depends on is complete on every CTA that worked on it.  The
      // wait sits AFTER the first weight stage has been requested (weights do not depend on the previous layer), right
      // before the first activation load.
      unsigned int dep_need = 0;
      const unsigned int* dep_ctr = counters;
      if (dep >= 0) {  // only the CTAs that had work in the dependency announce it
        const uint4 dr = c_entry_rec[dep];
        const uint32_t dcg = (c_layer_rec[(static_cast<int>(dr.x & 0xFFFFF) - layer0) * 2].x >> 23) & 0x1F;
        const unsigned int dwork = (dr.z - dr.y) * dcg;
        dep_need = dwork < grid ? dwork : grid;
        dep_ctr = counters + dep * kCtrStride;
        if ((dr.x >> 21) & 1) {  // per-image announce (same tiles on the same CTAs in both entries): wait for this CTA's image only
          dep_need = static_cast<unsigned int>(tiles_per_img);
          dep_ctr += 1 + (v < num_work ? v / tiles_per_img : 0);
        }
      }
      // One look at the dependency's counter is issued NOW and consumed only when the first activation load is due: its L2
      // round trip overlaps the waits for a free activation slot / weight granules below.
      unsigned int early_seen = 0;
      if (dep >= 0 && v < num_work && lane == 0 && !(debug & 16)) early_seen = ld_acquire_gpu(dep_ctr);
      // the dependency's counter shows every CTA that worked on it
      auto dependency_wait = [&]() {
        PROF_T0(pf);
        if (lane == 0) {
          if (!(debug & 16) && early_seen < dep_need) wait_entry_done(dep_ctr, dep, dep_need);
          if (!(debug & 512)) asm volatile("fence.proxy.async.global;" ::: "memory");  // TMA (async proxy) reads after generic-proxy stores (bit 512: timing experiment)
          // tell this CTA's epilogue warps (they read residual carriers written by earlier entries): acquire.gpu above,
          // release.cta here, acquire.cta on their side -- causality order is transitive
          asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(const_cast<uint32_t*>(dep_flag))), "r"(e + 1) : "memory");
        }
        __syncwarp();
        PROF_ADD(pf, 0);
        TL_MARK(1);
      };
      for (int w = v; w < num_work; w += static_cast<int>(grid)) {
        const int tile = tile_lo + w / col_groups;
        const int n = tile / tiles_per_img;
        const int t2 = tile - n * tiles_per_img;
        const int ty = t2 / tiles_x;
        const int x0 = (t2 - ty * tiles_x) * kTileW;
        const int y0 = ty * tile_h;
        for (int c = 0; c < num_chunks; ++c) {
          const int ac = a_c0 + (c % a_wrap) * 64;
          { PROF_T0(pf); ensure_stage(sa == 0 ? a_need[0] : a_need[1]); PROF_ADD(pf, 1); }  // activation slot free (waits on older stages only)
          if (c == 0 && w == v) TL_MARK(14);
          const int sa_used = sa;
          if (++sa == kNumASlots) sa = 0;
          auto load_activations = [&]() {
            if (elect_one_sync()) {
              if (debug & 4) {  // experiment: no loads at all (MMAs run on whatever is in smem)
                mbar_arrive(&fullA[sa_used]);
              } else {
                mbar_arrive_expect_tx(&fullA[sa_used], a_bytes);
                tma_load_4d(smem + sa_used * kASlot, tmA, &fullA[sa_used], ac, x0 - 1, y0 - 1, n);
              }
            }
            __syncwarp();
          };
          // Chunk 0 of an item: weight stages are requested BEFORE the activations as long as the dependency is still
          // open (weights do not depend on the previous layer) and as long as the ring has room without waiting on one of
          // this item's own stages (those cannot complete before the activations arrive).
          bool a_done = (c != 0);
          if (c != 0) load_activations();
          // the entry's first activation load waits for the dependency (neighbour form: every item's first load)
          const bool gated = (c == 0 && dep >= 0 && w == v);
          for (int d = 0; d < wsteps; ++d) {
            // stage d of this chunk holds w_taps consecutive taps of the centre-first order: dx in {1,0,2}, dy in {1,0,2}.
            // Packed rows are [dx][dy][n]; a 9-tap stage is the whole block, a 3-tap stage one dx column, a 1-tap stage one tile.
            int tap_row;
            if (w_taps == 9 || w_taps == 4) tap_row = 0;
            else tap_row = ((d == 0) ? 1 : (d == 1 ? 0 : 2)) * 3;
            if (gw + g > kWGranules) gw = 0;
            const uint32_t gmask = ((1u << g) - 1u) << gw;
            { PROF_T0(pf);
            if (!a_done && (d > 0)) {  // (measured: polling the dependency to squeeze more weight stages in front of it does not pay)
              if (gated) dependency_wait();
              load_activations();
              a_done = true;
            }
            while ((free_mask & gmask) != gmask) confirm_oldest();  // stages complete in order: confirm the oldest until the granules are free
            PROF_ADD(pf, 2); }
            if (c == 0 && d == 0 && w == v) TL_MARK(15);
            if (elect_one_sync()) {
              if (debug & 4) {
                mbar_arrive(&fullW[gw]);
              } else {
                mbar_arrive_expect_tx(&fullW[gw], wbytes);
                const long long row = w_row0 + (static_cast<long long>(c * col_groups + (w % col_groups)) * taps_per_chunk + tap_row) * tap_rows;
                bulk_load_1d(smemW + gw * kWGranule, packed_w + row * 128, wbytes, &fullW[gw]);
              }
            }
            __syncwarp();
            {
              const uint32_t slot4 = 4u * (issued - confirmed);  // at most kWGranules stages are outstanding
              fifo_start |= static_cast<uint64_t>(gw) << slot4;
              fifo_len |= static_cast<uint64_t>(g) << slot4;
              free_mask &= ~gmask;
              ++issued;
              if (d == wsteps - 1) {  // the chunk's last stage also releases its activation tile
                if (sa_used == 0) a_need[0] = issued; else a_need[1] = issued;
              }
            }
            gw += g;
          }
          if (!a_done) {
            if (gated) dependency_wait();
            load_activations();
          }
        }
      }
    }
    if (pf && lane == 0) {
      prof[3] = clock64() - pstart;
      for (int i = 0; i < 4; ++i) g_conv_prof[blockIdx.x * 12 + i] = prof[i];
    }
  } else if (warp == 1) {
    // ================================================== MMA issuer ==================================================
    // Whole warp runs the loops (uniform address math), one elected lane issues.  Descriptor hi words are loop
    // invariant; a K-step / tap advance is one 32-bit add on the lo word.
    uint32_t fA_bits = 0, fW_bits = 0;  // phase parity per A slot / W granule (full barriers)
    uint32_t acc_bits = 0;              // phase parity of the two accumulator stages (tempty barriers)
    int acc_toggle = 0, last_hold = 0;
    int sa = 0, gw = 0;
    int it = 0;
    const bool pf = (debug & 64) != 0;
    long long prof[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    const long long pstart = pf ? clock64() : 0;
    for (int e = 0; e < num_entries; ++e) {
      const long long _tp = pf ? clock64() : 0;
      const uint4 er = c_entry_rec[e];
      const int li = static_cast<int>(er.x & 0xFFFFF), slot = static_cast<int>((er.x >> 20) & 1);
      const int tile_lo = static_cast<int>(er.y), tile_hi = static_cast<int>(er.z), rot = static_cast<int>(er.w & 0xFFFF);
      const uint4 la = c_layer_rec[(li - layer0) * 2];
      const int n_cols = la.x & 0x1FF, num_chunks = (la.x >> 9) & 0x1F, ksteps_last = (la.x >> 14) & 0x7;
      const int w_taps = (la.x >> 19) & 0xF, col_groups = (la.x >> 23) & 0x1F;
      const int acc_col0 = la.y & 0xFF, acc_first = (la.y >> 8) & 1, acc_hold = (la.y >> 9) & 1;
      const bool has_epi = ((la.y >> 10) & 1) != 0;  // deferred partial-sum layers have no epilogue: nothing to hand over
      const int num_work = (tile_hi - tile_lo) * col_groups;
      const int k32 = static_cast<int>((la.y >> 11) & 1);
      const int down_mode = kVgg ? static_cast<int>((la.y >> 12) & 3) : 0, down_c64 = kVgg ? static_cast<int>((la.y >> 14) & 7) : 1;
      const int g = (w_taps * n_cols * (k32 ? 64 : 128) + kWGranule - 1) / kWGranule;
      const uint32_t idesc = make_idesc_16(128, n_cols, 0, 0, ((la.y >> 17) & 1) != 0);
      const uint32_t b_dy = static_cast<uint32_t>(n_cols) * (k32 ? 4u : 8u);  // bytes of one tap tile >> 4
      const uint32_t b_hi = k32 ? smem_desc_hi_sw64(512) : smem_desc_hi(1024);
      const int v = static_cast<int>((blockIdx.x + grid - static_cast<unsigned int>(rot)) % grid);
      if (pf) prof[8] += clock64() - _tp + (v == 0x7fffffff ? n_cols + idesc : 0);  // entry parameter fetch (forces the loads to be complete)
      for (int w = v; w < num_work; w += static_cast<int>(grid), ++it) {
        // accumulator stage: a pass layer uses its image group's resident block; ordinary layers alternate
        const int as = acc_hold ? slot : (acc_toggle & 1);
        if (!acc_hold) ++acc_toggle;
        if (acc_hold != last_hold) {
          // switching between the double-buffered layout and the fixed dense-block layout: both stages must be drained
          { PROF_T0(pf); mbar_wait(&tempty[as ^ 1], ((acc_bits >> (as ^ 1)) & 1u) ^ 1u); PROF_ADD(pf, 4); }
          last_hold = acc_hold;
        }
        { PROF_T0(pf); mbar_wait(&tempty[as], ((acc_bits >> as) & 1u) ^ 1u); PROF_ADD(pf, 4); }
        tcgen05_fence_after();
        TL_MARK(2);
        const uint32_t d_tmem = tmem_base + as * kAccStride + acc_col0;
        const uint32_t smemW_addr = smem_u32(smemW);
        const bool no_mma = (debug & 2) != 0;
        for (int c = 0; c < num_chunks; ++c) {
          const int ksteps = (c == num_chunks - 1) ? ksteps_last : 4;
          { PROF_T0(pf); mbar_wait(&fullA[sa], (fA_bits >> sa) & 1u); PROF_ADD(pf, 5); }
          if (c == 0) TL_MARK(3);
          const uint32_t a_lo = smem_desc_lo(smem_u32(smem + sa * kASlot), 16);
          const bool fresh = acc_first && c == 0;  // the very first MMA of a fresh item overwrites the accumulators
          const long long _ti = pf ? clock64() : 0;
#define B200SR_CHUNK(T, H, K) issue_chunk<T, H, K>(d_tmem, a_lo, smemW_addr, b_dy, idesc, fresh, g, gw, fW_bits, fullW, emptyW, no_mma, b_hi)
#define B200SR_CHUNK_K(T, H)                                   \
  switch (ksteps) {                                            \
    case 4: B200SR_CHUNK(T, H, 4); break;                      \
    case 3: B200SR_CHUNK(T, H, 3); break;                      \
    case 2: B200SR_CHUNK(T, H, 2); break;                      \
    default: B200SR_CHUNK(T, H, 1); break;                     \
  }
          if (kVgg && w_taps == 4) {
            // forward: the chunk's unshuffle phase (py, px) keeps rows {1,2} / {0,1} for py = 0 / 1; data gradient (flipped taps): the
            // column group's phase keeps rows {0,1} / {1,2} -- i.e. selector = phase (forward) or phase ^ 3 (data gradient)
            const int phase = (down_mode == 1) ? c / down_c64 : (w % col_groups) / down_c64;
            issue_chunk_down((down_mode == 1) ? phase : (phase ^ 3), d_tmem, a_lo, smemW_addr, b_dy, idesc, fresh, g, gw, fW_bits, fullW, emptyW, b_hi);
          } else if (w_taps == 9) { B200SR_CHUNK_K(9, 2) } else { B200SR_CHUNK_K(3, 2) }
#undef B200SR_CHUNK_K
#undef B200SR_CHUNK
          if (pf) prof[9] += clock64() - _ti;  // MMA issue incl. the weight-stage waits of this chunk
          fA_bits ^= (1u << sa);
          if (++sa == kNumASlots) sa = 0;
        }
        if (has_epi) {
          if (elect_one_sync()) umma_commit(&tfull[as]);  // accumulators ready for the epilogue warps
          __syncwarp();
          TL_MARK(4);
          acc_bits ^= (1u << as);
        }
      }
    }
    if (pf && lane == 0) {
      prof[7] = clock64() - pstart;
      for (int i = 4; i < 8; ++i) g_conv_prof[blockIdx.x * 12 + i] = prof[i];
      g_conv_prof[blockIdx.x * 12 + 11] = it;
      g_conv_prof[160 * 12 - 320 + blockIdx.x * 2] = prof[8];
      g_conv_prof[160 * 12 - 320 + blockIdx.x * 2 + 1] = prof[9];
    }
  } else if (warp == 10) {
    // =================================================== signaller ==================================================
    // Announces "this CTA's part of entry e is stored" on the entry's completion counter.  The gpu-scope fence (which
    // has to wait for the epilogue warps' stores to reach L2) runs here, off the epilogue's serial path; the mbarrier
    // hand-over (release.cta arrive / acquire.cta wait) plus fence cumulativity orders those stores before the atomic.
    const long long sc0 = clock64();
    const unsigned long long sg0 = globaltimer_ns();
    for (int e = 0; e < num_entries; ++e) {
      const uint4 er = c_entry_rec[e];
      const uint4 la = c_layer_rec[(static_cast<int>(er.x & 0xFFFFF) - layer0) * 2];
      const uint32_t cg = (la.x >> 23) & 0x1F;
      const bool has_epi = ((la.y >> 10) & 1) != 0;  // a partial-sum (filler) layer stores nothing: nothing to announce
      const unsigned int num_work = (er.z - er.y) * cg;
      const unsigned int v = (blockIdx.x + grid - (er.w & 0xFFFF)) % grid;
      mbar_wait(&sig[e & 1], (e >> 1) & 1);
      TL_MARK(11);
      if (lane == 0) {
        if (has_epi && v < num_work) {  // CTAs without work in this entry have nothing to publish and are not counted
          // release: the epilogue warps' stores (ordered before this thread by the mbarrier hand-over) become visible at gpu
          // scope before the counter update -- one red.release instead of __threadfence() (fence.sc) + atomicAdd
          // (same-box A/B: 12.14 -> 12.08 ms/step; bit 256 of the timing probes: plain relaxed add)
          unsigned int* ctr = counters + e * kCtrStride;
          if ((er.x >> 21) & 1) {  // per-image announce: one tile per CTA, image = tile / tiles of an image
            const uint32_t txy = c_layer_rec[(static_cast<int>(er.x & 0xFFFFF) - layer0) * 2 + 1].x;
            ctr += 1 + v / ((txy & 0xFFFF) * (txy >> 16));
          }
          if (debug & 256) atomicAdd(ctr, 1u);
          else asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
        }
        *sig_done = e + 1;
      }
      TL_MARK(7);
      __syncwarp();
    }
    if ((debug & 128) && blockIdx.x == 0 && lane == 0 && num_entries > 100) {  // SM clock actually sustained: cycles and ns of the whole launch
      g_conv_prof[160 * 12 - 16] = clock64() - sc0;
      g_conv_prof[160 * 12 - 15] = globaltimer_ns() - sg0;
    }
  } else {
    // =================================================== epilogue ===================================================
    // Eight warps; warps 2-5 own the upper 128-pixel half of every work item, warps 6-9 the lower half.  Layer
    // parameters + bias are staged in two smem slots private to these warps (the next entry is prefetched while the
    // current one runs); they synchronise among themselves with named barrier 1.
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    const int m = q * 32 + lane;
    const int half = (warp >= 6) ? 1 : 0;
    const int et = threadIdx.x - 64;  // 0..255
    // Stage entry e's layer parameters + bias into ring slot (e & 3) with cp.async: no register round trip, so the L2
    // latency never sits on this role's serial path (entries are staged two ahead).  What to fetch comes from the
    // constant-memory records.
    auto stage_entry = [&](int e) {
      if (e < num_entries) {
        const int li = static_cast<int>(c_entry_rec[e].x & 0xFFFFF);
        const uint4 lb = c_layer_rec[(li - layer0) * 2 + 1];
        const int nt = static_cast<int>(lb.w);      // bias floats the epilogue reads
        const uint32_t boff = lb.z;                 // bias byte offset from the packed buffer + 1 (0: no bias)
        if (et < static_cast<int>(sizeof(ConvParams) / 16)) {
          cp_async_16(sp_base + (e & 3) * 384 + et * 16, reinterpret_cast<const uint8_t*>(&layers[li].p) + et * 16);
        } else if (et >= 64 && et < 64 + kBiasSlot / 4) {
          const int i = et - 64;
          if (4 * i < nt) {
            uint8_t* dst = reinterpret_cast<uint8_t*>(sbias_base + (e & 3) * kBiasSlot) + i * 16;
            if (boff) cp_async_16(dst, packed_w + (boff - 1) + i * 16);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
      cp_async_commit();
    };
    stage_entry(0);
    stage_entry(1);
    int it = 0;
    uint32_t acc_bits = 0;  // phase parity of the two accumulator stages (tfull barriers)
    int acc_toggle = 0;
    const bool pf = (debug & 64) != 0;
    long long prof[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    const long long pstart = pf ? clock64() : 0;
    for (int e = 0; e < num_entries; ++e) {
      { PROF_T0(pf);
      cp_async_wait_group<1>();  // this thread's pieces of slot e have landed (only the group of e + 1 may be pending)
      if (et == 0) while (static_cast<int>(*sig_done) < e - 1) {}  // sig[e & 1] must have been consumed for entry e - 2
      epi_bar_sync();            // ... and everybody else's; every epilogue thread has left entry e - 1
      PROF_ADD(pf, 8); }
      if (warp == 2) TL_MARK(8);
      stage_entry(e + 2);        // ring slot (e + 2) & 3 was last read in entry e - 2
      {
        const uint4 la0 = c_layer_rec[(static_cast<int>(c_entry_rec[e].x & 0xFFFFF) - layer0) * 2];
        if (((la0.y >> 10) & 1) == 0) {  // partial-sum (filler) layer: no epilogue, only the hand-over to the signaller
          __syncwarp();
          if (lane == 0) mbar_arrive(&sig[e & 1]);
          continue;
        }
      }
      const ConvParams& p = *reinterpret_cast<const ConvParams*>(sp_base + (e & 3) * 384);
      const ConvEpilogue& ep = p.epi;
      const HW hw{p.H, p.W, (debug & 8) != 0};
      const uint4 er = c_entry_rec[e];
      const int ent_tile_lo = static_cast<int>(er.y), ent_tile_hi = static_cast<int>(er.z);
      const int ent_rot = static_cast<int>(er.w & 0xFFFF), ent_dep = static_cast<int>(er.w >> 16) - 1, ent_slot = static_cast<int>((er.x >> 20) & 1);
      const float* sbias = sbias_base + (e & 3) * kBiasSlot;
      const int tiles_per_img = p.tiles_x * p.tiles_y;
      const int num_work = (ent_tile_hi - ent_tile_lo) * p.col_groups;
      const int v = static_cast<int>((blockIdx.x + grid - static_cast<unsigned int>(ent_rot)) % grid);
      if (v < num_work && ent_dep >= 0 && p.epi_cols > 0) {
        // residuals written by earlier entries are read before the accumulator is ready: wait until the producer warp has
        // seen this entry's dependency complete (it must anyway before it can load the entry's activations)
        PROF_T0(pf);
        uint32_t seen;
        do {
          asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen) : "r"(smem_u32(const_cast<uint32_t*>(dep_flag))) : "memory");
        } while (static_cast<int>(seen) < e + 1);
        PROF_ADD(pf, 8);
      }
      if (warp == 2) TL_MARK(9);
      for (int w = v; w < ((p.epi_cols > 0) ? num_work : 0); w += static_cast<int>(grid), ++it) {
        const int tile = ent_tile_lo + w / p.col_groups;
        const int colbase = (w % p.col_groups) * p.n_cols;
        const int n = tile / tiles_per_img;
        const int t2 = tile - n * tiles_per_img;
        const int ty = t2 / p.tiles_x;
        const int x = (t2 - ty * p.tiles_x) * kTileW + (m & 7);
        // two-half items: this warp set owns half `half`; single-unit items: both warp sets see the same 128 pixels and
        // split the columns (set 0: columns 0-31, set 1: columns 32-63 if the epilogue has that many)
        const int y = ty * 32 + half * 16 + (m >> 3);
        const bool valid = (x < p.W) && (y < p.H);
        const int as = p.acc_hold ? ent_slot : (acc_toggle & 1);
        if (!p.acc_hold) ++acc_toggle;
        // Operands that do not depend on the accumulator are fetched BEFORE waiting for the MMAs, so their L2 latency
        // hides behind the tensor work: combined fp32 residual (<= 64 columns) and the LeakyReLU-derivative mask words.
        const bool pre = valid && !(debug & 1);
        const long long pix = (static_cast<long long>(n) * p.H + y) * p.W + x;
        // fp32 carriers are tile-blocked over 8 x 32 patches: a 16-row unit is half (ty & 1) of patch (n, ty / 2, tx)
        const long long cbase = carrier_base(tile, half, m);
        float res[32];
        uint32_t maskw[16];
        const bool has_res = (ep.r1 != nullptr) || (kVgg && ep.res_bf16 != nullptr);
        const bool has_mask = (ep.mask != nullptr);
        // residuals + mask words of 32 columns (only that many are held in registers at a time)
        auto prefetch_cols = [&](int c0) {
          if (kVgg && ep.res_bf16 != nullptr) {
            if (pre) {
              long long rpix; int rch;
              conv_store_dest<kVgg>(hw, ep, n, y, x, colbase + c0, rpix, rch);
              const uint4* rp = reinterpret_cast<const uint4*>(ep.res_bf16 + rpix * ep.res_bf16_stride + rch);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint4 r4 = __ldcg(rp + k);
                const bool hf = ep.f16 != 0;
                res[8 * k] = lo16_to_f32(r4.x, hf); res[8 * k + 1] = hi16_to_f32(r4.x, hf); res[8 * k + 2] = lo16_to_f32(r4.y, hf); res[8 * k + 3] = hi16_to_f32(r4.y, hf);
                res[8 * k + 4] = lo16_to_f32(r4.z, hf); res[8 * k + 5] = hi16_to_f32(r4.z, hf); res[8 * k + 6] = lo16_to_f32(r4.w, hf); res[8 * k + 7] = hi16_to_f32(r4.w, hf);
              }
            } else {
#pragma unroll
              for (int k = 0; k < 32; ++k) res[k] = 0.f;
            }
          } else if (pre && has_res) {
            const float* r1p = ep.r1 + cbase + ((colbase + c0) >> 2) * kCarrierChunkStride;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 r = __ldcg(reinterpret_cast<const float4*>(r1p + k * kCarrierChunkStride));
              res[4 * k] = ep.beta1 * r.x; res[4 * k + 1] = ep.beta1 * r.y; res[4 * k + 2] = ep.beta1 * r.z; res[4 * k + 3] = ep.beta1 * r.w;
            }
            if (ep.r2) {
              const float* r2p = ep.r2 + cbase + ((colbase + c0) >> 2) * kCarrierChunkStride;
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                const float4 r = __ldcg(reinterpret_cast<const float4*>(r2p + k * kCarrierChunkStride));
                res[4 * k] += ep.beta2 * r.x; res[4 * k + 1] += ep.beta2 * r.y; res[4 * k + 2] += ep.beta2 * r.z; res[4 * k + 3] += ep.beta2 * r.w;
              }
            }
          }
          if (pre && has_mask) {
            const uint4* mp = reinterpret_cast<const uint4*>(ep.mask + pix * ep.mask_stride + ep.mask_coff + colbase + c0);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint4 m4 = __ldcg(mp + k);
              maskw[4 * k] = m4.x; maskw[4 * k + 1] = m4.y; maskw[4 * k + 2] = m4.z; maskw[4 * k + 3] = m4.w;
            }
          }
        };
        if (0 < p.epi_cols) prefetch_cols(0);
        { PROF_T0(pf); mbar_wait(&tfull[as], (acc_bits >> as) & 1u); PROF_ADD(pf, 9); }
        if (warp == 2) TL_MARK(5);
        acc_bits ^= (1u << as);
        tcgen05_fence_after();
        const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * kAccStride + half * 128u + p.acc_col0;
        bool released = false;
        constexpr int kEpiGroups = kVgg ? 4 : 2;  // 32-column groups per work item: 64 columns, or 128 in the extended build (wide layers)
        // NOT unrolled: the epilogue's instruction footprint matters more than the loop overhead -- ncu's stall sampling shows ~15 % of the
        // epilogue warps' active samples waiting for instruction fetch (eleven warps of three roles share the SM's instruction caches)
#pragma unroll 1
        for (int gq = 0; gq < kEpiGroups; ++gq) {
          const int c0 = gq * 32;
          if (c0 < p.epi_cols) {
            float vv[32];
            const int ncol = (p.epi_cols - c0) >= 32 ? 32 : 16;
            if (__builtin_expect(ncol == 32, 1)) {
              uint32_t r[32];
              tmem_ld_32x32b_x32(t_addr + c0, r);
              tmem_ld_wait();
              if (warp == 2 && gq == 0) TL_MARK(10);
#pragma unroll
              for (int i = 0; i < 32; ++i) vv[i] = __uint_as_float(r[i]);
              if (c0 + 32 >= p.epi_cols) {  // last TMEM read of this warp set: release the accumulator before the global stores
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[as]);
                released = true;
              }
            } else {
              uint32_t r[16];
              tmem_ld_32x32b_x16(t_addr + c0, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) vv[i] = __uint_as_float(r[i]);
#pragma unroll
              for (int i = 16; i < 32; ++i) vv[i] = 0.f;
              tcgen05_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&tempty[as]);
              released = true;
            }
            if (warp == 2 && gq == 0) TL_MARK(12);
            float* feat_row = (kVgg && ep.feat_out && pre && ncol == 32) ? ep.feat_out + pix * ep.feat_stride + (colbase + c0) : nullptr;
            conv_epilogue_math<kVgg>(ep, sbias, res, has_res, maskw, has_mask, colbase + c0, ncol, vv, feat_row);
            // the residual / mask registers are free again: fetch the second 32 columns' while the first are stored
            if (kVgg ? ((gq + 1) * 32 < p.epi_cols) : (gq == 0 && 32 < p.epi_cols)) prefetch_cols((gq + 1) * 32);
            conv_epilogue_write<kVgg>(hw, ep, y_dyn, cbase, n, y, x, colbase + c0, vv, pre, lane);
            if (warp == 2 && gq == 0) TL_MARK(13);
          }
        }
        if (!released) {  // a warp set with no columns of its own still takes part in the accumulator hand-back
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[as]);
        }
      }
      // this warp's stores for entry e are issued: hand the announcement to the signaller warp
      __syncwarp();
      if (warp == 2) TL_MARK(6);
      if (lane == 0) mbar_arrive(&sig[e & 1]);
    }
    if (pf && threadIdx.x == 64) {
      prof[10] = clock64() - pstart;
      for (int i = 8; i < 11; ++i) g_conv_prof[blockIdx.x * 12 + i] = prof[i];
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_imm<kTmemCols>(tmem_base);
  }
}

}  // namespace b200sr
