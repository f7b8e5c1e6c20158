// libb200sr.so -- host side: network schedule ("plan"), TMA descriptor cache and the C ABI of include/b200sr.h.
//
// The plan turns the reference generator graph (ESRGAN/model.py:211-232 and its backward) into a flat list of
// kernel launches over caller-owned buffers:
//   forward : ingest -> conv1 -> 3*B dense blocks (5 convs each, writing channel slices of one dense buffer)
//             -> conv2 (+long skip) -> n_up phase-folded upsample convs -> conv3 -> conv4 (+clamp)
//   backward: the mirror image; every data-gradient is the SAME implicit-GEMM kernel over transposed/flipped
//             weights reading a dense gradient buffer [dY5|dY4|dY3|dY2|dY1]; weight gradients are one tcgen05 GEMM
//             per dense block slice (pixel axis = reduction) with fp32 reductions into the flat gradient buffer.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200sr.h"
#include "aux_kernels.cuh"
#include "conv_kernel.cuh"
#include "optim_kernels.cuh"
#include "iqa_kernels.cuh"
#include "vgg_kernels.cuh"
#include "disc_kernels.cuh"
#include "wgrad_kernel.cuh"

using namespace b200sr;

// ------------------------------------------------------------------------------------------------ error plumbing
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                            \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return fail(B200SR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int g_num_sms = 0;              // SM count of the device of the LAST runtime_init() call (every entry point calls it first)
static int g_dev_sms[64] = {0};        // per device: SM count, and whether the >48 KB dynamic shared memory opt-in has been set
static bool g_dev_attr_set[64] = {false};
static int g_ctas_per_sm = 1;
static int g_debug = 0;  // timing probes only (b200sr_debug_set)

static int runtime_init() {
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return fail(B200SR_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  // per DEVICE state: the compute-capability check, the SM count and the shared-memory opt-in (cudaFuncSetAttribute is per device)
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  const int di = dev & 63;
  if (!g_dev_sms[di]) {
    int major = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) return fail(B200SR_ERR_UNSUPPORTED, "libb200sr needs an sm_100 device (found sm_%d*)", major);
    CUDA_TRY(cudaDeviceGetAttribute(&g_dev_sms[di], cudaDevAttrMultiProcessorCount, dev));
  }
  g_num_sms = g_dev_sms[di];
  if (!g_dev_attr_set[di]) {
    CUDA_TRY(cudaFuncSetAttribute(conv3x3_chain_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, conv_smem_bytes(1)));
    CUDA_TRY(cudaFuncSetAttribute(conv3x3_chain_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, conv_smem_bytes(1)));
    CUDA_TRY(cudaFuncSetAttribute(conv3x3_chain_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, conv_smem_bytes(1)));
    CUDA_TRY(cudaFuncSetAttribute(wgrad3x3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemBytes));
    CUDA_TRY(cudaFuncSetAttribute(wgrad3x3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemBytes));
    g_dev_attr_set[di] = true;
  }
  return 0;
}

// NHWC bf16 activation map: dims (C, W, H, N), box (64, 10 | 8, rows, 1), 128B swizzle, zero OOB fill.
static int encode_act_map(CUtensorMap* m, void* base, int c_valid, int c_pix, int n, int h, int w, int box_rows, int box_w_in = -1) {
  const int box_w = box_w_in > 0 ? box_w_in : ((box_rows == kABoxRows) ? kABoxW : kTileW);  // conv tiles carry the horizontal halo, wgrad tiles do not
  cuuint64_t dims[4] = {(cuuint64_t)c_valid, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c_pix * 2, (cuuint64_t)w * c_pix * 2, (cuuint64_t)h * w * c_pix * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_w, (cuuint32_t)box_rows, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(B200SR_ERR_CUDA, "cuTensorMapEncodeTiled(act c=%d/%d n=%d h=%d w=%d) failed: %d", c_valid, c_pix, n, h, w, (int)r);
  return 0;
}
// packed weights: [rows][64] bf16, box (64, n_cols)
static int encode_w_map(CUtensorMap* m, void* base, long long rows, int n_cols) {
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)n_cols};
  cuuint32_t es[2] = {1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(B200SR_ERR_CUDA, "cuTensorMapEncodeTiled(weights rows=%lld n=%d) failed: %d", rows, n_cols, (int)r);
  return 0;
}

// ------------------------------------------------------------------------------------------------------ the plan
enum RefKind { RK_NULL = 0, RK_WS, RK_PACKED, RK_Y, RK_DY, RK_GRADS };
struct Ref {
  int kind = RK_NULL;
  long long off = 0;  // bytes
};
static Ref ws(long long off) { Ref r; r.kind = RK_WS; r.off = off; return r; }

struct ActMapSpec { long long off; int c_valid, c_pix, n, h, w, box_rows, box_w; };
struct Bases { void* ws; void* packed; void* y; const void* dy; void* grads; };

enum StepType { ST_CONV, ST_CHAIN, ST_WGRAD, ST_BIASGRAD, ST_UNPACK, ST_ADD, ST_MEMSET, ST_INGEST_X, ST_INGEST_DY,
                ST_VGG_INGEST, ST_VGG_POOL, ST_VGG_POOL_BWD,
                ST_DISC_UP, ST_DISC_UP_BWD, ST_DISC_ADD, ST_DISC_MASK, ST_DISC_INGEST_DY, ST_DISC_UNPACK,
                ST_TRUNK_INGEST, ST_TRUNK_EXPORT };

struct Step {
  int type = ST_CONV;
  // conv
  int amap = -1, wmap = -1;  // wmap: index into {16,32,64,128}
  ConvParams cp;
  Ref bias, mask, r1, r2, of, ofb, ob, cm, feat, resb;
  int pn = 0, ph = 0, pw = 0, pc = 0;  // VGG pool steps: geometry of the pooled layer's input
  dim3 grid;
  int smem = 0;
  int layer0 = 0, nlayers = 0, chain_grid = 0;  // ST_CHAIN: range of the plan's layer list
  int entry0 = 0, nentries = 0;                 // ... and of its entry list (filled when the device tables are built)
  // wgrad
  int xmap = -1, dymap = -1;
  WgradBatch wb;
  Ref seg_out[5];                 // bias-grad kernel outputs
  Ref wseg_out[kWgMaxProblems][kWgMaxSeg];  // wgrad batch outputs
  // bias grad
  BiasGradParams bp;
  Ref bg_g;
  int det_blocks = 0;  // deterministic plans: blocks (= partial-sum rows) of the bias-gradient launch, fixed at plan build
  // fold / add / memset / ingest
  Ref a, b, c, d2;
  long long count = 0;
  int i0 = 0, i1 = 0;
  float scale = 1.f;  // ST_TRUNK_INGEST: factor of the bf16 shadow
  // gradient-bucket announcement after this step
  long long cb_off = 0, cb_count = 0;
  bool needs_dx = false;  // only launched when the caller asks for the gradient w.r.t. the LR input
  bool needs_wgrad = false;  // discriminator plans: only launched when the caller asks for the parameter gradients
  // generator backward, for b200sr_backward_select: the dense block a data-gradient conv belongs to (R: the HR tail), and the
  // convs [wc0, wc1) whose parameter gradients a weight- / bias-gradient / carrier-sum step serves
  int blk = -1;
  int wc0 = 0, wc1 = 0;
};

struct b200sr_plan {
  b200sr_net_desc d;
  int R = 0;  // dense blocks
  int L = 0;  // upsample stages
  bool trunk = false;  // trunk plan (b200sr.h "Trunk plans"): the dense blocks alone, no conv1 / long skip / tail
  int t0 = 1;          // state_dict conv index of the first trunk conv (0 in trunk plans)
  bool unclamped = false;  // unclamped generator plan (b200sr.h "Unclamped plans"): y = conv4's output, no CMASK, dy ingested unmasked
  int xin_stride = 64;
  long long ws_bytes = 0;
  long long total_rows = 0, bias_floats = 0, packed_bytes = 0;
  std::vector<long long> param_off;  // flat fp32 offsets, 2 per conv (+ end)
  std::vector<PackOp> pack_ops;
  std::vector<BiasOp> bias_ops;
  std::vector<ActMapSpec> map_specs;
  std::vector<Step> fwd, bwd;
  // buffers (byte offsets into the workspace)
  long long o_xin = 0, o_t0 = 0, o_tr = 0, o_c1 = 0, o_c2 = 0, o_splt = 0, o_splc = 0, o_cmask = 0;
  std::vector<long long> o_dense, o_spl;
  long long o_dyp = 0, o_g3 = 0, o_gt = 0, o_gtb = 0, o_gr = 0, o_gc1 = 0, o_gc2 = 0, o_go1 = 0;
  std::vector<long long> o_dyb;      // output-gradient buffers [dY5|dY4|dY3|dY2|dY1] of the dense blocks, one per block: the whole
                                      // backward is ONE data-gradient chain, the weight gradients run after it
  cudaStream_t side_stream[3] = {nullptr, nullptr, nullptr};  // extra streams for the weight-gradient launches (tails / heads overlap)
  cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr};
  std::vector<long long> o_gu;
  int bwd_overlap_chain = -1;          // index in `bwd` of the trunk data-gradient chain the tail's weight gradients run beside (-1: none)
  bool tail_f16 = false;              // conv2 / upsampling / conv3 / conv4 as ONE fp16 product each instead of three split-bf16 products:
                                      // default for inference plans; training plans keep the split form (B200SR_TAIL_FP16=0/1 overrides)
  bool reassoc = true;                // dense blocks re-associated by input slice ("windowed": convs 1-4 resident in TMEM, 128 columns per
                                      // 128-pixel half, conv5 spread over filler layers); B200SR_REASSOC=0 or a frame with more 8x32 items
                                      // per image than SMs: plain per-conv schedule
  int groups = 1;                     // image groups that flow through a chain independently
  int plan_sms = 148;                 // SM count the schedule was laid out for
  bool det = false;                   // deterministic plan: ordered partial sums instead of atomics (b200sr.h "Deterministic plans")
  long long o_det = 0, det_lane_bytes = 0;  // its partial-sum area: one lane of det_lane_bytes per weight-gradient stream
  // VGG19 feature plans (b200sr_vgg_plan_create): the same step / chain machinery over another layer list
  bool is_vgg = false;
  b200sr_vgg_desc vd;
  long long o_vgg_feat[16] = {0}, o_vgg_g[16] = {0};  // fp32 pre-activation features / bf16 output gradients per conv (0: absent)
  int vgg_h[16] = {0}, vgg_w[16] = {0};
  // U-Net discriminator plans (b200sr_disc_plan_create)
  bool is_disc = false;
  b200sr_disc_desc dd;
  long long gw_bytes = 0;
  long long o_gw = 0;                 // staged weight gradients, per conv [tap][ci][co_pad] fp32
  std::vector<long long> gw_off;      // float offsets per conv into the staging buffer
  std::vector<UnpackOp> unpack_ops;   // one per conv, conv order
  UnpackOp* d_unpack_ops = nullptr;
  struct NamedBuf { std::string name; long long off, bytes; };
  std::vector<NamedBuf> named_bufs;   // workspace tensors by name (b200sr_debug_buffer)
  // device-side tables + descriptor cache
  PackOp* d_pack_ops = nullptr;
  BiasOp* d_bias_ops = nullptr;
  const float** d_params = nullptr;
  // TMA descriptors and the device layer list hold absolute addresses: one cached set per (workspace, packed) address pair, a few
  // of them (least recently used is replaced) -- callers whose allocator hands out alternating blocks (several forwards in flight,
  // the three discriminator passes of a GAN step) do not re-encode on every call
  struct MapSlot { void* ws = nullptr; void* packed = nullptr; std::vector<CUtensorMap> maps; LayerDesc* d_layers = nullptr; unsigned long long stamp = 0; };
  static constexpr int kMapSlots = 4;
  MapSlot slots[kMapSlots];
  int cur_slot = 0;
  unsigned long long slot_clock = 0;
  long long map_encodes = 0;  // cache misses so far (b200sr_debug: B200SR_TRACE=1 prints them)
  const std::vector<CUtensorMap>& maps() const { return slots[cur_slot].maps; }
  std::vector<Step> layer_steps;      // every conv launch of fwd then bwd, in execution order (= layer list)
  std::vector<LayerDesc> h_layers;
  LayerDesc* d_layers() const { return slots[cur_slot].d_layers; }
  bool tables_ready = false;
  std::vector<EntryDesc> h_entries;   // (layer, image group) entries of every chain, chain after chain
  EntryDesc* d_entries = nullptr;
  uint4* d_layer_rec = nullptr;       // constant-memory images of the two tables (copied device -> constant per launch)
  uint4* d_entry_rec = nullptr;
  unsigned int* d_counters = nullptr; // per-entry completion counters of the chain being launched, followed by the per-item flags
  size_t counters_bytes = 0;          // 16 KB of counters + the largest chain's (entries x items) flag matrix
};

static int wmap_index(int n_cols) { return n_cols == 16 ? 0 : n_cols == 32 ? 1 : n_cols == 64 ? 2 : 3; }
static const int kWmapCols[4] = {16, 32, 64, 128};

static long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }

namespace {
struct Builder {
  b200sr_plan& P;
  long long cursor = 0;
  explicit Builder(b200sr_plan& p) : P(p) {}
  long long alloc(long long bytes) {
    long long o = cursor;
    cursor = align_up(cursor + bytes, 1024);
    return o;
  }
  // the same, and the tensor can be looked up by name (b200sr_debug_buffer)
  long long alloc(const std::string& name, long long bytes) {
    const long long o = alloc(bytes);
    P.named_bufs.push_back({name, o, bytes});
    return o;
  }
  int add_map(long long off, int c_valid, int c_pix, int n, int h, int w, int box_rows, int box_w = -1) {
    for (size_t i = 0; i < P.map_specs.size(); ++i) {
      const ActMapSpec& s = P.map_specs[i];
      if (s.off == off && s.c_valid == c_valid && s.c_pix == c_pix && s.n == n && s.h == h && s.w == w && s.box_rows == box_rows &&
          s.box_w == box_w)
        return (int)i;
    }
    P.map_specs.push_back({off, c_valid, c_pix, n, h, w, box_rows, box_w});
    return (int)P.map_specs.size() - 1;
  }
  // packed rows for an op; returns row0
  int add_pack(PackOp op) {
    if (op.n_cols == 0) op.n_cols = op.n_total > 64 ? 64 : op.n_total;  // column groups of 64 (the upsample convs' four phases)
    op.row0 = (int)P.total_rows;
    P.total_rows += (long long)op.num_chunks * (op.down_c > 0 ? 4 : 9) * op.n_total / (op.k32 ? 2 : 1);  // 128-byte units
    P.pack_ops.push_back(op);
    return op.row0;
  }
  long long add_bias(int n, int b_index, int n_valid, int rep) {
    BiasOp b;
    b.off = (int)P.bias_floats;
    b.n = n; b.b_index = b_index; b.n_valid = n_valid; b.rep = rep;
    P.bias_floats += align_up(n, 4);
    P.bias_ops.push_back(b);
    return b.off;
  }
};

ConvParams base_conv_params(int n, int h, int w, int num_chunks, int ksteps_last, int a_c0, int a_wrap, int row0,
                            int n_cols, int n_total, int k32 = 0) {
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.N = n; p.H = h; p.W = w;
  p.tiles_x = (w + kTileW - 1) / kTileW;
  p.tiles_y = (h + kTileH - 1) / kTileH;
  p.num_tiles = n * p.tiles_x * p.tiles_y;
  p.num_chunks = num_chunks; p.ksteps_last = ksteps_last;
  p.a_c0 = a_c0; p.a_wrap = a_wrap;
  p.w_row0 = row0; p.n_cols = n_cols; p.n_total = n_total;
  p.col_groups = n_total / n_cols;
  p.k32 = k32;
  p.w_taps = (9 * n_cols * (k32 ? 64 : 128) <= 5 * kWGranule) ? 9 : 3;  // bytes per weight bulk copy <= 60 KB (n_cols <= 128: a dx column always fits)
  p.acc_col0 = 0; p.acc_first = 1; p.acc_hold = 0; p.epi_cols = n_cols; p.halves = 2;
  p.num_stages = conv_pick_stages(n_cols);
  p.epi.alpha = 1.f; p.epi.delta = 1.f; p.epi.beta1 = 1.f; p.epi.beta2 = 1.f;
  p.epi.res_stride = 64; p.epi.of_stride = 64;
  p.epi.store_mode = kStorePix;
  return p;
}

PackSeg seg(int k0, int klen, int w_index, int O, int I, int o_off, int i_off, int part) {
  PackSeg s; s.n0 = 0; s.nlen = 0; s.k0 = k0; s.klen = klen; s.w_index = w_index; s.O = O; s.I = I; s.o_off = o_off; s.i_off = i_off; s.part = part;
  return s;
}
PackSeg nseg(int n0, int nlen, int k0, int klen, int w_index, int O, int I, int o_off, int i_off) {  // segment limited to output columns [n0, n0+nlen)
  PackSeg s = seg(k0, klen, w_index, O, I, o_off, i_off, 0);
  s.n0 = n0; s.nlen = nlen;
  return s;
}
}  // namespace

// conv index helpers (state_dict order)
static int conv_index_rdb(const b200sr_plan& P, int r, int k /*1..5*/) { return P.t0 + r * 5 + (k - 1); }

static void conv_dims(const b200sr_plan& P, int ci, int* O, int* I) {
  const b200sr_net_desc& d = P.d;
  const int ntrunk = P.R * 5;
  if (ci < P.t0) { *O = d.channels; *I = d.in_channels; return; }
  if (ci < P.t0 + ntrunk) {
    const int k = (ci - P.t0) % 5 + 1;
    *O = (k < 5) ? d.growth : d.channels;
    *I = d.channels + d.growth * (k - 1);
    return;
  }
  const int t = ci - ntrunk - 1;  // 0: conv2, 1..L: up, L+1: conv3, L+2: conv4
  *I = d.channels;
  *O = (t == P.L + 2) ? d.out_channels : d.channels;
}

// SM count of the current device, 0 without one (plans built on a machine without a GPU lay out for 148)
static int device_sms() {
  int dev_count = 0, sms = 0;
  if (cudaGetDeviceCount(&dev_count) == cudaSuccess && dev_count > 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  } else {
    cudaGetLastError();
  }
  return sms;
}

static void plan_deterministic(b200sr_plan& P, int lanes, int wgrad_sms);

static int build_plan(b200sr_plan& P) {
  const b200sr_net_desc& d = P.d;
  if (d.channels != 64 || d.growth != 32) return fail(B200SR_ERR_INVALID, "only channels=64, growth=32 are supported (got %d, %d)", d.channels, d.growth);
  if (d.in_channels < 1 || d.in_channels > 64) return fail(B200SR_ERR_INVALID, "in_channels must be in [1,64]");
  if ((d.out_channels < 1 || d.out_channels > 16) && !P.trunk) return fail(B200SR_ERR_INVALID, "out_channels must be in [1,16]");
  if (d.num_blocks < 1 || d.n_up < 0 || d.n_up > 3) return fail(B200SR_ERR_INVALID, "bad num_blocks / n_up");
  if (d.batch < 1 || d.height < 1 || d.width < 1) return fail(B200SR_ERR_INVALID, "bad geometry");
  if (P.trunk && (d.n_up != 0 || d.in_channels != 64 || d.out_channels != 64))
    return fail(B200SR_ERR_INVALID, "a trunk plan needs n_up = 0 and in_channels = out_channels = 64 (got %d, %d, %d)", d.n_up,
                d.in_channels, d.out_channels);
  P.R = 3 * d.num_blocks;
  P.L = d.n_up;
  P.t0 = P.trunk ? 0 : 1;
  {
    // Image groups: >= 2 whenever the batch allows (latency hiding between groups).  The re-associated dense block keeps
    // one work item's partial sums in a CTA's TMEM across five passes, so every group must fit one item per CTA.
    const int sms = device_sms();
    if (sms > 0) P.plan_sms = sms;
    const int tpi = ((d.width + kTileW - 1) / kTileW) * ((d.height + kTileH - 1) / kTileH);  // resident 8 x 32 items per image
    P.groups = d.batch >= 2 ? 2 : 1;
    if (P.reassoc) {
      int g = P.groups;
      while (g <= d.batch && ((d.batch + g - 1) / g) * tpi > P.plan_sms) ++g;
      if (g <= d.batch) P.groups = g; else P.reassoc = false;  // a single image already exceeds one item per CTA
    }
  }
  const int R = P.R, L = P.L;
  const bool train = d.training != 0;
  const int N = d.batch, H = d.height, W = d.width;
  const long long Ppix = (long long)N * H * W;
  const bool trunk = P.trunk;
  const int nconv = trunk ? R * 5 : 1 + R * 5 + 1 + L + 2;
  const int ci_conv2 = 1 + R * 5, ci_up1 = ci_conv2 + 1, ci_conv3 = ci_conv2 + 1 + L, ci_conv4 = ci_conv3 + 1;  // (generator plans)

  // flat parameter offsets
  P.param_off.assign(2 * nconv + 1, 0);
  {
    long long off = 0;
    for (int c = 0; c < nconv; ++c) {
      int O, I;
      conv_dims(P, c, &O, &I);
      P.param_off[2 * c] = off; off += (long long)O * I * 9;
      P.param_off[2 * c + 1] = off; off += O;
    }
    P.param_off[2 * nconv] = off;
  }
  auto wref = [&](int c) { return ws(P.o_gw + P.gw_off[c] * 4); };  // weight gradients are staged, then unpacked
  auto bref = [&](int c) { Ref r; r.kind = RK_GRADS; r.off = P.param_off[2 * c + 1] * 4; return r; };

  Builder B(P);
  P.xin_stride = (int)align_up(3 * d.in_channels, 64);
  // ---- workspace layout (trunk plans keep only what the dense blocks read and write: the carriers TR / C1 / C2, the D buffers and,
  // for the backward, GR / GC1 / GC2, the DYB buffers and the weight-gradient staging)
  if (!trunk) P.o_xin = B.alloc("xin", Ppix * P.xin_stride * 2);
  // fp32 carriers: tile-blocked layout over the LR lattice's 8 x 32 tiles (padded to whole tiles)
  const long long carrier_bytes = (long long)N * ((W + kTileW - 1) / kTileW) * ((H + kTileH - 1) / kTileH) * kCarrierBytesPerTile;
  if (!trunk) P.o_t0 = B.alloc("T0", carrier_bytes);
  P.o_tr = B.alloc("TR", carrier_bytes);
  P.o_c1 = B.alloc("C1", carrier_bytes);
  P.o_c2 = B.alloc("C2", carrier_bytes);
  const int ndense = train ? R : 2;
  for (int i = 0; i < ndense; ++i) P.o_dense.push_back(B.alloc("D" + std::to_string(i), Ppix * 192 * 2));
  // tail activations: fp16 [pixels][64] (one fp16 product per conv), or the [hi | lo] bf16 pairs of the split-precision form
  // (training keeps a bf16 twin of every fp16 tail activation next to it, channels [64, 128): the weight-gradient GEMM pairs it with
  // the bf16 output gradients -- tcgen05 kind::f16 takes ONE 16-bit format for both operands, and the gradients stay bf16 for range)
  const bool tf16 = P.tail_f16;
  const int ts = (tf16 && !train) ? 64 : 128;  // channels per pixel of the tail activation buffers
  if (!trunk) {
    P.o_splt = B.alloc("SPLT", Ppix * ts * 2);
    for (int l = 0; l <= L; ++l) P.o_spl.push_back(B.alloc("SPL" + std::to_string(l), (Ppix << (2 * l)) * ts * 2));
    P.o_splc = B.alloc("SPLC", (Ppix << (2 * L)) * ts * 2);
  }
  const long long HRpix = Ppix << (2 * L);
  if (train) {
    if (!trunk) {
      if (!P.unclamped) P.o_cmask = B.alloc("CMASK", HRpix * d.out_channels);
      P.o_dyp = B.alloc("DYP", HRpix * 64 * 2);
      P.o_g3 = B.alloc("G3", HRpix * 64 * 2);
    }
    P.o_gu.assign(L + 1, 0);
    for (int l = 1; l <= L; ++l) P.o_gu[l] = B.alloc("GU" + std::to_string(l), (Ppix << (2 * (l - 1))) * 256 * 2);
    {
      // weight-gradient staging: per conv [9][ci][co_pad] fp32 (upsample convs: the four phase kernels, co = 256)
      long long off = 0;
      int blocks = 0;
      P.gw_off.assign(nconv, 0);
      for (int c = 0; c < nconv; ++c) {
        int O, I;
        conv_dims(P, c, &O, &I);
        const bool is_up = (c >= ci_up1 && c < ci_conv3);
        const int co_stage = is_up ? 256 : (int)align_up(O, 4);
        P.gw_off[c] = off;
        UnpackOp u;
        u.src_off = off; u.dst_off = P.param_off[2 * c]; u.co = O; u.ci = I; u.co_pad = co_stage; u.fold = is_up ? 1 : 0;
        u.block0 = blocks; u.nblocks = ((O + 31) / 32) * ((I + 31) / 32);
        blocks += u.nblocks;
        P.unpack_ops.push_back(u);
        off += align_up(9LL * I * co_stage, 4);
      }
      P.o_gw = B.alloc(off * 4);
      P.gw_bytes = off * 4;
    }
    if (!trunk) {
      P.o_gt = B.alloc("GT", carrier_bytes);
      P.o_gtb = B.alloc("GTB", Ppix * 64 * 2);
    }
    P.o_gr = B.alloc("GR", carrier_bytes);
    P.o_gc1 = B.alloc("GC1", carrier_bytes);
    P.o_gc2 = B.alloc("GC2", carrier_bytes);
    if (!trunk) P.o_go1 = B.alloc("GO1", Ppix * 64 * 2);
    P.o_dyb.assign(R, 0);
    for (size_t i = 0; i < P.o_dyb.size(); ++i) P.o_dyb[i] = B.alloc("DYB" + std::to_string(i), Ppix * 192 * 2);
  }
  P.ws_bytes = B.cursor;

  auto dense_off = [&](int r) { return P.o_dense[train ? r : (r & 1)]; };
  auto conv_step = [&](int amap, const ConvParams& cp, int grid_y) {
    Step s;
    s.type = ST_CONV;
    s.amap = amap;
    s.wmap = wmap_index(cp.n_cols);
    s.cp = cp;
    s.grid = dim3(1, grid_y, 1);
    s.smem = 0;
    return s;
  };
  auto packed_bias = [&](long long off_floats) { Ref r; r.kind = RK_PACKED; r.off = -1 - off_floats; return r; };  // fixed up later

  // ================================================================ forward ================================================================
  if (trunk) {  // the trunk input takes the place of conv1's output: fp32 carrier TR and its bf16 shadow in D0
    Step s; s.type = ST_TRUNK_INGEST; s.a = ws(P.o_tr); s.c = ws(dense_off(0)); s.b.kind = RK_NULL;
    P.fwd.push_back(s);
  } else {
    Step s; s.type = ST_INGEST_X;
    P.fwd.push_back(s);
  }
  // conv1: [hi|lo|hi] input, weights [w_hi|w_hi|w_lo]
  if (!trunk) {
    const int C = d.in_channels;
    PackOp op; memset(&op, 0, sizeof(op));
    op.n_total = 64; op.n_valid = 64; op.num_chunks = P.xin_stride / 64; op.mode = kPackFwd; op.nseg = 3;
    op.seg[0] = seg(0, C, 0, 64, C, 0, 0, 0);
    op.seg[1] = seg(C, C, 0, 64, C, 0, 0, 0);
    op.seg[2] = seg(2 * C, C, 0, 64, C, 0, 0, 1);
    const int row0 = B.add_pack(op);
    const int last_valid = 3 * C - 64 * (op.num_chunks - 1);
    ConvParams cp = base_conv_params(N, H, W, op.num_chunks, (last_valid + 15) / 16, 0, 1 << 20, row0, 64, 64);
    Step s = conv_step(B.add_map(P.o_xin, P.xin_stride, P.xin_stride, N, H, W, kABoxRows), cp, 1);
    s.bias = packed_bias(B.add_bias(64, 1, 64, 0));
    s.of = ws(P.o_t0); s.ofb = ws(P.o_tr);
    s.ob = ws(dense_off(0)); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 0;
    P.fwd.push_back(s);
  }
  // trunk
  const bool reassoc = P.reassoc;
  for (int r = 0; r < R; ++r) {
    const int j = r % 3;
    const long long D = dense_off(r);
    // epilogue of the block's last conv (conv5): residual scalings, fp32 carrier, bf16 shadow into the next dense buffer
    auto conv5_epilogue = [&](Step& s) {
      const long long cin_c = (j == 0) ? P.o_tr : (j == 1 ? P.o_c1 : P.o_c2);
      const long long cout_c = (j == 0) ? P.o_c1 : (j == 1 ? P.o_c2 : P.o_tr);
      s.cp.epi.alpha = (j == 2) ? 0.04f : 0.2f;
      s.r1 = ws(cin_c); s.cp.epi.beta1 = (j == 2) ? 0.2f : 1.f;
      if (j == 2) { s.r2 = ws(P.o_tr); s.cp.epi.beta2 = 1.f; }
      s.of = ws(cout_c);
      if (r < R - 1) {
        s.ob = ws(dense_off(r + 1)); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 0;
      } else if (!trunk) {  // (trunk plans: nothing reads a bf16 copy of the trunk output, the epilogue skips the store)
        s.ob = ws(P.o_splt); s.cp.epi.ob_stride = ts; s.cp.epi.ob_coff = 0; s.cp.epi.split_off = (ts == 128) ? 64 : 0;
        s.cp.epi.f16 = tf16;  // (only the STORE format: this layer's own operands are the trunk's bf16, mma_f16 stays 0)
      }
    };
    if (reassoc) {
      // WINDOWED re-association: passes 0..3 feed slice q (x, o1, o2, o3) to convs q+1..4 at once (N = 128, 96, 64, 32);
      // their partial sums (4 x 32 columns per 128-pixel half, so 8 x 32-pixel items and two resident image groups still
      // fit the 512 TMEM columns) stay in TMEM between the passes.  An SS tcgen05.mma costs ~(32 + N/4) cycles (shared-memory
      // operand reads), so a pass with N = 128 does four convs' worth of work in 1.6x the time of one.
      // conv5 (N = 64, K = 192) is SPREAD over the block: once the epilogues of passes 0 and 1 have taken conv1 / conv2 out,
      // accumulator columns [0, 64) are free, and conv5's contributions of the slices that already exist run there as
      // FILLER layers without epilogue -- F1 = x (emitted after pass 2), F2 = o1|o2 (after pass 3) -- which the MMA warp
      // works off while the other image group's next pass waits for its cross-CTA dependency.  Only the o3|o4 share (K = 64)
      // and the epilogue are left for the block's last layer.
      const int ci5 = conv_index_rdb(P, r, 5);
      auto conv5_piece = [&](int k0, int klen, bool first, bool last) {
        PackOp op; memset(&op, 0, sizeof(op));
        op.n_total = 64; op.n_cols = 64; op.n_valid = 64; op.num_chunks = 1; op.mode = kPackFwd; op.nseg = 1;
        op.seg[0] = seg(0, klen, 2 * ci5, 64, 192, 0, k0, 0);
        const int row0 = B.add_pack(op);
        ConvParams cp = base_conv_params(N, H, W, 1, klen / 16, k0, 1 << 20, row0, 64, 64);
        cp.acc_hold = 1; cp.acc_first = first ? 1 : 0; cp.acc_col0 = 0; cp.epi_cols = last ? 64 : 0;
        Step s = conv_step(B.add_map(D, k0 + klen, 192, N, H, W, kABoxRows), cp, 1);
        if (last) {
          s.bias = packed_bias(B.add_bias(64, 2 * ci5 + 1, 64, 0));
          conv5_epilogue(s);
        }
        P.fwd.push_back(s);
      };
      for (int q = 0; q < 4; ++q) {
        const int c_q = (q == 0) ? 0 : 64 + 32 * (q - 1);
        const int klen = (q == 0) ? 64 : 32;
        const int col_lo = 32 * q, ncols = 128 - col_lo;
        PackOp op; memset(&op, 0, sizeof(op));
        op.n_total = ncols; op.n_cols = ncols; op.n_valid = ncols; op.num_chunks = 1; op.mode = kPackFwd; op.nseg = 0;
        op.k32 = (klen == 32) ? 1 : 0;  // K = 32 pass layers carry 64-byte weight rows
        for (int k = q + 1; k <= 4; ++k)
          op.seg[op.nseg++] = nseg(32 * (k - 1) - col_lo, 32, 0, klen, 2 * conv_index_rdb(P, r, k), 32, 64 + 32 * (k - 1), 0, c_q);
        const int row0 = B.add_pack(op);
        ConvParams cp = base_conv_params(N, H, W, 1, klen / 16, c_q, 1 << 20, row0, ncols, ncols, op.k32);
        cp.acc_col0 = col_lo; cp.acc_first = (q == 0); cp.acc_hold = 1; cp.epi_cols = 32;
        Step s = conv_step(B.add_map(D, c_q + klen, 192, N, H, W, kABoxRows), cp, 1);
        s.bias = packed_bias(B.add_bias(32, 2 * conv_index_rdb(P, r, q + 1) + 1, 32, 0));
        s.cp.epi.act = 1;
        s.ob = ws(D); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 64 + 32 * q;
        P.fwd.push_back(s);
        if (q == 2) conv5_piece(0, 64, true, false);     // F1: x        (after pass 2; columns [0, 64) are free once pass 1's epilogue ran)
        if (q == 3) conv5_piece(64, 64, false, false);   // F2: o1 | o2  (after pass 3)
      }
      conv5_piece(128, 64, false, true);                 // o3 | o4 + epilogue
      continue;
    }
    for (int k = 1; k <= 5; ++k) {
      const int ci = conv_index_rdb(P, r, k);
      const int cin = 64 + 32 * (k - 1), cout = (k < 5) ? 32 : 64;
      PackOp op; memset(&op, 0, sizeof(op));
      op.n_total = cout; op.n_valid = cout; op.num_chunks = (cin + 63) / 64; op.mode = kPackFwd; op.nseg = 1;
      op.seg[0] = seg(0, cin, 2 * ci, cout, cin, 0, 0, 0);
      const int row0 = B.add_pack(op);
      ConvParams cp = base_conv_params(N, H, W, op.num_chunks, (cin - 64 * (op.num_chunks - 1)) / 16, 0, 1 << 20, row0, cout, cout);
      Step s = conv_step(B.add_map(D, cin, 192, N, H, W, kABoxRows), cp, 1);
      s.bias = packed_bias(B.add_bias(cout, 2 * ci + 1, cout, 0));
      if (k < 5) {
        s.cp.epi.act = 1;
        s.ob = ws(D); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 64 + 32 * (k - 1);
      } else {
        conv5_epilogue(s);
      }
      P.fwd.push_back(s);
    }
  }
  // tail convs (conv2, upsampling, conv3, conv4): ONE fp16 product (default), or the split-precision form -- input [hi|lo] 128-wide,
  // weights [w_hi|w_hi|w_lo], three bf16 products.  Pure bf16 misses the 5e-3 output bar (6.6e-3); fp16 operands measure 7.8e-4.
  const int tch = tf16 ? 1 : 3, twrap = tf16 ? (1 << 20) : 2, tsplit = (ts == 128) ? 64 : 0;
  const int tvalid = tf16 ? 64 : 128;  // channels of the tail buffers the forward convs read
  const int wg_c0 = tf16 ? 64 : 0;     // first channel of the bf16 operand the tail weight gradients read (twin copy / hi half)
  auto split_pack = [&](int ci, int n_total, int n_valid, int mode) {
    int O, I; conv_dims(P, ci, &O, &I);
    PackOp op; memset(&op, 0, sizeof(op));
    if (tf16) {  // ONE fp16 product: K = 64 in a single chunk
      op.n_total = n_total; op.n_valid = n_valid; op.num_chunks = 1; op.mode = mode; op.nseg = 1; op.f16 = 1;
      op.seg[0] = seg(0, 64, 2 * ci, O, I, 0, 0, 0);
      return B.add_pack(op);
    }
    op.n_total = n_total; op.n_valid = n_valid; op.num_chunks = 3; op.mode = mode; op.nseg = 3;
    op.seg[0] = seg(0, 64, 2 * ci, O, I, 0, 0, 0);
    op.seg[1] = seg(64, 64, 2 * ci, O, I, 0, 0, 0);
    op.seg[2] = seg(128, 64, 2 * ci, O, I, 0, 0, 1);
    return B.add_pack(op);
  };
  const int hH = H << L, hW = W << L;
  if (!trunk) {
    // conv2 (+ long skip)
    {
      const int row0 = split_pack(ci_conv2, 64, 64, kPackFwd);
      ConvParams cp = base_conv_params(N, H, W, tch, 4, 0, twrap, row0, 64, 64);
      Step s = conv_step(B.add_map(P.o_splt, tvalid, ts, N, H, W, kABoxRows), cp, 1);
      s.bias = packed_bias(B.add_bias(64, 2 * ci_conv2 + 1, 64, 0));
      s.r1 = ws(P.o_t0);
      s.ob = ws(P.o_spl[0]); s.cp.epi.ob_stride = ts; s.cp.epi.split_off = tsplit; s.cp.epi.f16 = tf16; s.cp.mma_f16 = tf16;
      P.fwd.push_back(s);
    }
    // upsample stages: nearest x2 + conv == 4 phase convs on the low-res lattice, pixel-shuffled on store
    for (int l = 1; l <= L; ++l) {
      const int ci = ci_up1 + (l - 1);
      const int h = H << (l - 1), w = W << (l - 1);
      const int row0 = split_pack(ci, 256, 256, kPackUpFwd);
      ConvParams cp = base_conv_params(N, h, w, tch, 4, 0, twrap, row0, 64, 256);  // 4 column groups (phases) of 64
      Step s = conv_step(B.add_map(P.o_spl[l - 1], tvalid, ts, N, h, w, kABoxRows), cp, 2);
      s.bias = packed_bias(B.add_bias(256, 2 * ci + 1, 64, 64));
      s.cp.epi.act = 1;
      s.cp.epi.store_mode = kStoreShuffle;
      s.ob = ws(P.o_spl[l]); s.cp.epi.ob_stride = ts; s.cp.epi.split_off = tsplit; s.cp.epi.f16 = tf16; s.cp.mma_f16 = tf16;
      P.fwd.push_back(s);
    }
    // conv3
    {
      const int row0 = split_pack(ci_conv3, 64, 64, kPackFwd);
      ConvParams cp = base_conv_params(N, hH, hW, tch, 4, 0, twrap, row0, 64, 64);
      Step s = conv_step(B.add_map(P.o_spl[L], tvalid, ts, N, hH, hW, kABoxRows), cp, 1);
      s.bias = packed_bias(B.add_bias(64, 2 * ci_conv3 + 1, 64, 0));
      s.cp.epi.act = 1;
      s.ob = ws(P.o_splc); s.cp.epi.ob_stride = ts; s.cp.epi.split_off = tsplit; s.cp.epi.f16 = tf16; s.cp.mma_f16 = tf16;
      P.fwd.push_back(s);
    }
    // conv4 + clamp (unclamped plans: conv4 alone)
    {
      const int row0 = split_pack(ci_conv4, 16, d.out_channels, kPackFwd);
      ConvParams cp = base_conv_params(N, hH, hW, tch, 4, 0, twrap, row0, 16, 16);
      Step s = conv_step(B.add_map(P.o_splc, tvalid, ts, N, hH, hW, kABoxRows), cp, 1);
      s.cp.epi.f16 = tf16; s.cp.mma_f16 = tf16;
      s.bias = packed_bias(B.add_bias(16, 2 * ci_conv4 + 1, d.out_channels, 0));
      s.cp.epi.store_mode = kStoreFinal;
      s.cp.epi.n_valid = d.out_channels;
      s.cp.epi.unclamped = P.unclamped;
      s.of.kind = RK_Y;
      if (train && !P.unclamped) s.cm = ws(P.o_cmask);
      P.fwd.push_back(s);
    }
  } else {  // the trunk output leaves as NCHW fp32
    Step s; s.type = ST_TRUNK_EXPORT; s.a = ws(P.o_tr);
    P.fwd.push_back(s);
  }

  // ================================================================ backward ===============================================================
  if (train) {
    // a wgrad launch = batch of problems over one (X, dY) tensor-map pair
    auto wgrad_batch = [&](long long x_off, int x_cvalid, int x_cpix, long long dy_off, int dy_cvalid, int dy_cpix, int n, int h, int w) {
      Step s; s.type = ST_WGRAD;
      s.xmap = B.add_map(x_off, x_cvalid, x_cpix, n, h, w, kWgXRows);
      s.dymap = B.add_map(dy_off, dy_cvalid, dy_cpix, n, h, w, kWgTileH);
      WgradBatch& wb = s.wb; memset(&wb, 0, sizeof(wb));
      wb.N = n; wb.H = h; wb.W = w;
      wb.tiles_x = (w + kTileW - 1) / kTileW; wb.tiles_y = (h + kWgTileH - 1) / kWgTileH; wb.num_tiles = n * wb.tiles_x * wb.tiles_y;
      return s;
    };
    auto add_problem = [&](Step& s, int a_c0, int b_c0, int n_cols, int a_blocks = 2) {
      WgradParams& wp = s.wb.prob[s.wb.num_problems++];
      wp.b_c0 = b_c0; wp.n_cols = n_cols; wp.n_blocks = (n_cols + 63) / 64;
      wgrad_set_a(wp, a_c0, a_blocks);
      return s.wb.num_problems - 1;
    };
    // packed problem: M block 0 = X channels [c0, c0 + 64) at tap dx0, block 1 = the same channels at tap dx1 (>= 0) or all ones (-1)
    auto add_packed = [&](Step& s, int c0, int dx0, int dx1, int b_c0, int n_cols) {
      WgradParams& wp = s.wb.prob[s.wb.num_problems++];
      wp.b_c0 = b_c0; wp.n_cols = n_cols; wp.n_blocks = (n_cols + 63) / 64;
      wp.blk[0].kind = kWgBlkX; wp.blk[0].c0 = c0; wp.blk[0].dx = dx0;
      wp.blk[1].kind = dx1 >= 0 ? kWgBlkX : kWgBlkOnes; wp.blk[1].c0 = c0; wp.blk[1].dx = dx1 >= 0 ? dx1 : 0;
      return s.wb.num_problems - 1;
    };
    auto add_seg = [&](Step& s, int cb, int ce, Ref out, int ci_total, int ci0, int co_pad, int blk_mask = 0) {  // to the LAST problem added
      const int pj = s.wb.num_problems - 1;
      WgradParams& wp = s.wb.prob[pj];
      WgradSegment& g = wp.seg[wp.num_seg];
      g.col_begin = cb; g.col_end = ce; g.out = nullptr; g.ci_total = ci_total; g.ci0 = ci0; g.co_pad = co_pad; g.blk_mask = blk_mask;
      s.wseg_out[pj][wp.num_seg] = out;
      wp.num_seg++;
    };
    auto wgrad_step = [&](long long x_off, int x_cvalid, int x_cpix, long long dy_off, int dy_cvalid, int dy_cpix, int n, int h, int w,
                          int a_c0, int b_c0, int n_cols) {  // single-problem launch
      Step s = wgrad_batch(x_off, x_cvalid, x_cpix, dy_off, dy_cvalid, dy_cpix, n, h, w);
      add_problem(s, a_c0, b_c0, n_cols, (x_cvalid - a_c0 > 64) ? 2 : 1);
      return s;
    };
    auto biasgrad_step = [&](long long g_off, long long npix, int stride, int c0, int ncols) {
      Step s; s.type = ST_BIASGRAD;
      memset(&s.bp, 0, sizeof(s.bp));
      s.bg_g = ws(g_off); s.bp.P = npix; s.bp.stride = stride; s.bp.c0 = c0; s.bp.ncols = ncols;
      return s;
    };
    auto add_bseg = [&](Step& s, int cb, int ce, Ref out, int n_valid) {
      BiasGradSeg& g = s.bp.seg[s.bp.nseg];
      g.col_begin = cb; g.col_end = ce; g.out = nullptr; g.n_valid = n_valid;
      s.seg_out[s.bp.nseg] = out;
      s.bp.nseg++;
    };
    auto unpack_step = [&](int c_begin, int c_end) {  // staged weight grads of convs [c_begin, c_end) -> flat buffer, then announce
      Step s; s.type = ST_UNPACK; s.i0 = c_begin; s.i1 = c_end;
      s.cb_off = P.param_off[2 * c_begin]; s.cb_count = P.param_off[2 * c_end] - s.cb_off;
      return s;
    };
    auto dgrad_pack1 = [&](int ci, int n_total, int klen) {  // plain single-conv dgrad: n = ci (64), k = co
      int O, I; conv_dims(P, ci, &O, &I);
      PackOp op; memset(&op, 0, sizeof(op));
      op.n_total = n_total; op.n_valid = n_total; op.num_chunks = (klen + 63) / 64; op.mode = kPackDgrad; op.nseg = 1;
      op.seg[0] = seg(0, klen, 2 * ci, O, I, 0, 0, 0);
      return B.add_pack(op);
    };
    {
      Step s; s.type = ST_MEMSET; s.a.kind = RK_GRADS; s.a.off = 0; s.count = P.param_off[2 * nconv] * 4;
      P.bwd.push_back(s);
      Step m; m.type = ST_MEMSET; m.a = ws(P.o_gw); m.count = P.gw_bytes;
      P.bwd.push_back(m);
      Step g; g.type = ST_INGEST_DY;
      if (trunk) {  // dy takes the place of conv2's data gradient: GR and the last dense block's dY5 = bf16(0.04 dy)
        g.type = ST_TRUNK_INGEST; g.a = ws(P.o_gr); g.c = ws(P.o_dyb[R - 1]); g.b.kind = RK_DY; g.scale = 0.04f;
      }
      P.bwd.push_back(g);
    }
    // Launch order inside one gradient bucket: all data-gradient convs first (they form ONE chain launch), then the
    // weight/bias-gradient kernels that consume what the chain produced, then the unpack + bucket announcement.
    std::vector<Step> seg_convs, seg_others;
    int cur_blk = R, cur_c0 = 0, cur_c1 = 0;  // what the steps emitted next belong to (set by serves())
    auto serves = [&](int blk, int c0, int c1) { cur_blk = blk; cur_c0 = c0; cur_c1 = c1; };
    auto emit = [&](Step st) {
      st.blk = cur_blk; st.wc0 = cur_c0; st.wc1 = cur_c1;
      if (st.type == ST_CONV) seg_convs.push_back(st); else seg_others.push_back(st);
    };
    if (!trunk) {  // the HR tail (trunk plans start at the last dense block: see the ingest above)
      // conv4: wgrad, bias grad, dgrad (-> G3, masked by lrelu'(conv3 out))
      {
        serves(R, ci_conv4, ci_conv4 + 1);
        Step w4 = wgrad_step(P.o_splc, wg_c0 + 64, ts, P.o_dyp, 16, 64, N, hH, hW, wg_c0, 0, 16);
        add_seg(w4, 0, 16, wref(ci_conv4), 64, 0, (int)align_up(d.out_channels, 4));
        emit(w4);
        Step b4 = biasgrad_step(P.o_dyp, HRpix, 64, 0, 16);
        add_bseg(b4, 0, 16, bref(ci_conv4), d.out_channels);
        emit(b4);
        const int row0 = dgrad_pack1(ci_conv4, 64, d.out_channels);
        ConvParams cp = base_conv_params(N, hH, hW, 1, 1, 0, 1 << 20, row0, 64, 64);
        Step s = conv_step(B.add_map(P.o_dyp, 16, 64, N, hH, hW, kABoxRows), cp, 1);
        s.mask = ws(P.o_splc); s.cp.epi.mask_stride = ts; s.cp.epi.mask_coff = 0;
        s.ob = ws(P.o_g3); s.cp.epi.ob_stride = 64;
        emit(s);
      }
      // conv3
      {
        serves(R, ci_conv3, ci_conv3 + 1);
        Step w3 = wgrad_step(P.o_spl[L], wg_c0 + 64, ts, P.o_g3, 64, 64, N, hH, hW, wg_c0, 0, 64);
        add_seg(w3, 0, 64, wref(ci_conv3), 64, 0, 64);
        emit(w3);
        Step b3 = biasgrad_step(P.o_g3, HRpix, 64, 0, 64);
        add_bseg(b3, 0, 64, bref(ci_conv3), 64);
        emit(b3);
        const int row0 = dgrad_pack1(ci_conv3, 64, 64);
        ConvParams cp = base_conv_params(N, hH, hW, 1, 4, 0, 1 << 20, row0, 64, 64);
        Step s = conv_step(B.add_map(P.o_g3, 64, 64, N, hH, hW, kABoxRows), cp, 1);
        if (L >= 1) {
          s.mask = ws(P.o_spl[L]); s.cp.epi.mask_stride = ts;
          s.ob = ws(P.o_gu[L]); s.cp.epi.ob_stride = 256; s.cp.epi.store_mode = kStoreUnshuffle;
        } else {
          s.of = ws(P.o_gt);
          s.ob = ws(P.o_gtb); s.cp.epi.ob_stride = 64;
        }
        emit(s);
      }
      // upsample stages, top down
      for (int l = L; l >= 1; --l) {
        const int ci = ci_up1 + (l - 1);
        const int h = H << (l - 1), w = W << (l - 1);
        const long long npix = Ppix << (2 * (l - 1));
        serves(R, ci, ci + 1);
        for (int half = 0; half < 2; ++half) {
          Step wu = wgrad_step(P.o_spl[l - 1], wg_c0 + 64, ts, P.o_gu[l], 256, 256, N, h, w, wg_c0, 128 * half, 128);
          Ref out = wref(ci);
          out.off += (long long)half * 32 * 64 * 4 * 4;  // 16-byte column chunks [32*half, +32) of the [tap][64 chunks][64 ci][4] staging tensor
          add_seg(wu, 0, 128, out, 64, 0, 256);
          emit(wu);
        }
        {
          Step bu = biasgrad_step(P.o_gu[l], npix, 256, 0, 256);
          for (int ph = 0; ph < 4; ++ph) add_bseg(bu, 64 * ph, 64 * ph + 64, bref(ci), 64);
          emit(bu);
        }
        PackOp op; memset(&op, 0, sizeof(op));
        op.n_total = 64; op.n_valid = 64; op.num_chunks = 4; op.mode = kPackUpDgrad; op.nseg = 1;
        op.seg[0] = seg(0, 256, 2 * ci, 64, 64, 0, 0, 0);
        const int row0 = B.add_pack(op);
        ConvParams cp = base_conv_params(N, h, w, 4, 4, 0, 1 << 20, row0, 64, 64);
        Step s = conv_step(B.add_map(P.o_gu[l], 256, 256, N, h, w, kABoxRows), cp, 1);
        if (l >= 2) {
          s.mask = ws(P.o_spl[l - 1]); s.cp.epi.mask_stride = ts;
          s.ob = ws(P.o_gu[l - 1]); s.cp.epi.ob_stride = 256; s.cp.epi.store_mode = kStoreUnshuffle;
        } else {
          s.of = ws(P.o_gt);
          s.ob = ws(P.o_gtb); s.cp.epi.ob_stride = 64;
        }
        emit(s);
      }
      // conv2
      {
        serves(R, ci_conv2, ci_conv2 + 1);
        Step w2 = wgrad_step(P.o_splt, wg_c0 + 64, ts, P.o_gtb, 64, 64, N, H, W, wg_c0, 0, 64);
        add_seg(w2, 0, 64, wref(ci_conv2), 64, 0, 64);
        emit(w2);
        Step b2 = biasgrad_step(P.o_gtb, Ppix, 64, 0, 64);
        add_bseg(b2, 0, 64, bref(ci_conv2), 64);
        emit(b2);
        const int row0 = dgrad_pack1(ci_conv2, 64, 64);
        ConvParams cp = base_conv_params(N, H, W, 1, 4, 0, 1 << 20, row0, 64, 64);
        Step s = conv_step(B.add_map(P.o_gtb, 64, 64, N, H, W, kABoxRows), cp, 1);
        s.of = ws(P.o_gr);
        s.ob = ws(P.o_dyb[R - 1]); s.cp.epi.ob_stride = 192; s.cp.epi.delta = 0.04f;
        emit(s);
        // tail bucket: conv2 .. conv4 are contiguous at the end of the flat buffer
        emit(unpack_step(ci_conv2, nconv));
      }
    }
    // The data-gradient chain is cut ONCE, behind the HR tail: the tail's weight / bias gradients (HR-sized, L2-heavy, 8 % of the
    // weight-gradient FLOPs but 12 % of their time) then run on the side streams WHILE the trunk chain -- latency-bound, launched on one
    // CTA per work item of an image group (128 of 148 SMs at config 2) -- walks the 69 dense blocks (run_steps defers them behind it).
    if (P.reassoc && P.groups >= 2) {
      for (const Step& c : seg_convs) P.bwd.push_back(c);
      for (const Step& o : seg_others) P.bwd.push_back(o);
      seg_convs.clear(); seg_others.clear();
    }
    // trunk, last dense block first
    int bucket_hi = P.t0 + 5 * R;  // conv index (exclusive) up to which trunk gradients have been announced
    for (int r = R - 1; r >= 0; --r) {
      const int j = r % 3;
      const long long D = P.o_dense[r];
      const long long DYc = P.o_dyb[r];
      const long long DYn = P.o_dyb[r > 0 ? r - 1 : 0];
      serves(r, conv_index_rdb(P, r, 1), conv_index_rdb(P, r, 5) + 1);
      // epilogue of the block-input (x) slice: fp32 gradient carriers and the next block's dY5
      auto xslice_epilogue = [&](Step& s) {
        if (j == 2) { s.r1 = ws(P.o_gr); s.cp.epi.beta1 = 0.2f; s.of = ws(P.o_gc2); s.cp.epi.delta = 0.2f; }
        else if (j == 1) { s.r1 = ws(P.o_gc2); s.of = ws(P.o_gc1); s.cp.epi.delta = 0.2f; }
        else { s.r1 = ws(P.o_gc1); s.r2 = ws(P.o_gr); s.of = ws(P.o_gr); s.cp.epi.delta = 0.04f; }
        if (r > 0) { s.ob = ws(DYn); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 0; }
      };
      if (P.reassoc) {
        // Mirror image of the windowed forward: passes 0..3 feed dY_{5-q} to the growth slices o_{4-q}..o_1 it reads
        // (accumulator columns [o4 | o3 | o2 | o1], N = 128, 96, 64, 32).  The block-input gradient (N = 64, K = 192 over
        // [dY5|dY4|dY3|dY2|dY1]) is spread like conv5 in the forward: filler layers G1 = dY5 (after pass 2), G2 = dY4|dY3
        // (after pass 3) accumulate into the freed columns [0, 64) while the other group's pass waits for its dependency; the
        // last layer adds dY2|dY1's share (K = 64) and runs the epilogue.
        auto xgrad_piece = [&](int k0, int klen, bool first, bool last) {  // dY channels [k0, k0 + klen) -> x-slice gradient
          PackOp op; memset(&op, 0, sizeof(op));
          op.n_total = 64; op.n_cols = 64; op.n_valid = 64; op.num_chunks = 1; op.mode = kPackDgrad; op.nseg = 0;
          for (int k = 5; k > 0; --k) {
            const int kc0 = (k == 5) ? 0 : 64 + 32 * (4 - k);   // dY_k inside [dY5|dY4|dY3|dY2|dY1]
            const int kcl = (k == 5) ? 64 : 32;
            if (kc0 < k0 || kc0 + kcl > k0 + klen) continue;
            op.seg[op.nseg++] = seg(kc0 - k0, kcl, 2 * conv_index_rdb(P, r, k), kcl, 64 + 32 * (k - 1), 0, 0, 0);
          }
          const int row0 = B.add_pack(op);
          ConvParams cp = base_conv_params(N, H, W, 1, klen / 16, k0, 1 << 20, row0, 64, 64);
          cp.acc_hold = 1; cp.acc_first = first ? 1 : 0; cp.acc_col0 = 0; cp.epi_cols = last ? 64 : 0;
          Step s = conv_step(B.add_map(DYc, k0 + klen, 192, N, H, W, kABoxRows), cp, 1);
          if (last) xslice_epilogue(s);
          emit(s);
        };
        for (int q = 0; q < 4; ++q) {
          const int kk = 5 - q;
          const int klen = (kk == 5) ? 64 : 32;
          const int a_c0 = (q == 0) ? 0 : 64 + 32 * (q - 1);
          const int ci = conv_index_rdb(P, r, kk);
          const int col_lo = 32 * q, ncols = 128 - col_lo;
          PackOp op; memset(&op, 0, sizeof(op));
          op.n_total = ncols; op.n_cols = ncols; op.n_valid = ncols; op.num_chunks = 1; op.mode = kPackDgrad; op.nseg = 0;
          op.k32 = (klen == 32) ? 1 : 0;
          for (int sidx = 4 - q; sidx >= 1; --sidx)
            op.seg[op.nseg++] = nseg(32 * (4 - sidx) - col_lo, 32, 0, klen, 2 * ci, klen, 64 + 32 * (kk - 1), 0, 64 + 32 * (sidx - 1));
          const int row0 = B.add_pack(op);
          ConvParams cp = base_conv_params(N, H, W, 1, klen / 16, a_c0, 1 << 20, row0, ncols, ncols, op.k32);
          cp.acc_col0 = col_lo; cp.acc_first = (q == 0); cp.acc_hold = 1; cp.epi_cols = 32;
          Step s = conv_step(B.add_map(DYc, a_c0 + klen, 192, N, H, W, kABoxRows), cp, 1);
          const int sl = 4 - q;  // completed slice o_sl
          s.mask = ws(D); s.cp.epi.mask_stride = 192; s.cp.epi.mask_coff = 64 + 32 * (sl - 1);
          s.ob = ws(DYc); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 64 + 32 * q;
          emit(s);
          if (q == 2) xgrad_piece(0, 64, true, false);     // G1: dY5
          if (q == 3) xgrad_piece(64, 64, false, false);   // G2: dY4 | dY3
        }
        xgrad_piece(128, 64, false, true);                 // dY2 | dY1 + epilogue
      } else
      for (int sl = 4; sl >= 0; --sl) {
        // gradient w.r.t. input slice sl (0: the 64-ch block input x, 1..4: growth outputs o_sl) = sum over consumer convs
        const int c_s = (sl == 0) ? 0 : 64 + 32 * (sl - 1);
        const int nsl = (sl == 0) ? 64 : 32;
        const int kin = 64 + 32 * (4 - sl);  // DY prefix [dY5 | dY4 | ... | dY_{sl+1}]
        PackOp op; memset(&op, 0, sizeof(op));
        op.n_total = nsl; op.n_valid = nsl; op.num_chunks = (kin + 63) / 64; op.mode = kPackDgrad;
        op.nseg = 0;
        for (int k = 5; k > sl; --k) {
          const int ci = conv_index_rdb(P, r, k);
          const int k0 = (k == 5) ? 0 : 64 + 32 * (4 - k);
          const int klen = (k == 5) ? 64 : 32;
          op.seg[op.nseg++] = seg(k0, klen, 2 * ci, klen, 64 + 32 * (k - 1), 0, c_s, 0);
        }
        const int row0 = B.add_pack(op);
        ConvParams cp = base_conv_params(N, H, W, op.num_chunks, (kin - 64 * (op.num_chunks - 1)) / 16, 0, 1 << 20, row0, nsl, nsl);
        Step s = conv_step(B.add_map(DYc, kin, 192, N, H, W, kABoxRows), cp, 1);
        if (sl > 0) {
          s.mask = ws(D); s.cp.epi.mask_stride = 192; s.cp.epi.mask_coff = c_s;
          s.ob = ws(DYc); s.cp.epi.ob_stride = 192; s.cp.epi.ob_coff = 64 + 32 * (4 - sl);
        } else {
          xslice_epilogue(s);
        }
        emit(s);
      }
      // weight gradients of the five convs, re-associated by input slice.
      // ONE launch per dense block, five problems, no idle accumulator rows: the 64-channel slices (x for conv1, o3|o4 for
      // conv4 / conv5) put two horizontal taps into one CTA's M = 128, and the third tap shares its CTA with an all-ones block
      // whose column sums are the bias gradients of all five convs.  Per 128-pixel tile: 7 CTA-units of (M = 128) x N x 24
      // MMAs (3 x 160 + 160 + 96 + 32 + 32 = 800 columns); three channel-block problems with idle M rows and a separate bias
      // problem would take 9 + 1/3 (928 columns).
      const int c5 = conv_index_rdb(P, r, 5), c4 = conv_index_rdb(P, r, 4), c3 = conv_index_rdb(P, r, 3), c2 = conv_index_rdb(P, r, 2),
                c1 = conv_index_rdb(P, r, 1);
      Step wg = wgrad_batch(D, 192, 192, DYc, 192, 192, N, H, W);
      add_problem(wg, 0, 0, 160);             // x, o1, o2 rows at the CTA's tap x [dY5|dY4|dY3|dY2]
      add_seg(wg, 0, 64, wref(c5), 192, 0, 64);
      add_seg(wg, 64, 96, wref(c4), 160, 0, 32);
      add_seg(wg, 96, 128, wref(c3), 128, 0, 32);
      add_seg(wg, 128, 160, wref(c2), 96, 0, 32);
      add_packed(wg, 128, 2, -1, 0, 160);     // (o3|o4 at dx 2 | ones) x [dY5|dY4|dY3|dY2]
      add_seg(wg, 0, 64, wref(c5), 192, 128, 64, 1);
      add_seg(wg, 64, 96, wref(c4), 160, 128, 32, 1);
      add_seg(wg, 0, 64, bref(c5), 1, 0, 64, 2);
      add_seg(wg, 64, 96, bref(c4), 1, 0, 32, 2);
      add_seg(wg, 96, 128, bref(c3), 1, 0, 32, 2);
      add_seg(wg, 128, 160, bref(c2), 1, 0, 32, 2);
      add_packed(wg, 128, 0, 1, 0, 96);       // (o3|o4 at dx 0 | o3|o4 at dx 1) x [dY5|dY4]
      add_seg(wg, 0, 64, wref(c5), 192, 128, 64);
      add_seg(wg, 64, 96, wref(c4), 160, 128, 32);
      add_packed(wg, 0, 0, 1, 160, 32);       // (x at dx 0 | x at dx 1) x dY1
      add_seg(wg, 0, 32, wref(c1), 64, 0, 32);
      add_packed(wg, 0, 2, -1, 160, 32);      // (x at dx 2 | ones) x dY1
      add_seg(wg, 0, 32, wref(c1), 64, 0, 32, 1);
      add_seg(wg, 0, 32, bref(c1), 1, 0, 32, 2);
      emit(wg);
      if (j == 0) {
        // gradient buckets: G RRDBs each (their convs are contiguous in the flat buffer); the LAST trunk bucket is at most two
        // RRDBs so that little communication is left after the final kernels
        const int blk = r / 3;
        const int G = d.grad_bucket_rrdbs > 0 ? d.grad_bucket_rrdbs : 1;
        if (blk % G == 0 || (G > 2 && blk == 2)) {
          emit(unpack_step(conv_index_rdb(P, r, 1), bucket_hi));
          bucket_hi = conv_index_rdb(P, r, 1);
        }
      }
    }
    // conv1: gradient of its output = trunk path (GR) + long skip (GT)
    if (!trunk) {
      serves(-1, 0, 1);
      Step ad; ad.type = ST_ADD; ad.a = ws(P.o_gr); ad.b = ws(P.o_gt); ad.c = ws(P.o_go1); ad.count = Ppix * 64;
      emit(ad);
      Step w1 = wgrad_step(P.o_xin, P.xin_stride, P.xin_stride, P.o_go1, 64, 64, N, H, W, 0, 0, 64);
      add_seg(w1, 0, 64, wref(0), d.in_channels, 0, 64);
      emit(w1);
      Step b1 = biasgrad_step(P.o_go1, Ppix, 64, 0, 64);
      add_bseg(b1, 0, 64, bref(0), 64);
      emit(b1);
      emit(unpack_step(0, 1));
    }
    // ONE data-gradient chain for the whole backward pass (no pipeline drain / refill at every gradient bucket), then
    // the weight- and bias-gradient kernels bucket by bucket: every dense block has its own dY buffer for that.
    for (const Step& c : seg_convs) P.bwd.push_back(c);
    for (const Step& o : seg_others) P.bwd.push_back(o);
    seg_convs.clear(); seg_others.clear();
    // Gradient w.r.t. the LR input = conv1's data gradient of GO1 (64 -> in_channels), stored fp32 NCHW to the caller's dx.
    // The reference produces it whenever x.requires_grad (input-gradient probes); it is launched only when dx != NULL.
    if (!trunk) {
      const int C = d.in_channels;
      const int npad = (int)align_up(C, 16);
      PackOp op; memset(&op, 0, sizeof(op));
      op.n_total = npad; op.n_cols = 16; op.n_valid = C; op.num_chunks = 1; op.mode = kPackDgrad; op.nseg = 1;
      op.seg[0] = seg(0, 64, 0, 64, C, 0, 0, 0);
      const int row0 = B.add_pack(op);
      ConvParams cp = base_conv_params(N, H, W, 1, 4, 0, 1 << 20, row0, 16, npad);
      Step s = conv_step(B.add_map(P.o_go1, 64, 64, N, H, W, kABoxRows), cp, 1);
      s.cp.epi.store_mode = kStoreNCHW;
      s.cp.epi.n_valid = C;
      s.of.kind = RK_Y;
      s.needs_dx = true;
      P.bwd.push_back(s);
    } else {  // the trunk-input gradient is GR after the first dense block's epilogue
      Step s; s.type = ST_TRUNK_EXPORT; s.a = ws(P.o_gr); s.needs_dx = true;
      P.bwd.push_back(s);
    }
  }

  // packed buffer = bf16 tile rows followed by the fp32 biases
  const long long bias_base = align_up(P.total_rows * 128, 1024);
  P.packed_bytes = bias_base + P.bias_floats * 4;
  auto fix = [&](std::vector<Step>& v) {
    for (Step& s : v)
      if (s.bias.kind == RK_PACKED) s.bias.off = bias_base + (-1 - s.bias.off) * 4;
  };
  fix(P.fwd);
  fix(P.bwd);
  // merge consecutive conv launches into chains over one global layer list
  auto chainify = [&](std::vector<Step>& v) {
    std::vector<Step> out;
    for (Step& s : v) {
      if (s.type != ST_CONV) { out.push_back(s); continue; }
      const int work = s.cp.num_tiles * s.cp.col_groups;
      // A chain is limited by the constant-memory tables (layers, entries = layers x image groups).  Long chains are cut
      // where a layer starts fresh accumulators (never inside a dense block whose partial sums live in TMEM).
      const int max_layers = std::min(kMaxChainLayers, kMaxChainEntries / (P.groups > 0 ? P.groups : 1)) - 8;
      const bool cut = !out.empty() && out.back().type == ST_CHAIN &&
                       ((out.back().nlayers >= max_layers && s.cp.acc_first && !(s.cp.acc_hold && s.cp.epi_cols == 0)) ||
                        out.back().needs_dx != s.needs_dx);
      if (out.empty() || out.back().type != ST_CHAIN || cut) {
        Step c; c.type = ST_CHAIN; c.layer0 = (int)P.layer_steps.size(); c.nlayers = 0; c.chain_grid = 0;
        c.needs_dx = s.needs_dx;
        out.push_back(c);
      }
      out.back().nlayers++;
      if (work > out.back().chain_grid) out.back().chain_grid = work;
      P.layer_steps.push_back(s);
    }
    v.swap(out);
  };
  chainify(P.fwd);
  chainify(P.bwd);
  {  // a trunk-only data-gradient chain behind a cut (see above) runs on one CTA per work item of an image group
    int nchains = 0, last = -1;
    for (size_t i = 0; i < P.bwd.size(); ++i)
      if (P.bwd[i].type == ST_CHAIN && !P.bwd[i].needs_dx) { ++nchains; last = (int)i; }
    if (nchains >= 2 && P.groups >= 2 && !P.trunk) {  // (trunk plans: no tail gradients to run beside it)
      Step& c = P.bwd[last];
      int per_group = 0;
      for (int l = 0; l < c.nlayers; ++l) {
        const ConvParams& cp = P.layer_steps[c.layer0 + l].cp;
        const int w = ((cp.N + P.groups - 1) / P.groups) * cp.tiles_x * cp.tiles_y * cp.col_groups;
        if (w > per_group) per_group = w;
      }
      if (per_group > 0 && per_group < c.chain_grid) c.chain_grid = per_group;
      P.bwd_overlap_chain = last;
    }
  }
  if (P.det && train) plan_deterministic(P, 4, P.plan_sms / 2);  // run_steps: four weight-gradient streams on half the SMs each
  return 0;
}

// ------------------------------------------------------------------------------------------------------ execution
static void* resolve(const Ref& r, const Bases& b) {
  switch (r.kind) {
    case RK_WS: return (char*)b.ws + r.off;
    case RK_PACKED: return (char*)b.packed + r.off;
    case RK_Y: return (char*)b.y + r.off;
    case RK_DY: return (char*)b.dy + r.off;
    case RK_GRADS: return (char*)b.grads + r.off;
    default: return nullptr;
  }
}

static void* resolve(const Ref& r, const Bases& b);
static int ensure_maps(b200sr_plan& P, void* wsp, void* packed, cudaStream_t st) {
  ++P.slot_clock;
  int victim = 0;
  for (int i = 0; i < b200sr_plan::kMapSlots; ++i) {
    b200sr_plan::MapSlot& sl = P.slots[i];
    if (sl.ws == wsp && sl.packed == packed && sl.maps.size() == P.map_specs.size() && sl.d_layers) {
      sl.stamp = P.slot_clock;
      P.cur_slot = i;
      return 0;
    }
    if (sl.stamp < P.slots[victim].stamp) victim = i;
  }
  static const bool trace = [] { const char* e = getenv("B200SR_TRACE"); return e && atoi(e) != 0; }();
  ++P.map_encodes;
  if (trace) fprintf(stderr, "b200sr: plan %p encodes descriptors for workspace %p / packed %p (miss %lld, slot %d)\n", (void*)&P, wsp, packed, P.map_encodes, victim);
  b200sr_plan::MapSlot& slot = P.slots[victim];
  slot.ws = nullptr;  // invalid until fully rebuilt
  P.cur_slot = victim;
  slot.maps.resize(P.map_specs.size());
  for (size_t i = 0; i < P.map_specs.size(); ++i) {
    const ActMapSpec& s = P.map_specs[i];
    int rc = encode_act_map(&slot.maps[i], (char*)wsp + s.off, s.c_valid, s.c_pix, s.n, s.h, s.w, s.box_rows, s.box_w);
    if (rc) return rc;
  }
  // device-resident layer list (pointers resolved against this workspace / packed buffer)
  Bases b{wsp, packed, nullptr, nullptr, nullptr};
  P.h_layers.resize(P.layer_steps.size());
  for (size_t i = 0; i < P.layer_steps.size(); ++i) {
    const Step& s = P.layer_steps[i];
    LayerDesc& L = P.h_layers[i];
    L.tmA = slot.maps[s.amap];
    L.p = s.cp;
    L.p.epi.bias = (const float*)resolve(s.bias, b);
    L.p.epi.mask = (const __nv_bfloat16*)resolve(s.mask, b);
    L.p.epi.r1 = (const float*)resolve(s.r1, b);
    L.p.epi.r2 = (const float*)resolve(s.r2, b);
    L.p.epi.out_f32 = (float*)resolve(s.of, b);   // RK_Y resolves to nullptr here: the final layer uses the y_dyn kernel argument
    L.p.epi.out_f32_b = (float*)resolve(s.ofb, b);
    L.p.epi.out_bf16 = (__nv_bfloat16*)resolve(s.ob, b);
    L.p.epi.clamp_mask = (unsigned char*)resolve(s.cm, b);
    L.p.epi.feat_out = (float*)resolve(s.feat, b);
    L.p.epi.res_bf16 = (const __nv_bfloat16*)resolve(s.resb, b);
  }
  // entry lists: every layer of a chain is split into (up to) two image groups that flow through the chain independently
  if (P.h_entries.empty()) {
    auto build_entries = [&](std::vector<Step>& steps) {
      for (Step& s : steps) {
        if (s.type != ST_CHAIN) continue;
        const int grid = s.chain_grid < g_num_sms ? s.chain_grid : g_num_sms;
        const int groups = P.groups;
        s.entry0 = (int)P.h_entries.size();
        // emission order: ordinary layers go (layer, group A), (layer, group B), ...  The layers of a dense block (passes +
        // fillers, whose accumulators occupy the CTA's TMEM throughout) go pair of groups by pair of groups -- two groups are
        // resident at a time -- interleaved layer by layer; a FILLER (partial sums, no epilogue) directly follows the producing
        // layer of ITS OWN GROUP it was emitted after: the producer warp first resolves that layer's dependency and then streams
        // the filler's operands, and the MMA warp works the filler off while the OTHER group's dependency is in flight:
        //   p0A p0B p1A p1B | p2A F1A p2B F1B | p3A F2A p3B F2B | c5A c5B
        std::vector<std::pair<int, int>> order;  // (layer, group)
        auto is_filler = [&](int l) { return P.layer_steps[s.layer0 + l].cp.epi_cols == 0; };
        for (int l = 0; l < s.nlayers;) {
          const ConvParams& cp = P.layer_steps[s.layer0 + l].cp;
          if (cp.acc_hold && cp.acc_first && !is_filler(l)) {
            int l1 = l + 1;
            // a dense block = the run of resident layers up to (not including) the next block's first pass
            while (l1 < s.nlayers && P.layer_steps[s.layer0 + l1].cp.acc_hold &&
                   !(P.layer_steps[s.layer0 + l1].cp.acc_first && !is_filler(l1))) ++l1;
            for (int g0 = 0; g0 < groups; g0 += 2) {
              for (int ll = l; ll < l1; ++ll) {
                if (!is_filler(ll) && ll + 1 < l1 && is_filler(ll + 1)) {
                  for (int g = g0; g < g0 + 2 && g < groups; ++g) { order.push_back({ll, g}); order.push_back({ll + 1, g}); }
                  ++ll;
                } else {
                  for (int g = g0; g < g0 + 2 && g < groups; ++g) order.push_back({ll, g});
                }
              }
            }
            l = l1;
          } else {
            for (int g = 0; g < groups; ++g) order.push_back({l, g});
            ++l;
          }
        }
        std::vector<int> index_of((size_t)s.nlayers * groups, -1);
        for (size_t i = 0; i < order.size(); ++i) index_of[(size_t)order[i].first * groups + order[i].second] = (int)i;
        for (size_t i = 0; i < order.size(); ++i) {
          const int l = order[i].first, g = order[i].second;
          const ConvParams& cp = P.layer_steps[s.layer0 + l].cp;
          const int tpi = cp.tiles_x * cp.tiles_y;
          const int img_lo = (int)((long long)cp.N * g / groups), img_hi = (int)((long long)cp.N * (g + 1) / groups);
          EntryDesc e; memset(&e, 0, sizeof(e));
          e.layer = s.layer0 + l;
          e.tile_lo = img_lo * tpi; e.tile_hi = img_hi * tpi;
          // dependency = the nearest earlier layer that PRODUCES data (has an epilogue).  A filler only reads slices whose
          // producing layers an EARLIER entry of the same group already waited for (it is emitted after the pass that follows
          // them), so it carries no dependency of its own.
          int lp = l - 1;
          while (lp >= 0 && P.layer_steps[s.layer0 + lp].cp.epi_cols == 0) --lp;
          e.dep = (lp >= 0 && cp.epi_cols > 0) ? index_of[(size_t)lp * groups + g] : -1;
          e.rot = (int)(((long long)img_lo * tpi * cp.col_groups) % grid);
          e.slot = g & 1;  // each group starts where the previous one's last round ended
          e.pad[0] = 0;
          P.h_entries.push_back(e);
        }
        s.nentries = (int)P.h_entries.size() - s.entry0;
        // Per-image announcements: an entry whose consumers all run the SAME tiles on the SAME CTAs (one tile per CTA) is announced
        // image by image, and each consumer CTA waits only for the tiles of its own image -- a conv reads nothing of another image,
        // and everything older is covered transitively (release / acquire chains stay inside the image's CTAs, which have
        // themselves seen every earlier whole-entry announcement).  Images then drift apart instead of meeting at a 128-CTA
        // rendezvous after every layer.
        std::vector<int> ok((size_t)s.nentries, -1);  // -1: no consumer yet, 1: all consumers eligible so far, 0: not eligible
        for (int i = 0; i < s.nentries; ++i) {
          const EntryDesc& e = P.h_entries[s.entry0 + i];
          if (e.dep < 0) continue;
          const EntryDesc& dpe = P.h_entries[s.entry0 + e.dep];
          const ConvParams& ce = P.layer_steps[e.layer].cp;
          const ConvParams& cd = P.layer_steps[dpe.layer].cp;
          const int tpi = ce.tiles_x * ce.tiles_y, ntiles = e.tile_hi - e.tile_lo;
          const bool same = ce.col_groups == 1 && cd.col_groups == 1 && e.tile_lo == dpe.tile_lo && e.tile_hi == dpe.tile_hi && e.rot == dpe.rot &&
                            ce.tiles_x == cd.tiles_x && ce.tiles_y == cd.tiles_y && ntiles <= grid && tpi >= 2 && ntiles / tpi <= kCtrStride - 1;
          if (!same) ok[e.dep] = 0;
          else if (ok[e.dep] < 0) ok[e.dep] = 1;
        }
        for (int i = 0; i < s.nentries; ++i)
          if (ok[i] == 1) P.h_entries[s.entry0 + i].pad[0] = 1;
      }
    };
    build_entries(P.fwd);
    build_entries(P.bwd);
  }
  if (!slot.d_layers) CUDA_TRY(cudaMalloc(&slot.d_layers, P.h_layers.size() * sizeof(LayerDesc)));
  if (!P.tables_ready) {
    P.tables_ready = true;
    CUDA_TRY(cudaMalloc(&P.d_entries, P.h_entries.size() * sizeof(EntryDesc)));
    P.counters_bytes = (size_t)kMaxChainEntries * kCtrStride * sizeof(unsigned int);  // completion counters of the chain being launched
    CUDA_TRY(cudaMalloc(&P.d_counters, P.counters_bytes));
    CUDA_TRY(cudaMemcpyAsync(P.d_entries, P.h_entries.data(), P.h_entries.size() * sizeof(EntryDesc), cudaMemcpyHostToDevice, st));
    std::vector<uint4> lrec(P.h_layers.size() * 2), erec(P.h_entries.size());
    for (size_t i = 0; i < P.h_layers.size(); ++i) make_layer_rec(P.h_layers[i].p, &lrec[2 * i], packed);
    for (size_t i = 0; i < P.h_entries.size(); ++i) erec[i] = make_entry_rec(P.h_entries[i]);
    CUDA_TRY(cudaMalloc(&P.d_layer_rec, lrec.size() * sizeof(uint4)));
    CUDA_TRY(cudaMalloc(&P.d_entry_rec, erec.size() * sizeof(uint4)));
    CUDA_TRY(cudaMemcpyAsync(P.d_layer_rec, lrec.data(), lrec.size() * sizeof(uint4), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(P.d_entry_rec, erec.data(), erec.size() * sizeof(uint4), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));  // lrec / erec are pageable host vectors that die at scope exit
  }
  CUDA_TRY(cudaMemcpyAsync(slot.d_layers, P.h_layers.data(), P.h_layers.size() * sizeof(LayerDesc), cudaMemcpyHostToDevice, st));
  slot.ws = wsp;
  slot.packed = packed;
  slot.stamp = P.slot_clock;
  return 0;
}

// The constant-memory tables are one per device: chain launches issued to DIFFERENT streams of a device are ordered
// after one another with an event (they fill the whole GPU anyway), so a later upload can never overtake an earlier
// launch that still reads its own tables.
struct ChainOrder { cudaEvent_t ev = nullptr; cudaStream_t last = nullptr; bool any = false; };
static ChainOrder g_chain_order[64];
static std::mutex g_chain_mutex;

static int launch_chain(b200sr_plan& P, const Step& s, const Bases& b, cudaStream_t st) {
  std::lock_guard<std::mutex> lock(g_chain_mutex);
  int grid = s.chain_grid < g_num_sms ? s.chain_grid : g_num_sms;
  if (grid < 1) grid = 1;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  ChainOrder& co = g_chain_order[dev & 63];
  if (!co.ev) CUDA_TRY(cudaEventCreateWithFlags(&co.ev, cudaEventDisableTiming));
  if (co.any && co.last != st) CUDA_TRY(cudaStreamWaitEvent(st, co.ev, 0));
  if (s.nentries > kMaxChainEntries || s.nlayers > kMaxChainLayers)
    return fail(B200SR_ERR_INVALID, "chain too long (%d entries, %d layers)", s.nentries, s.nlayers);
  // the producer / MMA warps read their parameters from constant memory: load this chain's slice (stream ordered)
  CUDA_TRY(cudaMemcpyToSymbolAsync(c_layer_rec, P.d_layer_rec + 2 * (size_t)s.layer0, (size_t)s.nlayers * 2 * sizeof(uint4), 0, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(cudaMemcpyToSymbolAsync(c_entry_rec, P.d_entry_rec + s.entry0, (size_t)s.nentries * sizeof(uint4), 0, cudaMemcpyDeviceToDevice, st));
  int layer0 = s.layer0;
  const LayerDesc* layers = P.d_layers();
  const EntryDesc* entries = P.d_entries + s.entry0;
  int ne = s.nentries;
  float* y = (float*)b.y;
  int dbg = g_debug;
  unsigned int* ctr = P.d_counters;
  CUDA_TRY(cudaMemsetAsync(ctr, 0, (size_t)s.nentries * kCtrStride * sizeof(unsigned int), st));
  const uint8_t* pw = (const uint8_t*)b.packed;
  void* args[] = {(void*)&layers, (void*)&entries, (void*)&ne, (void*)&pw, (void*)&ctr, (void*)&y, (void*)&dbg, (void*)&layer0};
  // <1, 0>: probes compiled in; <0, 1>: the VGG feature build (ReLU, feature store, 512-column bias vectors)
  const void* fn = (P.is_vgg || P.is_disc) ? (const void*)conv3x3_chain_kernel<0, 1>
                            : (dbg ? (const void*)conv3x3_chain_kernel<1, 0> : (const void*)conv3x3_chain_kernel<0, 0>);
  if (P.is_vgg || P.is_disc) dbg = 0;
  if (ne > 1) {
    CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kConvThreads), args, (size_t)conv_smem_bytes(1), st));
  } else {
    CUDA_TRY(cudaLaunchKernel(fn, dim3(grid), dim3(kConvThreads), args, (size_t)conv_smem_bytes(1), st));
  }
  if (co.last != st || !co.any) {  // (same stream again: stream order already protects the tables)
    co.last = st;
    co.any = true;
  }
  CUDA_TRY(cudaEventRecord(co.ev, st));
  return 0;
}

// deal the CTAs of one wave of `sms` SMs out in proportion to each problem's cost (max of tensor cycles and L2->SM bytes / 42 B
// per clock): sets the problems' split counts and CTA ranges
static void wgrad_deal(WgradBatch& wb, int sms) {
  double work[kWgMaxProblems], total = 0;
  for (int j = 0; j < wb.num_problems; ++j) {
    WgradParams& wp = wb.prob[j];
    const int nacc = wp.dy_mask ? __builtin_popcount(wp.dy_mask) : 3;
    const double mma = nacc * 8.0 * (wp.n_cols / 2.0);
    const double ld = wgrad_load_bytes(wp) / 42.0;
    work[j] = (mma > ld ? mma : ld) * wgrad_ntap(wp);
    total += work[j];
  }
  int ctas = 0;
  for (int j = 0; j < wb.num_problems; ++j) {
    WgradParams& wp = wb.prob[j];
    const int ntap = wgrad_ntap(wp);
    int splits = (int)(sms * work[j] / total / ntap + 0.5);
    if (splits < 1) splits = 1;
    if (splits > wb.num_tiles) splits = wb.num_tiles;
    wp.splits = splits;
    wb.cta_begin[j] = ctas;
    ctas += splits * ntap;
  }
  wb.cta_begin[wb.num_problems] = ctas;
}

// ordered_sum_kernel over a list of jobs (at most kMaxSumJobs), about 1024 elements per block
template <typename T>
static int launch_ordered_sum(const SumJob<T>* jobs, int n, cudaStream_t st) {
  if (n < 1 || n > kMaxSumJobs) return fail(B200SR_ERR_INVALID, "internal: %d ordered-sum jobs", n);
  SumJobs<T> J;
  memset(&J, 0, sizeof(J));
  J.n = n;
  int blocks = 0;
  for (int j = 0; j < n; ++j) {
    J.job[j] = jobs[j];
    J.block0[j] = blocks;
    const long long total = (long long)jobs[j].n0 * jobs[j].n1 * jobs[j].n2 * jobs[j].n3;
    if (total < 1 || total >= (1LL << 31)) return fail(B200SR_ERR_INVALID, "internal: ordered-sum job of %lld elements", total);
    blocks += (int)std::min<long long>((total + 1023) / 1024, 1024);
  }
  J.block0[n] = blocks;
  ordered_sum_kernel<T><<<blocks, 256, 0, st>>>(J);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
// a row job: dst[i] = sum over r < rows of src[r * stride + i], i < n
template <typename T>
static SumJob<T> sum_rows_t(T* dst, const T* src, int rows, long long stride, int n) {
  SumJob<T> j;
  memset(&j, 0, sizeof(j));
  j.dst = dst; j.src = src; j.stride = stride; j.S = rows; j.n0 = n; j.n1 = j.n2 = j.n3 = 1;
  return j;
}
static SumJob<double> sum_rows(double* dst, const double* src, int rows, long long stride, int n) { return sum_rows_t(dst, src, rows, stride, n); }

// Deterministic launches: the segment a split flushes into -- the part of the staging tensor that `g` of problem `wp` writes
// (input channels [ci0, ci_total) up to two 64-row M blocks, the output channels of its columns), as a compact tensor of its own
static WgradSegment wgrad_det_segment(const WgradParams& wp, const WgradSegment& g) {
  WgradSegment c = g;
  c.ci0 = 0;
  c.ci_total = std::max(1, std::min(g.ci0 + (wp.blk[1].kind == kWgBlkIdle ? 64 : 128), g.ci_total) - g.ci0);
  c.co_pad = std::min(g.co_pad, std::min(g.col_end, wp.n_cols) - g.col_begin);
  return c;
}
// floats of one split's copy of that segment
static long long wgrad_det_region(const WgradParams& wp, const WgradSegment& g) {
  const WgradSegment c = wgrad_det_segment(wp, g);
  return 9LL * c.co_pad * c.ci_total;
}
// first bit and length of a contiguous tap mask (0 = all three); length 0 when the bits are not contiguous
static int tap_range(int mask, int* lo) {
  const int m = mask ? mask : 7;
  *lo = __builtin_ctz(m);
  const int n = __builtin_popcount(m);
  return (m >> *lo) == (1 << n) - 1 ? n : 0;
}
// bias-gradient blocks of a launch (at most two per SM: see bias_grad_vec_kernel)
static int bias_grad_blocks(const BiasGradParams& bp, int sms) {
  const int plv = kBiasGradThreads / (bp.ncols / 8);
  long long blocks = (bp.P + plv * 8 - 1) / (plv * 8);
  if (blocks > 2 * sms) blocks = 2 * sms;
  return (int)blocks;
}

// Deterministic plans: the split counts of every weight-gradient launch are dealt once, here, for `wgrad_sms` SMs (what
// run_steps gives one launch), and the workspace gains one partial-sum lane per weight-gradient stream, sized for the largest
// launch.  A launch and its ordered sum run on one stream, so the lane is reused in stream order.
static void plan_deterministic(b200sr_plan& P, int lanes, int wgrad_sms) {
  long long lane = 0;
  for (Step& s : P.bwd) {
    long long bytes = 0;
    if (s.type == ST_WGRAD) {
      wgrad_deal(s.wb, wgrad_sms);
      for (int j = 0; j < s.wb.num_problems; ++j)
        for (int i = 0; i < s.wb.prob[j].num_seg; ++i) bytes += 4LL * s.wb.prob[j].splits * wgrad_det_region(s.wb.prob[j], s.wb.prob[j].seg[i]);
    } else if (s.type == ST_BIASGRAD) {
      s.det_blocks = bias_grad_blocks(s.bp, P.plan_sms);
      bytes = 4LL * s.det_blocks * s.bp.ncols;
    }
    lane = std::max(lane, bytes);
  }
  P.det_lane_bytes = align_up(lane, 1024);
  P.o_det = align_up(P.ws_bytes, 1024);
  P.ws_bytes = P.o_det + lanes * P.det_lane_bytes;
}

// sms_cap: SMs one wgrad wave may use (0: all).  slab: the partial-sum lane of the stream (deterministic plans), else nullptr
static int launch_wgrad(const Step& s, const CUtensorMap& tmX, const CUtensorMap& tmDY, const Bases& b, cudaStream_t st, int sms_cap,
                        char* slab = nullptr) {
  WgradBatch wb = s.wb;
  for (int j = 0; j < wb.num_problems; ++j)
    for (int i = 0; i < wb.prob[j].num_seg; ++i) wb.prob[j].seg[i].out = (float*)resolve(s.wseg_out[j][i], b);
  if (!slab) {
    wgrad_deal(wb, (sms_cap > 0 && sms_cap < g_num_sms) ? sms_cap : g_num_sms);
    wgrad3x3_kernel<false><<<dim3(wb.cta_begin[wb.num_problems]), kWgThreads, kWgSmemBytes, st>>>(tmX, tmDY, wb);
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
  // deterministic: the splits dealt at plan build; every segment flushes into its own slab (one compact copy per split), and one job
  // per M block adds the split copies over exactly the box of the staging tensor that block writes (taps x channel quads x channels)
  SumJob<float> jobs[kMaxSumJobs];
  int nj = 0;
  long long off = 0;
  for (int j = 0; j < wb.num_problems; ++j) {
    WgradParams& wp = wb.prob[j];
    for (int i = 0; i < wp.num_seg; ++i) {
      const WgradSegment g = wp.seg[i];  // the staging tensor's view
      WgradSegment& c = wp.seg[i];       // the slab's
      c = wgrad_det_segment(wp, g);
      c.out = (float*)slab + off;
      off += wp.splits * wgrad_det_region(wp, g);
      for (int bk = 0; bk < 2; ++bk) {
        const int kind = wp.blk[bk].kind;
        if (kind == kWgBlkIdle || (g.blk_mask && !((g.blk_mask >> bk) & 1))) continue;
        const bool ones = kind == kWgBlkOnes;
        const int ci_lo = g.ci0 + (ones ? 0 : wp.blk[bk].c0 - wp.blk[0].c0);
        const int ci_hi = std::min(ci_lo + 64, g.ci_total);
        const int ncq = std::min(std::min(g.col_end, wp.n_cols) - g.col_begin, g.co_pad) / 4;
        if (ci_lo >= ci_hi || ncq < 1) continue;
        int dy_lo = 0, dx_lo = 0, ndy = 1, ndx = 1;
        if (!ones) {
          ndy = tap_range(wp.dy_mask, &dy_lo);
          if (wp.blk[bk].dx >= 0) dx_lo = wp.blk[bk].dx;
          else ndx = tap_range(wp.dx_mask, &dx_lo);
        }
        if (!ndy || !ndx || nj == kMaxSumJobs) return fail(B200SR_ERR_INVALID, "internal: deterministic wgrad launch not expressible as boxes");
        const long long tap_d = (long long)(g.co_pad / 4) * g.ci_total * 4, tap_s = (long long)(c.co_pad / 4) * c.ci_total * 4;
        const int tap0 = dy_lo * 3 + dx_lo;
        SumJob<float>& jb = jobs[nj++];
        jb.dst = g.out + tap0 * tap_d + ci_lo * 4LL;
        jb.src = c.out + tap0 * tap_s + (ci_lo - g.ci0) * 4LL;
        jb.stride = 9LL * c.co_pad * c.ci_total; jb.S = wp.splits;
        jb.n0 = (ci_hi - ci_lo) * 4; jb.n1 = ncq; jb.n2 = ndx; jb.n3 = ndy;
        jb.d1 = g.ci_total * 4LL; jb.d2 = tap_d; jb.d3 = 3 * tap_d;
        jb.s1 = c.ci_total * 4LL; jb.s2 = tap_s; jb.s3 = 3 * tap_s;
      }
    }
  }
  wgrad3x3_kernel<true><<<dim3(wb.cta_begin[wb.num_problems]), kWgThreads, kWgSmemBytes, st>>>(tmX, tmDY, wb);
  CUDA_TRY(cudaGetLastError());
  return launch_ordered_sum(jobs, nj, st);
}

// What a selective generator backward (b200sr_backward_select) computes.  Chosen per call: the plan and its step list serve
// every freeze pattern, and run_steps skips what nobody asked for.
struct GradSelect {
  std::vector<uint8_t> want;  // per conv: its weight and/or bias gradient is wanted
  int stop_blk = -1;          // data-gradient layers of dense blocks below this one are not launched (R: tail only, R + 1: none)
  int R = 0;
  int t0 = 1;                 // conv index of the first dense-block conv
  bool any(int c0, int c1) const {
    for (int c = c0; c < c1; ++c)
      if (want[c]) return true;
    return false;
  }
  // the convs a launch wrote: a dense block's one weight-gradient launch writes all five of its convs if any is wanted
  bool written(int c) const {
    if (c < t0 || c >= t0 + 5 * R) return want[c] != 0;
    const int c0 = t0 + (c - t0) / 5 * 5;
    return any(c0, c0 + 5);
  }
};

// mask: per conv (NULL: all); grads: a flat gradient buffer is written; dx: the input gradient is wanted
static GradSelect make_select(const b200sr_plan& P, const uint8_t* mask, bool grads, bool dx) {
  const int nconv = ((int)P.param_off.size() - 1) / 2;
  GradSelect g;
  g.R = P.R;
  g.t0 = P.t0;
  g.want.assign(nconv, 0);
  if (grads)
    for (int c = 0; c < nconv; ++c) g.want[c] = mask ? (mask[c] != 0) : 1;
  // conv1's output gradient GO1 = GR + GT needs the whole trunk (as does a trunk plan's dx); otherwise the walk ends after the lowest
  // wanted dense block
  if (dx || (!P.trunk && g.want[0])) {
    g.stop_blk = -1;
  } else {
    g.stop_blk = P.R + 1;
    for (int r = 0; r < P.R; ++r)
      if (g.any(conv_index_rdb(P, r, 1), conv_index_rdb(P, r, 5) + 1)) { g.stop_blk = r; break; }
    if (g.stop_blk > P.R && g.any(P.t0 + 5 * P.R, nconv)) g.stop_blk = P.R;
  }
  return g;
}

// layers of data-gradient chain s that a selection launches: a prefix, the chain walks from the tail down to block 0
static int chain_layers(const b200sr_plan& P, const Step& s, const GradSelect* g) {
  if (!g || s.needs_dx) return s.nlayers;
  int n = 0;
  while (n < s.nlayers && P.layer_steps[s.layer0 + n].blk >= g->stop_blk) ++n;
  return n;
}

// whether a non-chain step of the generator backward runs under a selection (grads / dx: the caller passed those buffers; cb: a
// bucket callback is installed, otherwise one merged unpack covers every conv)
static bool step_selected(const Step& s, const GradSelect* g, bool grads, bool dx, bool cb) {
  if (!g) return true;
  switch (s.type) {
    case ST_MEMSET: return grads || s.a.kind != RK_GRADS;
    case ST_WGRAD: case ST_BIASGRAD: return g->any(s.wc0, s.wc1);
    case ST_ADD: return dx || g->want[0];  // GO1 feeds conv1's weight / bias gradients and the input gradient
    case ST_UNPACK: return cb ? g->any(s.i0, s.i1) : g->any(0, (int)g->want.size());
    default: return true;
  }
}

static int launch_chain(b200sr_plan& P, const Step& s, const Bases& b, cudaStream_t st);

// launches the first `nlayers` layers of chain s (all of them: the chain itself)
static int launch_chain_prefix(b200sr_plan& P, const Step& s, int nlayers, const Bases& b, cudaStream_t st) {
  if (nlayers == s.nlayers) return launch_chain(P, s, b, st);
  // entries go layer block by layer block, so those of a layer prefix are a prefix of the entry list (their dependencies
  // point backwards only)
  Step c = s;
  c.nlayers = nlayers;
  c.nentries = 0;
  for (int i = 0; i < s.nentries; ++i) {
    if (P.h_entries[s.entry0 + i].layer >= s.layer0 + nlayers) continue;
    if (i != c.nentries) return fail(B200SR_ERR_INVALID, "internal: the entries of a chain's layer prefix are not a prefix");
    ++c.nentries;
  }
  return launch_chain(P, c, b, st);
}

static int run_steps(b200sr_plan& P, std::vector<Step>& steps, const Bases& b, const void* x, int x_dtype, const int64_t* xs,
                     b200sr_bucket_cb cb, void* user, cudaStream_t st, const GradSelect* sel = nullptr) {
  const b200sr_net_desc& d = P.d;
  // Weight-gradient launches of different dense blocks are independent of one another: once the data-gradient chain is
  // done they alternate between the caller's stream and a side stream, so the flush tail of one launch overlaps the ramp-up
  // of the next (each launch fills the GPU with one CTA per SM).  Everything that consumes their results joins first.
  // Generator plans (round 2, same-box scans over streams x CTAs per launch): FOUR streams with HALF of the SMs per launch
  // -- fewer pixel splits per dense block = fewer partial sums flushed with red.global.add into the same addresses, and the launches
  // of neighbouring blocks run side by side -- 11.93 -> 11.73 ms/step (2 streams x all SMs: the round-1 setting, kept for the
  // discriminator / VGG plans).
  const bool gen_plan = !P.is_disc && !P.is_vgg;
  const int nstreams = gen_plan ? 4 : 2;
  const int wgrad_cap = gen_plan ? g_num_sms / 2 : 0;  // two launches exactly side by side (74 + 74 on 148 SMs)
  const bool alternate = &steps == &P.bwd;
  bool forked = false, side_dirty = false;
  int wcount = 0;
  auto join = [&]() -> int {
    if (side_dirty) {
      for (int k = 0; k < nstreams - 1; ++k) {
        CUDA_TRY(cudaEventRecord(P.ev_join[k], P.side_stream[k]));
        CUDA_TRY(cudaStreamWaitEvent(st, P.ev_join[k], 0));
      }
      side_dirty = false;
    }
    return 0;
  };
  auto ensure_streams = [&]() -> int {
    if (!P.ev_fork) {
      for (int k = 0; k < 3; ++k) {
        CUDA_TRY(cudaStreamCreateWithFlags(&P.side_stream[k], cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&P.ev_join[k], cudaEventDisableTiming));
      }
      CUDA_TRY(cudaEventCreateWithFlags(&P.ev_fork, cudaEventDisableTiming));
    }
    return 0;
  };
  // deterministic plans: partial-sum lane k belongs to weight-gradient stream k (0: the caller's stream, k: side_stream[k - 1])
  auto lane_of = [&](int k) -> char* { return P.det ? (char*)b.ws + P.o_det + k * P.det_lane_bytes : nullptr; };
  auto do_biasgrad = [&](const Step& s, cudaStream_t bs, char* slab) -> int {
    BiasGradParams bp = s.bp;
    bp.g = (const __nv_bfloat16*)resolve(s.bg_g, b);
    for (int i = 0; i < bp.nseg; ++i) bp.seg[i].out = (float*)resolve(s.seg_out[i], b);
    // every plan's bias-gradient steps satisfy this (ncols 16 / 64 / 256, c0 = 0, stride 64 / 256, 1024-aligned buffers)
    if (bp.ncols % 8 != 0 || bp.ncols / 8 > kBiasGradThreads || bp.c0 % 8 != 0 || bp.stride % 8 != 0 ||
        (reinterpret_cast<uintptr_t>(bp.g) & 15) != 0)
      return fail(B200SR_ERR_INVALID, "internal: bias-gradient step with ncols %d, c0 %d, stride %d is not 16-byte vectorisable",
                  bp.ncols, bp.c0, bp.stride);
    if (!slab) {
      bias_grad_vec_kernel<false><<<bias_grad_blocks(bp, g_num_sms), kBiasGradThreads, 0, bs>>>(bp);
      CUDA_TRY(cudaGetLastError());
      return 0;
    }
    // deterministic: the block rows [block][ncols] are summed row by row; the segments must split the columns into equal parts
    // that all go to one output (the four phases of an upsample conv's bias), so the rows are [block][segment][width]
    const int wd = bp.seg[0].col_end - bp.seg[0].col_begin;
    for (int i = 0; i < bp.nseg; ++i)
      if (bp.seg[i].col_begin != i * wd || bp.seg[i].col_end != (i + 1) * wd || bp.seg[i].out != bp.seg[0].out ||
          bp.seg[i].n_valid != bp.seg[0].n_valid)
        return fail(B200SR_ERR_INVALID, "internal: bias-gradient segments are not equal column groups of one output");
    if (bp.nseg * wd != bp.ncols) return fail(B200SR_ERR_INVALID, "internal: bias-gradient segments do not cover the columns");
    float* out = bp.seg[0].out;
    bp.seg[0].out = (float*)slab;
    bias_grad_vec_kernel<true><<<s.det_blocks, kBiasGradThreads, 0, bs>>>(bp);
    CUDA_TRY(cudaGetLastError());
    const SumJob<float> j = sum_rows_t(out, (const float*)slab, s.det_blocks * bp.nseg, wd, bp.seg[0].n_valid);
    return launch_ordered_sum(&j, 1, bs);
  };
  // Weight / bias gradients that sit between two data-gradient chains (the HR tail's, see build_plan) are DEFERRED behind the launch of
  // the second chain and go to the side streams only: the trunk chain, enqueued first, takes its SMs, they fill the rest and run beside it.
  const int overlap_chain = (alternate && !cb && b.grads) ? P.bwd_overlap_chain : -1;
  std::vector<int> deferred;
  for (size_t si = 0; si < steps.size(); ++si) {
    Step& s = steps[si];
    if (s.needs_wgrad && !b.grads) continue;  // discriminator backward for the generator update: data gradients only
    if (s.needs_dx && !b.y) continue;         // nobody asked for the input gradient
    if (!step_selected(s, sel, b.grads != nullptr, b.y != nullptr, cb != nullptr)) continue;
    if (overlap_chain >= 0 && (int)si < overlap_chain && (s.type == ST_WGRAD || s.type == ST_BIASGRAD)) {
      deferred.push_back((int)si);
      continue;
    }
    if (overlap_chain >= 0 && (int)si == overlap_chain) {
      int rc = ensure_streams(); if (rc) return rc;
      CUDA_TRY(cudaEventRecord(P.ev_fork, st));  // everything the deferred kernels read exists once the FIRST chain is done
      const int nl = chain_layers(P, s, sel);   // 0: only tail gradients wanted, the deferred kernels run alone
      if (nl > 0) rc = launch_chain_prefix(P, s, nl, b, st);
      if (rc) return rc;
      for (int k = 0; k < nstreams - 1; ++k) CUDA_TRY(cudaStreamWaitEvent(P.side_stream[k], P.ev_fork, 0));
      int lane = 0;
      for (int di : deferred) {
        const int k = lane++ % (nstreams - 1);
        cudaStream_t ds = P.side_stream[k];
        if (steps[di].type == ST_WGRAD)
          rc = launch_wgrad(steps[di], P.maps()[steps[di].xmap], P.maps()[steps[di].dymap], b, ds, wgrad_cap, lane_of(k + 1));
        else rc = do_biasgrad(steps[di], ds, lane_of(k + 1));
        if (rc) return rc;
      }
      side_dirty = true;
      forked = false;  // the trunk's own weight gradients fork again, behind this chain
      continue;
    }
    if (s.type == ST_DISC_UNPACK) { int rc = join(); if (rc) return rc; }
    if (alternate) {
      // the gradient unpack consumes what the weight-gradient launches of BOTH streams produced: join first (without a
      // bucket callback only the last unpack step launches anything)
      if (s.type == ST_UNPACK && (cb || s.i0 == 0)) { int rc = join(); if (rc) return rc; }
      // the carrier add feeds conv1's weight gradient: the side stream has to be forked again after it
      if (s.type == ST_ADD) forked = false;
    }
    switch (s.type) {
      case ST_CONV:
        return fail(B200SR_ERR_INVALID, "internal: unchained conv step");
      case ST_CHAIN: {
        const int nl = chain_layers(P, s, sel);
        if (nl == 0) break;
        int rc = launch_chain_prefix(P, s, nl, b, st);
        if (rc) return rc;
        forked = false;  // weight gradients behind this chain read what it produces: the side streams fork again after it
        break;
      }
      case ST_WGRAD: {
        cudaStream_t ws = st;
        int lane_ = 0;
        if (alternate) {
          { int rc = ensure_streams(); if (rc) return rc; }
          if (!forked) {  // the side stream starts after everything enqueued so far (the data-gradient chain)
            CUDA_TRY(cudaEventRecord(P.ev_fork, st));
            for (int k = 0; k < nstreams - 1; ++k) CUDA_TRY(cudaStreamWaitEvent(P.side_stream[k], P.ev_fork, 0));
            forked = true;
          }
          lane_ = wcount++ % nstreams;
          if (lane_ > 0) { ws = P.side_stream[lane_ - 1]; side_dirty = true; }
        }
        int rc = launch_wgrad(s, P.maps()[s.xmap], P.maps()[s.dymap], b, ws, wgrad_cap, lane_of(lane_));
        if (rc) return rc;
        break;
      }
      case ST_BIASGRAD: {
        int rc = do_biasgrad(s, st, lane_of(0));
        if (rc) return rc;
        break;
      }
      case ST_UNPACK: {
        // without a bucket callback nobody consumes gradients early: unpack everything once, at the last bucket (conv1)
        int c0 = s.i0, c1 = s.i1;
        if (!cb) {
          if (s.i0 != 0) break;
          c1 = (int)P.unpack_ops.size();
        }
        int blocks = 0;
        for (int c = c0; c < c1; ++c) blocks += P.unpack_ops[c].nblocks;
        unpack_wgrad_kernel<<<blocks, 256, 0, st>>>(P.d_unpack_ops, c0, c1, (const float*)((char*)b.ws + P.o_gw), (float*)b.grads);
        CUDA_TRY(cudaGetLastError());
        if (sel) {  // unwanted convs of a wanted dense block got gradients from its one launch: their entries are zero again
          for (int c = c0; c < c1;) {
            int e = c;
            while (e < c1 && !sel->want[e] && sel->written(e)) ++e;
            if (e == c) { ++c; continue; }
            CUDA_TRY(cudaMemsetAsync((float*)b.grads + P.param_off[2 * c], 0, (size_t)(P.param_off[2 * e] - P.param_off[2 * c]) * 4, st));
            c = e;
          }
        }
        break;
      }
      case ST_ADD: {
        const int tx = (d.width + kTileW - 1) / kTileW, ty = (d.height + kTileH - 1) / kTileH;
        const long long total = (long long)d.batch * tx * ty * 2 * 16 * 128;
        add_carriers_to_bf16_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>((const float*)resolve(s.a, b), (const float*)resolve(s.b, b),
                                                                               (__nv_bfloat16*)resolve(s.c, b), d.batch, d.height, d.width, tx, ty);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_MEMSET:
        CUDA_TRY(cudaMemsetAsync(resolve(s.a, b), 0, (size_t)s.count, st));
        break;
      case ST_INGEST_X: {
        const long long npix = (long long)d.batch * d.height * d.width;
        __nv_bfloat16* out = (__nv_bfloat16*)((char*)b.ws + P.o_xin);
        const int blocks = (int)((npix + 127) / 128);
        if (P.is_disc && d.in_channels == 3) {  // HR-sized RGB inputs: vectorised row stores
#define B200SR_DISC_INGEST(T) (P.dd.fp16 ? disc_ingest_input_kernel<T, 3, true> : disc_ingest_input_kernel<T, 3, false>)<<<blocks, 128, 0, st>>>( \
            (const T*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.height, d.width, out)
          if (x_dtype == B200SR_F32) B200SR_DISC_INGEST(float);
          else if (x_dtype == B200SR_F16) B200SR_DISC_INGEST(__half);
          else if (x_dtype == B200SR_BF16) B200SR_DISC_INGEST(__nv_bfloat16);
          else
            return fail(B200SR_ERR_INVALID, "unknown x dtype %d", x_dtype);
#undef B200SR_DISC_INGEST
          CUDA_TRY(cudaGetLastError());
          break;
        }
        if (x_dtype == B200SR_F32)
          ingest_input_kernel<float><<<blocks, 128, 0, st>>>((const float*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.in_channels, d.height, d.width, out, P.xin_stride);
        else if (x_dtype == B200SR_F16)
          ingest_input_kernel<__half><<<blocks, 128, 0, st>>>((const __half*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.in_channels, d.height, d.width, out, P.xin_stride);
        else if (x_dtype == B200SR_BF16)
          ingest_input_kernel<__nv_bfloat16><<<blocks, 128, 0, st>>>((const __nv_bfloat16*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.in_channels, d.height, d.width, out, P.xin_stride);
        else
          return fail(B200SR_ERR_INVALID, "unknown x dtype %d", x_dtype);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_VGG_INGEST: {
        const long long npix = (long long)P.vd.batch * P.vd.height * P.vd.width;
        VggNorm nm;
        for (int c = 0; c < 3; ++c) { nm.mean[c] = P.vd.mean[c]; nm.std[c] = P.vd.std[c]; }
        nm.mean[3] = 0.f; nm.std[3] = 1.f;
        vgg_ingest_kernel<<<(unsigned)((npix + 127) / 128), 128, 0, st>>>((const float*)x, xs[0], xs[1], xs[2], xs[3], P.vd.batch, P.vd.height, P.vd.width, nm,
                                                                          (__nv_bfloat16*)((char*)b.ws + P.o_xin));
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_VGG_POOL: {
        const long long n = (long long)s.pn * (s.ph >> 1) * (s.pw >> 1) * (s.pc >> 3);
        vgg_maxpool_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (__nv_bfloat16*)resolve(s.c, b), s.pn, s.ph, s.pw, s.pc);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_VGG_POOL_BWD: {
        const long long n = (long long)s.pn * ((s.ph + 1) >> 1) * ((s.pw + 1) >> 1) * (s.pc >> 1);
        vgg_maxpool_relu_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (const __nv_bfloat16*)resolve(s.b, b),
                                                                                (__nv_bfloat16*)resolve(s.c, b), s.pn, s.ph, s.pw, s.pc);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_UP: {
        const dim3 g((unsigned)((s.pw * (s.pc >> 3) + 255) / 256), (unsigned)s.ph, (unsigned)s.pn);
        (P.dd.fp16 ? disc_bilinear_up_kernel<true> : disc_bilinear_up_kernel<false>)<<<g, 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (const __nv_bfloat16*)resolve(s.b, b),
                                                                            (__nv_bfloat16*)resolve(s.c, b), s.pn, s.ph, s.pw, s.pc);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_UP_BWD: {
        const dim3 g((unsigned)((s.pw * (s.pc >> 3) + 255) / 256), (unsigned)s.ph, (unsigned)s.pn);
        (P.dd.fp16 ? disc_bilinear_bwd_kernel<true> : disc_bilinear_bwd_kernel<false>)<<<g, 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (const __nv_bfloat16*)resolve(s.b, b),
                                                                             (__nv_bfloat16*)resolve(s.c, b), (__nv_bfloat16*)resolve(s.d2, b), s.pn, s.ph, s.pw, s.pc);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_ADD: {
        const long long n = (long long)s.pn * s.ph * s.pw * (s.pc >> 3);
        (P.dd.fp16 ? disc_add_u_kernel<true> : disc_add_u_kernel<false>)<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (const __nv_bfloat16*)resolve(s.b, b),
                                                                      (__nv_bfloat16*)resolve(s.c, b), s.pn, s.ph, s.pw, s.pc);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_MASK: {
        const long long n8 = (long long)s.pn * s.ph * s.pw * (s.pc >> 3);
        (P.dd.fp16 ? disc_lrelu_mask_kernel<true> : disc_lrelu_mask_kernel<false>)<<<(unsigned)((n8 + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)resolve(s.a, b), (const __nv_bfloat16*)resolve(s.b, b),
                                                                           (__nv_bfloat16*)resolve(s.c, b), n8);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_INGEST_DY: {
        const long long npix = (long long)s.pn * s.ph * s.pw;
        (P.dd.fp16 ? disc_ingest_grad_kernel<true> : disc_ingest_grad_kernel<false>)<<<(unsigned)((npix + 127) / 128), 128, 0, st>>>((const float*)b.dy, s.pn, s.pc, s.ph, s.pw, (__nv_bfloat16*)resolve(s.c, b), 64);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_DISC_UNPACK: {
        int blocks = 0;
        for (const UnpackOp& u : P.unpack_ops) blocks += u.nblocks;
        unpack_wgrad_kernel<<<blocks, 256, 0, st>>>(P.d_unpack_ops, 0, (int)P.unpack_ops.size(), (const float*)((char*)b.ws + P.o_gw), (float*)b.grads);
        CUDA_TRY(cudaGetLastError());
        for (const UnpackOp& u : P.unpack_ops) {
          if (u.fold != 2) continue;
          const long long n = 16LL * u.co * u.ci;
          unpack_wgrad_down_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float*)((char*)b.ws + P.o_gw) + u.src_off, (float*)b.grads + u.dst_off, u.co, u.ci, u.co_pad);
          CUDA_TRY(cudaGetLastError());
        }
        break;
      }
      case ST_TRUNK_INGEST: {
        const int tx = (d.width + kTileW - 1) / kTileW, ty = (d.height + kTileH - 1) / kTileH;
        const int blocks = d.batch * tx * ty;  // one 256-thread block per 8 x 32 tile
        float* carrier = (float*)resolve(s.a, b);
        __nv_bfloat16* shadow = (__nv_bfloat16*)resolve(s.c, b);
        if (s.b.kind == RK_DY) {  // dy: fp32 contiguous NCHW
          const long long plane = (long long)d.height * d.width;
          trunk_ingest_kernel<float><<<blocks, 256, 0, st>>>((const float*)b.dy, 64 * plane, plane, d.width, 1, d.batch, d.height, d.width, tx, ty,
                                                             s.scale, carrier, shadow, 192);
        } else if (x_dtype == B200SR_F32) {
          trunk_ingest_kernel<float><<<blocks, 256, 0, st>>>((const float*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.height, d.width, tx, ty, s.scale,
                                                             carrier, shadow, 192);
        } else if (x_dtype == B200SR_F16) {
          trunk_ingest_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.height, d.width, tx, ty, s.scale,
                                                              carrier, shadow, 192);
        } else if (x_dtype == B200SR_BF16) {
          trunk_ingest_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, xs[0], xs[1], xs[2], xs[3], d.batch, d.height, d.width, tx,
                                                                     ty, s.scale, carrier, shadow, 192);
        } else {
          return fail(B200SR_ERR_INVALID, "unknown x dtype %d", x_dtype);
        }
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_TRUNK_EXPORT: {  // to the caller's y (forward) or dx (backward)
        const int tx = (d.width + kTileW - 1) / kTileW, ty = (d.height + kTileH - 1) / kTileH;
        trunk_export_kernel<<<d.batch * tx * ty, 256, 0, st>>>((const float*)resolve(s.a, b), (float*)b.y, d.batch, d.height, d.width, tx, ty);
        CUDA_TRY(cudaGetLastError());
        break;
      }
      case ST_INGEST_DY: {
        const int hH = d.height << P.L, hW = d.width << P.L;
        const long long npix = (long long)d.batch * hH * hW;
        (P.unclamped ? ingest_grad_kernel<false> : ingest_grad_kernel<true>)<<<(int)((npix + 127) / 128), 128, 0, st>>>(
            (const float*)b.dy, (const unsigned char*)((char*)b.ws + P.o_cmask), d.batch, d.out_channels, hH, hW,
            (__nv_bfloat16*)((char*)b.ws + P.o_dyp), 64);
        CUDA_TRY(cudaGetLastError());
        break;
      }
    }
    if (cb && s.cb_count > 0) cb(user, s.cb_off, s.cb_count);
  }
  return join();
}

// ------------------------------------------------------------------------------------------------ VGG19 feature plan
// torchvision vgg19().features up to conv5_4: sixteen 3x3 convs (+ReLU), 2x2 max-pools after convs 1, 3, 7, 11.
static const int kVggCin[16] = {3, 64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512};
static const int kVggCout[16] = {64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512};
static const bool kVggPoolAfter[16] = {false, true, false, true, false, false, false, true, false, false, false, true, false, false, false, false};

static int build_vgg_plan(b200sr_plan& P) {
  const b200sr_vgg_desc& v = P.vd;
  if (v.batch < 1 || v.height < 1 || v.width < 1) return fail(B200SR_ERR_INVALID, "bad geometry");
  if (v.last_conv < 0 || v.last_conv > 15) return fail(B200SR_ERR_INVALID, "last_conv must be in [0, 15]");
  if (v.grad_conv > v.last_conv || v.grad_images > v.batch) return fail(B200SR_ERR_INVALID, "bad gradient request");
  const bool bwd = v.grad_conv >= 0 && v.grad_images > 0;
  P.is_vgg = true;
  P.reassoc = false;
  P.groups = v.batch >= 2 ? 2 : 1;
  memset(&P.d, 0, sizeof(P.d));
  P.d.batch = v.batch; P.d.height = v.height; P.d.width = v.width; P.d.training = bwd ? 1 : 0;
  const int NL = v.last_conv + 1;
  const int N = v.batch, NB = v.grad_images;
  Builder B(P);
  P.param_off.assign(2 * NL + 1, 0);
  {
    long long off = 0;
    for (int l = 0; l < NL; ++l) {
      P.param_off[2 * l] = off; off += 9LL * kVggCin[l] * kVggCout[l];
      P.param_off[2 * l + 1] = off; off += kVggCout[l];
    }
    P.param_off[2 * NL] = off;
  }
  int h = v.height, w = v.width;
  P.xin_stride = 64;
  P.o_xin = B.alloc("xin", (long long)N * h * w * 64 * 2);
  std::vector<long long> o_act(NL, 0), o_pool(NL, 0);
  for (int l = 0; l < NL; ++l) {
    if (h < 1 || w < 1) return fail(B200SR_ERR_INVALID, "input too small for conv %d", l);
    P.vgg_h[l] = h; P.vgg_w[l] = w;
    const std::string ls = std::to_string(l);
    o_act[l] = B.alloc("A" + ls, (long long)N * h * w * kVggCout[l] * 2);
    if ((v.feat_mask >> l) & 1) P.o_vgg_feat[l] = B.alloc("F" + ls, (long long)N * h * w * kVggCout[l] * 4) + 1;  // +1: 0 means absent
    if (kVggPoolAfter[l] && l + 1 < NL) {
      o_pool[l] = B.alloc("P" + ls, (long long)N * (h >> 1) * (w >> 1) * kVggCout[l] * 2);
      h >>= 1; w >>= 1;
    }
  }
  std::vector<long long> o_gpool(NL, 0);
  if (bwd) {
    for (int l = 0; l <= v.grad_conv; ++l) {
      const std::string ls = std::to_string(l);
      P.o_vgg_g[l] = B.alloc("G" + ls, (long long)NB * P.vgg_h[l] * P.vgg_w[l] * kVggCout[l] * 2) + 1;
      if (kVggPoolAfter[l] && l + 1 <= v.grad_conv) o_gpool[l] = B.alloc("GP" + ls, (long long)NB * (P.vgg_h[l] >> 1) * (P.vgg_w[l] >> 1) * kVggCout[l] * 2);
    }
  }
  if (P.det) P.o_det = B.alloc(kVggL1MaxBlocks * sizeof(double));  // per-block partials of b200sr_vgg_feature_l1
  P.ws_bytes = B.cursor;
  auto packed_bias = [&](long long off_floats) { Ref r; r.kind = RK_PACKED; r.off = -1 - off_floats; return r; };
  auto conv_step = [&](int amap, const ConvParams& cp) {
    Step s; s.type = ST_CONV; s.amap = amap; s.wmap = 0; s.cp = cp; s.grid = dim3(1, 1, 1); s.smem = 0;
    return s;
  };
  // ---- forward
  { Step s; s.type = ST_VGG_INGEST; P.fwd.push_back(s); }
  for (int l = 0; l < NL; ++l) {
    const int cin = kVggCin[l], cout = kVggCout[l], hh = P.vgg_h[l], ww = P.vgg_w[l];
    const int n_cols = (cout % 128 == 0) ? 128 : 64;  // column groups of 128 for the wide layers, else 64
    PackOp op; memset(&op, 0, sizeof(op));
    op.n_total = cout; op.n_cols = n_cols; op.n_valid = cout; op.mode = kPackFwd;
    int amap, chunks, ksl;
    if (l == 0) {  // [hi | lo | hi] input x [w_hi | w_hi | w_lo] weights: fp32-accurate products from bf16 MMAs
      op.num_chunks = 1; op.nseg = 3;
      op.seg[0] = seg(0, 3, 0, cout, 3, 0, 0, 0); op.seg[1] = seg(3, 3, 0, cout, 3, 0, 0, 0); op.seg[2] = seg(6, 3, 0, cout, 3, 0, 0, 1);
      amap = B.add_map(P.o_xin, 64, 64, N, hh, ww, kABoxRows); chunks = 1; ksl = 1;
    } else {
      const long long in_off = (kVggPoolAfter[l - 1]) ? o_pool[l - 1] : o_act[l - 1];
      op.num_chunks = cin / 64; op.nseg = 1;
      op.seg[0] = seg(0, cin, 2 * l, cout, cin, 0, 0, 0);
      amap = B.add_map(in_off, cin, cin, N, hh, ww, kABoxRows); chunks = cin / 64; ksl = 4;
    }
    const int row0 = B.add_pack(op);
    ConvParams cp = base_conv_params(N, hh, ww, chunks, ksl, 0, 1 << 20, row0, n_cols, cout);
    Step s = conv_step(amap, cp);
    s.bias = packed_bias(B.add_bias(cout, 2 * l + 1, cout, 0));
    s.cp.epi.act = 2;  // ReLU
    s.ob = ws(o_act[l]); s.cp.epi.ob_stride = cout; s.cp.epi.ob_coff = 0;
    if (P.o_vgg_feat[l]) {
      s.feat = ws(P.o_vgg_feat[l] - 1); s.cp.epi.feat_stride = cout;
      // torchvision's feature extractor returns the conv's output tensor, which the NEXT module -- ReLU(inplace=True) -- then
      // overwrites: every node but the one that ends the extracted graph is effectively read AFTER the ReLU
      if (l < v.last_conv) s.cp.epi.mask_relu |= 2;
    }
    P.fwd.push_back(s);
    if (kVggPoolAfter[l] && l + 1 < NL) {
      Step pl; pl.type = ST_VGG_POOL; pl.a = ws(o_act[l]); pl.c = ws(o_pool[l]); pl.pn = N; pl.ph = hh; pl.pw = ww; pl.pc = cout;
      P.fwd.push_back(pl);
    }
  }
  // ---- backward (data gradients only: the VGG weights are frozen): G[l] = gradient w.r.t. conv l's pre-activation output
  if (bwd) {
    for (int l = v.grad_conv; l >= 0; --l) {
      const int cin = kVggCin[l], cout = kVggCout[l], hh = P.vgg_h[l], ww = P.vgg_w[l];
      const int nin = (l == 0) ? 16 : cin;  // dgrad output channels (conv 0: 3 padded to 16, stored NCHW fp32 to dx)
      const int n_cols = (l == 0) ? 16 : ((cin % 128 == 0) ? 128 : 64);
      PackOp op; memset(&op, 0, sizeof(op));
      op.n_total = nin; op.n_cols = n_cols; op.n_valid = (l == 0) ? 3 : cin; op.num_chunks = cout / 64; op.mode = kPackDgrad; op.nseg = 1;
      op.seg[0] = seg(0, cout, 2 * l, cout, cin, 0, 0, 0);
      const int row0 = B.add_pack(op);
      ConvParams cp = base_conv_params(NB, hh, ww, cout / 64, 4, 0, 1 << 20, row0, n_cols, nin);
      Step s = conv_step(B.add_map(P.o_vgg_g[l] - 1, cout, cout, NB, hh, ww, kABoxRows), cp);
      if (l == 0) {
        s.cp.epi.store_mode = kStoreNCHW; s.cp.epi.n_valid = 3; s.of.kind = RK_Y;
        P.bwd.push_back(s);
      } else if (kVggPoolAfter[l - 1]) {
        // conv l reads the POOLED activation of conv l-1: its data gradient lives on the pooled lattice, then pool + ReLU backward
        s.ob = ws(o_gpool[l - 1]); s.cp.epi.ob_stride = cin; s.cp.epi.ob_coff = 0;
        P.bwd.push_back(s);
        Step pb; pb.type = ST_VGG_POOL_BWD; pb.a = ws(o_act[l - 1]); pb.b = ws(o_gpool[l - 1]); pb.c = ws(P.o_vgg_g[l - 1] - 1);
        pb.pn = NB; pb.ph = P.vgg_h[l - 1]; pb.pw = P.vgg_w[l - 1]; pb.pc = cin;
        P.bwd.push_back(pb);
      } else {
        s.mask = ws(o_act[l - 1]); s.cp.epi.mask_stride = cin; s.cp.epi.mask_coff = 0; s.cp.epi.mask_relu = 1;
        s.ob = ws(P.o_vgg_g[l - 1] - 1); s.cp.epi.ob_stride = cin; s.cp.epi.ob_coff = 0;
        P.bwd.push_back(s);
      }
    }
  }
  const long long bias_base = align_up(P.total_rows * 128, 1024);
  P.packed_bytes = bias_base + P.bias_floats * 4;
  auto fix = [&](std::vector<Step>& vv) {
    for (Step& s : vv)
      if (s.bias.kind == RK_PACKED) s.bias.off = bias_base + (-1 - s.bias.off) * 4;
  };
  fix(P.fwd); fix(P.bwd);
  auto chainify = [&](std::vector<Step>& vv) {
    std::vector<Step> out;
    for (Step& s : vv) {
      if (s.type != ST_CONV) { out.push_back(s); continue; }
      if (out.empty() || out.back().type != ST_CHAIN) {
        Step c; c.type = ST_CHAIN; c.layer0 = (int)P.layer_steps.size(); c.nlayers = 0; c.chain_grid = 0;
        out.push_back(c);
      }
      out.back().nlayers++;
      const int work = s.cp.num_tiles * s.cp.col_groups;
      if (work > out.back().chain_grid) out.back().chain_grid = work;
      P.layer_steps.push_back(s);
    }
    vv.swap(out);
  };
  chainify(P.fwd); chainify(P.bwd);
  return 0;
}


// ------------------------------------------------------------------------------------------------ U-Net discriminator plan
// DiscriminatorUNet (BSRGAN/model.py:91-167).  Conv order = parameter order: 0 conv1, 1..3 down1..3, 4..6 up1..3, 7 conv2, 8 conv3, 9 conv4.
// Tensors that feed a stride-2 conv (out1, down1, down2) live in U layout ([N, h/2, w/2, 4C], channel (py*2+px)*C + c): the 4x4
// stride-2 conv is then an ordinary 3x3 conv over 4C channels (weights packed with structural zeros, kPackDownFwd), its data
// gradient an ordinary 3x3 dgrad whose 4C output columns are pixel-shuffled back to the plain layout on store, and its weight
// gradient the ordinary 3x3 wgrad over the U-layout input, gathered to [co][c][4][4] by unpack_wgrad_down_kernel.
static int build_disc_plan(b200sr_plan& P) {
  const b200sr_disc_desc& v = P.dd;
  if (v.channels != 64) return fail(B200SR_ERR_INVALID, "only channels=64 is supported (got %d)", v.channels);
  if (v.in_channels < 1 || v.in_channels > 16 || v.out_channels < 1 || v.out_channels > 16) return fail(B200SR_ERR_INVALID, "in/out channels must be in [1,16]");
  if (v.batch < 1 || v.height < 8 || v.width < 8 || (v.height & 7) || (v.width & 7)) return fail(B200SR_ERR_INVALID, "height and width must be multiples of 8");
  P.is_disc = true;
  P.reassoc = false;
  P.groups = v.batch >= 2 ? 2 : 1;
  if (v.in_channels != 3) P.dd.fp16 = 0;  // the fp16 ingest kernel is specialised for RGB inputs; other widths run in bf16
  memset(&P.d, 0, sizeof(P.d));
  P.d.in_channels = v.in_channels; P.d.out_channels = v.out_channels; P.d.channels = 64; P.d.growth = 32;
  P.d.batch = v.batch; P.d.height = v.height; P.d.width = v.width; P.d.training = v.training;
  const bool train = v.training != 0;
  const int N = v.batch, H = v.height, W = v.width, CI = v.in_channels, CO = v.out_channels;
  const int nconv = 10;
  // conv geometry: output channels, input channels (of the reference tensor), kernel size, lattice the conv RUNS on (level: H >> lvl)
  const int cO[10] = {64, 128, 256, 512, 256, 128, 64, 64, 64, CO};
  const int cI[10] = {CI, 64, 128, 256, 512, 256, 128, 64, 64, 64};
  const int cK[10] = {3, 4, 4, 4, 3, 3, 3, 3, 3, 3};
  const int cLvl[10] = {0, 1, 2, 3, 2, 1, 0, 0, 0, 0};
  const bool cBias[10] = {true, false, false, false, false, false, false, false, false, true};
  P.param_off.assign(2 * nconv + 1, 0);
  {
    long long off = 0;
    for (int c = 0; c < nconv; ++c) {
      P.param_off[2 * c] = off; off += (long long)cO[c] * cI[c] * cK[c] * cK[c];
      P.param_off[2 * c + 1] = off; off += cBias[c] ? cO[c] : 0;
    }
    P.param_off[2 * nconv] = off;
  }
  auto lh = [&](int lvl) { return H >> lvl; };
  auto lw = [&](int lvl) { return W >> lvl; };
  auto npx = [&](int lvl) { return (long long)N * lh(lvl) * lw(lvl); };
  Builder B(P);
  P.xin_stride = 64;
  P.o_xin = B.alloc("xin", npx(0) * 64 * 2);
  // forward activations (all kept: the backward pass reads every one of them)
  const long long T0u = B.alloc("T0u", npx(0) * 64 * 2), T1u = B.alloc("T1u", npx(1) * 128 * 2), T2u = B.alloc("T2u", npx(2) * 256 * 2),
                  T3 = B.alloc("T3", npx(3) * 512 * 2);
  const long long B1 = B.alloc("B1", npx(2) * 512 * 2), A1 = B.alloc("A1", npx(2) * 256 * 2), B2 = B.alloc("B2", npx(1) * 256 * 2),
                  A2 = B.alloc("A2", npx(1) * 128 * 2);
  const long long B3 = B.alloc("B3", npx(0) * 128 * 2), A3 = B.alloc("A3", npx(0) * 64 * 2), S3 = B.alloc("S3", npx(0) * 64 * 2),
                  A4 = B.alloc("A4", npx(0) * 64 * 2), A5 = B.alloc("A5", npx(0) * 64 * 2);
  long long DYP = 0, G5 = 0, G4 = 0, GS3 = 0, G3 = 0, GB3 = 0, GS2 = 0, GA2 = 0, GB2 = 0, GS1 = 0, GA1 = 0, GB1 = 0, GT3 = 0, GT2 = 0, GT1 = 0, G0 = 0;
  // effective (as computed) input channels / staged output channels of every conv's weight gradient
  int eI[10], coPad[10];
  for (int c = 0; c < nconv; ++c) { eI[c] = (cK[c] == 4) ? 4 * cI[c] : cI[c]; coPad[c] = (int)align_up(cO[c], 4); }
  if (train) {
    DYP = B.alloc("DYP", npx(0) * 64 * 2); G5 = B.alloc("G5", npx(0) * 64 * 2); G4 = B.alloc("G4", npx(0) * 64 * 2);
    GS3 = B.alloc("GS3", npx(0) * 64 * 2); G3 = B.alloc("G3", npx(0) * 64 * 2);
    GB3 = B.alloc("GB3", npx(0) * 128 * 2); GS2 = B.alloc("GS2", npx(1) * 128 * 2); GA2 = B.alloc("GA2", npx(1) * 128 * 2);
    GB2 = B.alloc("GB2", npx(1) * 256 * 2);
    GS1 = B.alloc("GS1", npx(2) * 256 * 2); GA1 = B.alloc("GA1", npx(2) * 256 * 2); GB1 = B.alloc("GB1", npx(2) * 512 * 2);
    GT3 = B.alloc("GT3", npx(3) * 512 * 2);
    GT2 = B.alloc("GT2", npx(2) * 256 * 2); GT1 = B.alloc("GT1", npx(1) * 128 * 2); G0 = B.alloc("G0", npx(0) * 64 * 2);
    long long off = 0;
    int blocks = 0;
    P.gw_off.assign(nconv, 0);
    for (int c = 0; c < nconv; ++c) {
      P.gw_off[c] = off;
      UnpackOp u;
      u.src_off = off; u.dst_off = P.param_off[2 * c]; u.co = cO[c]; u.ci = cI[c]; u.co_pad = coPad[c]; u.fold = (cK[c] == 4) ? 2 : 0;
      u.block0 = blocks; u.nblocks = (cK[c] == 4) ? 0 : ((cO[c] + 31) / 32) * ((cI[c] + 31) / 32);  // fold 2: unpack_wgrad_down_kernel
      blocks += u.nblocks;
      P.unpack_ops.push_back(u);
      off += align_up(9LL * eI[c] * coPad[c], 4);
    }
    P.o_gw = B.alloc(off * 4);
    P.gw_bytes = off * 4;
  }
  P.ws_bytes = B.cursor;

  auto packed_bias = [&](long long off_floats) { Ref r; r.kind = RK_PACKED; r.off = -1 - off_floats; return r; };
  auto conv_step = [&](int amap, const ConvParams& cp) {
    Step s; s.type = ST_CONV; s.amap = amap; s.wmap = 0; s.cp = cp; s.grid = dim3(1, 1, 1); s.smem = 0;
    return s;
  };
  // generic layer: input buffer [.., c_in] (plain or U layout: the conv does not care), K = c_in channels in chunks of 64
  auto fwd_conv = [&](int c, long long in_off, int c_in, int mode, long long out_off, int out_stride, int act) {
    const int lvl = cLvl[c], cout = cO[c];
    // column groups of 128 for the wide stride-1 layers (an N = 128 tcgen05.mma does twice the work of an N = 64 one in 4/3 of the
    // time, and the activation tile is re-read half as often); the 4-tap stride-2 stages stay at 64 columns (32 KB per stage)
    const int n_total = (c == 9) ? 16 : cout, n_cols = (c == 9) ? 16 : ((mode == kPackFwd && cout % 128 == 0) ? 128 : 64);
    PackOp op; memset(&op, 0, sizeof(op));
    op.n_total = n_total; op.n_cols = n_cols; op.n_valid = cout; op.mode = mode; op.num_chunks = c_in / 64; op.nseg = 1;
    op.seg[0] = seg(0, c_in, 2 * c, cout, cI[c], 0, 0, 0);
    if (mode == kPackDownFwd) op.down_c = cI[c];
    const int row0 = B.add_pack(op);
    ConvParams cp = base_conv_params(N, lh(lvl), lw(lvl), op.num_chunks, 4, 0, 1 << 20, row0, n_cols, n_total);
    if (op.down_c > 0) { cp.w_taps = 4; cp.down_mode = 1; cp.down_c64 = cI[c] / 64; }
    Step s = conv_step(B.add_map(in_off, c_in, c_in, N, lh(lvl), lw(lvl), kABoxRows), cp);
    if (cBias[c]) s.bias = packed_bias(B.add_bias(n_total, 2 * c + 1, cout, 0));
    s.cp.epi.act = act;
    if (out_off >= 0) { s.ob = ws(out_off); s.cp.epi.ob_stride = out_stride; s.cp.epi.ob_coff = 0; }
    return s;
  };
  auto up_step = [&](long long in_off, long long skip_u, long long out_off, int lvl_in, int C) {
    Step s; s.type = ST_DISC_UP; s.a = ws(in_off); if (skip_u >= 0) s.b = ws(skip_u); s.c = ws(out_off);
    s.pn = N; s.ph = lh(lvl_in); s.pw = lw(lvl_in); s.pc = C;
    return s;
  };
  // ================================================================ forward ================================================================
  { Step s; s.type = ST_INGEST_X; P.fwd.push_back(s); }
  {  // conv1: [hi | lo | hi] input x [w_hi | w_hi | w_lo] weights, no activation, stored in U layout for down1
    PackOp op; memset(&op, 0, sizeof(op));
    op.n_total = 64; op.n_cols = 64; op.n_valid = 64; op.mode = kPackFwd; op.num_chunks = 1; op.nseg = 3;
    op.seg[0] = seg(0, CI, 0, 64, CI, 0, 0, 0); op.seg[1] = seg(CI, CI, 0, 64, CI, 0, 0, 0); op.seg[2] = seg(2 * CI, CI, 0, 64, CI, 0, 0, 1);
    const int row0 = B.add_pack(op);
    ConvParams cp = base_conv_params(N, H, W, 1, (3 * CI + 15) / 16, 0, 1 << 20, row0, 64, 64);
    Step s = conv_step(B.add_map(P.o_xin, 64, 64, N, H, W, kABoxRows), cp);
    s.bias = packed_bias(B.add_bias(64, 1, 64, 0));
    s.ob = ws(T0u); s.cp.epi.ob_stride = 256; s.cp.epi.store_mode = kStoreUnshuffle; s.cp.epi.shuf_c = 64;
    P.fwd.push_back(s);
  }
  {
    Step d1 = fwd_conv(1, T0u, 256, kPackDownFwd, T1u, 512, 1);
    d1.cp.epi.store_mode = kStoreUnshuffle; d1.cp.epi.shuf_c = 128;
    P.fwd.push_back(d1);
    Step d2 = fwd_conv(2, T1u, 512, kPackDownFwd, T2u, 1024, 1);
    d2.cp.epi.store_mode = kStoreUnshuffle; d2.cp.epi.shuf_c = 256;
    P.fwd.push_back(d2);
    P.fwd.push_back(fwd_conv(3, T2u, 1024, kPackDownFwd, T3, 512, 1));
  }
  P.fwd.push_back(up_step(T3, -1, B1, 3, 512));
  P.fwd.push_back(fwd_conv(4, B1, 512, kPackFwd, A1, 256, 1));
  P.fwd.push_back(up_step(A1, T2u, B2, 2, 256));        // (up1 + down2) upsampled
  P.fwd.push_back(fwd_conv(5, B2, 256, kPackFwd, A2, 128, 1));
  P.fwd.push_back(up_step(A2, T1u, B3, 1, 128));        // (up2 + down1) upsampled
  P.fwd.push_back(fwd_conv(6, B3, 128, kPackFwd, A3, 64, 1));
  { Step s; s.type = ST_DISC_ADD; s.a = ws(A3); s.b = ws(T0u); s.c = ws(S3); s.pn = N; s.ph = H; s.pw = W; s.pc = 64; P.fwd.push_back(s); }  // up3 + out1
  P.fwd.push_back(fwd_conv(7, S3, 64, kPackFwd, A4, 64, 1));
  P.fwd.push_back(fwd_conv(8, A4, 64, kPackFwd, A5, 64, 1));
  {
    Step s = fwd_conv(9, A5, 64, kPackFwd, -1, 0, 0);
    s.cp.epi.store_mode = kStoreNCHW; s.cp.epi.n_valid = CO; s.of.kind = RK_Y;
    P.fwd.push_back(s);
  }
  // ================================================================ backward ===============================================================
  if (train) {
    // data gradient of conv c: reads the gradient w.r.t. its pre-activation output (K = k_in valid channels of a buffer with
    // `in_stride` channels), produces n_total input-gradient columns
    auto dgrad_conv = [&](int c, long long in_off, int k_in, int in_stride, int mode, int n_total, int n_cols, int n_valid) {
      const int lvl = cLvl[c];
      PackOp op; memset(&op, 0, sizeof(op));
      op.n_total = n_total; op.n_cols = n_cols; op.n_valid = n_valid; op.mode = mode; op.num_chunks = (k_in + 63) / 64; op.nseg = 1;
      op.seg[0] = seg(0, cO[c], 2 * c, cO[c], cI[c], 0, 0, 0);
      if (mode == kPackDownDgrad) op.down_c = cI[c];
      const int row0 = B.add_pack(op);
      const int kl = k_in - 64 * (op.num_chunks - 1);
      ConvParams cp = base_conv_params(N, lh(lvl), lw(lvl), op.num_chunks, (kl + 15) / 16, 0, 1 << 20, row0, n_cols, n_total);
      if (op.down_c > 0) { cp.w_taps = 4; cp.down_mode = 2; cp.down_c64 = cI[c] / 64; }
      return conv_step(B.add_map(in_off, k_in, in_stride, N, lh(lvl), lw(lvl), kABoxRows), cp);
    };
    auto out_to = [&](Step& s, long long off, int stride) { s.ob = ws(off); s.cp.epi.ob_stride = stride; s.cp.epi.ob_coff = 0; };
    auto mask_by = [&](Step& s, long long off, int stride) { s.mask = ws(off); s.cp.epi.mask_stride = stride; s.cp.epi.mask_coff = 0; };
    auto up_bwd = [&](long long gout, long long act, long long gs, long long ga, int lvl_in, int C) {
      Step s; s.type = ST_DISC_UP_BWD; s.a = ws(gout); s.b = ws(act); if (gs >= 0) s.c = ws(gs); s.d2 = ws(ga);
      s.pn = N; s.ph = lh(lvl_in); s.pw = lw(lvl_in); s.pc = C;
      return s;
    };
    {
      Step m; m.type = ST_MEMSET; m.a.kind = RK_GRADS; m.a.off = 0; m.count = P.param_off[2 * nconv] * 4; m.needs_wgrad = true;
      P.bwd.push_back(m);
      Step m2; m2.type = ST_MEMSET; m2.a = ws(P.o_gw); m2.count = P.gw_bytes; m2.needs_wgrad = true;
      P.bwd.push_back(m2);
      Step g; g.type = ST_DISC_INGEST_DY; g.c = ws(DYP); g.pn = N; g.ph = H; g.pw = W; g.pc = CO;
      P.bwd.push_back(g);
    }
    { Step s = dgrad_conv(9, DYP, 16, 64, kPackDgrad, 64, 64, 64); s.cp.ksteps_last = 1; mask_by(s, A5, 64); out_to(s, G5, 64); P.bwd.push_back(s); }
    { Step s = dgrad_conv(8, G5, 64, 64, kPackDgrad, 64, 64, 64); mask_by(s, A4, 64); out_to(s, G4, 64); P.bwd.push_back(s); }
    { Step s = dgrad_conv(7, G4, 64, 64, kPackDgrad, 64, 64, 64); out_to(s, GS3, 64); P.bwd.push_back(s); }   // gradient of (up3 + out1)
    { Step s; s.type = ST_DISC_MASK; s.a = ws(GS3); s.b = ws(A3); s.c = ws(G3); s.pn = N; s.ph = H; s.pw = W; s.pc = 64; P.bwd.push_back(s); }
    { Step s = dgrad_conv(6, G3, 64, 64, kPackDgrad, 128, 128, 128); out_to(s, GB3, 128); P.bwd.push_back(s); }
    P.bwd.push_back(up_bwd(GB3, A2, GS2, GA2, 1, 128));
    { Step s = dgrad_conv(5, GA2, 128, 128, kPackDgrad, 256, 128, 256); out_to(s, GB2, 256); P.bwd.push_back(s); }
    P.bwd.push_back(up_bwd(GB2, A1, GS1, GA1, 2, 256));
    { Step s = dgrad_conv(4, GA1, 256, 256, kPackDgrad, 512, 128, 512); out_to(s, GB1, 512); P.bwd.push_back(s); }
    P.bwd.push_back(up_bwd(GB1, T3, -1, GT3, 3, 512));
    // stride-2 convs: 4C output columns on the conv's own lattice, pixel-shuffled to the plain layout of the finer lattice; the
    // skip connection's gradient (plain layout, finer lattice) joins before the LeakyReLU derivative of the U-layout activation
    {
      Step s = dgrad_conv(3, GT3, 512, 512, kPackDownDgrad, 1024, 64, 1024);
      s.cp.epi.store_mode = kStoreShuffle; s.cp.epi.shuf_c = 256; out_to(s, GT2, 256);
      s.resb = ws(GS1); s.cp.epi.res_bf16_stride = 256; mask_by(s, T2u, 1024);
      P.bwd.push_back(s);
    }
    {
      Step s = dgrad_conv(2, GT2, 256, 256, kPackDownDgrad, 512, 64, 512);
      s.cp.epi.store_mode = kStoreShuffle; s.cp.epi.shuf_c = 128; out_to(s, GT1, 128);
      s.resb = ws(GS2); s.cp.epi.res_bf16_stride = 128; mask_by(s, T1u, 512);
      P.bwd.push_back(s);
    }
    {
      Step s = dgrad_conv(1, GT1, 128, 128, kPackDownDgrad, 256, 64, 256);   // out1 has no activation: no mask
      s.cp.epi.store_mode = kStoreShuffle; s.cp.epi.shuf_c = 64; out_to(s, G0, 64);
      s.resb = ws(GS3); s.cp.epi.res_bf16_stride = 64;
      P.bwd.push_back(s);
    }
    {  // gradient w.r.t. the input image (the generator update): conv1's data gradient, fp32 NCHW
      Step s = dgrad_conv(0, G0, 64, 64, kPackDgrad, 16, 16, CI);
      s.cp.epi.store_mode = kStoreNCHW; s.cp.epi.n_valid = CI; s.of.kind = RK_Y; s.needs_dx = true;
      P.bwd.push_back(s);
    }
    // ---- weight gradients: blocks of (<= 128 input channels) x (<= 128 output channels), four problems per launch
    auto wref = [&](int c, long long extra_floats) { return ws(P.o_gw + (P.gw_off[c] + extra_floats) * 4); };
    auto wgrad_conv = [&](int c, long long x_off, int x_cvalid, int x_cpix, long long dy_off, int dy_cvalid, int dy_cpix, int ci_total) {
      const int lvl = cLvl[c];
      const int n = N, h = lh(lvl), w = lw(lvl);
      const int ncols_all = (c == 9) ? 16 : cO[c];
      Step cur; bool open = false;
      for (int cib = 0; cib < x_cvalid; cib += 128) {
        for (int cob = 0; cob < ncols_all; cob += 128) {
          if (!open) {
            cur = Step(); cur.type = ST_WGRAD; cur.needs_wgrad = true;
            cur.xmap = B.add_map(x_off, x_cvalid, x_cpix, n, h, w, kWgXRows);
            cur.dymap = B.add_map(dy_off, dy_cvalid, dy_cpix, n, h, w, kWgTileH);
            WgradBatch& wb = cur.wb; memset(&wb, 0, sizeof(wb));
            wb.N = n; wb.H = h; wb.W = w;
            wb.tiles_x = (w + kTileW - 1) / kTileW; wb.tiles_y = (h + kWgTileH - 1) / kWgTileH; wb.num_tiles = n * wb.tiles_x * wb.tiles_y;
            open = true;
          }
          const int ncols = std::min(128, ncols_all - cob);
          const int pj = cur.wb.num_problems++;
          WgradParams& wp = cur.wb.prob[pj];
          wp.b_c0 = cob; wp.n_cols = ncols; wp.n_blocks = (ncols + 63) / 64;
          wgrad_set_a(wp, cib, (x_cvalid - cib > 64) ? 2 : 1);
          WgradSegment& g = wp.seg[0];
          g.col_begin = 0; g.col_end = ncols; g.out = nullptr; g.ci_total = ci_total; g.ci0 = cib; g.co_pad = coPad[c];
          if (cK[c] == 4) {
            // U-layout input channels [cib, cib + 128): phases of the first and the last channel of the block (equal when a phase
            // is >= 128 channels wide); a phase (py, px) keeps tap rows {1,2} / {0,1} for py = 0 / 1, columns alike
            const int hi = std::min(cib + 128, x_cvalid) - 1;
            const int p0 = cib / cI[c], p1 = hi / cI[c];
            int dym = 0, dxm = 0;
            for (int ph = p0; ph <= p1; ++ph) { dym |= (ph >> 1) ? 3 : 6; dxm |= (ph & 1) ? 3 : 6; }
            wp.dy_mask = dym; wp.dx_mask = dxm;
          }
          cur.wseg_out[pj][0] = wref(c, (long long)(cob / 4) * ci_total * 4);
          wp.num_seg = 1;
          if (cur.wb.num_problems == 4) { P.bwd.push_back(cur); open = false; }
        }
      }
      if (open) P.bwd.push_back(cur);
    };
    auto bias_grad = [&](int c, long long g_off, int ncols, int n_valid) {
      Step s; s.type = ST_BIASGRAD; s.needs_wgrad = true;
      memset(&s.bp, 0, sizeof(s.bp));
      s.bg_g = ws(g_off); s.bp.P = npx(0); s.bp.stride = 64; s.bp.c0 = 0; s.bp.ncols = ncols;
      BiasGradSeg& g = s.bp.seg[0];
      g.col_begin = 0; g.col_end = ncols; g.out = nullptr; g.n_valid = n_valid;
      s.seg_out[0].kind = RK_GRADS; s.seg_out[0].off = P.param_off[2 * c + 1] * 4;
      s.bp.nseg = 1;
      P.bwd.push_back(s);
    };
    bias_grad(9, DYP, 16, CO);
    bias_grad(0, G0, 64, 64);
    wgrad_conv(9, A5, 64, 64, DYP, 16, 64, 64);
    wgrad_conv(8, A4, 64, 64, G5, 64, 64, 64);
    wgrad_conv(7, S3, 64, 64, G4, 64, 64, 64);
    wgrad_conv(6, B3, 128, 128, G3, 64, 64, 128);
    wgrad_conv(5, B2, 256, 256, GA2, 128, 128, 256);
    wgrad_conv(4, B1, 512, 512, GA1, 256, 256, 512);
    wgrad_conv(3, T2u, 1024, 1024, GT3, 512, 512, 1024);
    wgrad_conv(2, T1u, 512, 512, GT2, 256, 256, 512);
    wgrad_conv(1, T0u, 256, 256, GT1, 128, 128, 256);
    wgrad_conv(0, P.o_xin, 64, 64, G0, 64, 64, CI);   // rows >= CI of the [hi | lo | hi] input are not flushed
    { Step s; s.type = ST_DISC_UNPACK; s.needs_wgrad = true; P.bwd.push_back(s); }
  }
  const long long bias_base = align_up(P.total_rows * 128, 1024);
  P.packed_bytes = bias_base + P.bias_floats * 4;
  auto fix = [&](std::vector<Step>& vv) {
    for (Step& s : vv) {
      if (s.bias.kind == RK_PACKED) s.bias.off = bias_base + (-1 - s.bias.off) * 4;
      // 16-bit format of every tensor of this plan: fp16 (the reference's autocast format) or bf16
      s.cp.epi.f16 = P.dd.fp16 ? 1 : 0;
      s.cp.mma_f16 = P.dd.fp16 ? 1 : 0;
      s.wb.a_f16 = s.wb.b_f16 = P.dd.fp16 ? 1 : 0;
      s.bp.f16 = P.dd.fp16 ? 1 : 0;
    }
  };
  fix(P.fwd); fix(P.bwd);
  for (PackOp& op : P.pack_ops) op.f16 = P.dd.fp16 ? 1 : 0;
  auto chainify = [&](std::vector<Step>& vv) {
    std::vector<Step> out;
    for (Step& s : vv) {
      if (s.type != ST_CONV) { out.push_back(s); continue; }
      if (out.empty() || out.back().type != ST_CHAIN || out.back().needs_dx != s.needs_dx) {
        Step c; c.type = ST_CHAIN; c.layer0 = (int)P.layer_steps.size(); c.nlayers = 0; c.chain_grid = 0; c.needs_dx = s.needs_dx;
        out.push_back(c);
      }
      out.back().nlayers++;
      const int work = s.cp.num_tiles * s.cp.col_groups;
      if (work > out.back().chain_grid) out.back().chain_grid = work;
      P.layer_steps.push_back(s);
    }
    vv.swap(out);
  };
  chainify(P.fwd); chainify(P.bwd);
  if (P.det && train) {
    const int sms = device_sms();
    if (sms > 0) P.plan_sms = sms;
    plan_deterministic(P, 2, P.plan_sms);  // run_steps: two weight-gradient streams on all SMs
  }
  return 0;
}

// =================================================================================================== C ABI =====
extern "C" {

const char* b200sr_last_error(void) { return g_err; }
int b200sr_version(void) { return 103; }
void b200sr_debug_set(int flags) { g_debug = flags; }
int b200sr_debug_read_profile(unsigned long long* out_host, int n) {
  CUDA_TRY(cudaMemcpyFromSymbol(out_host, g_conv_prof, sizeof(unsigned long long) * (size_t)n));
  return 0;
}
int b200sr_debug_buffer(const b200sr_plan* p, const char* name, int64_t* offset_bytes, int64_t* bytes) {
  if (!p || !name || !offset_bytes || !bytes) return fail(B200SR_ERR_INVALID, "null argument");
  for (const b200sr_plan::NamedBuf& nb : p->named_bufs) {
    if (nb.name == name) { *offset_bytes = nb.off; *bytes = nb.bytes; return 0; }
  }
  return fail(B200SR_ERR_INVALID, "the plan has no workspace tensor named '%s'", name);
}

static int net_plan_create(const b200sr_net_desc* desc, bool trunk, bool unclamped, b200sr_plan** out) {
  if (!desc || !out) return fail(B200SR_ERR_INVALID, "null argument");
  b200sr_plan* p = new b200sr_plan();
  p->d = *desc;
  p->trunk = trunk;
  p->unclamped = unclamped;
  p->det = desc->deterministic != 0;
  if (const char* e = getenv("B200SR_REASSOC")) p->reassoc = atoi(e) != 0;  // 0: per-conv schedule everywhere
  p->tail_f16 = desc->training == 0;  // training: the L1 loss' sign(sr - gt) amplifies the fp16 rounding of the tail past the 1e-2 gradient bar
  if (const char* e = getenv("B200SR_TAIL_FP16")) p->tail_f16 = atoi(e) != 0;  // 0: split-precision bf16 tail everywhere, 1: fp16 tail everywhere
  int rc = build_plan(*p);
  if (rc) { delete p; return rc; }
  *out = p;
  return 0;
}

int b200sr_plan_create(const b200sr_net_desc* desc, b200sr_plan** out) { return net_plan_create(desc, false, false, out); }
int b200sr_unclamped_plan_create(const b200sr_net_desc* desc, b200sr_plan** out) { return net_plan_create(desc, false, true, out); }
int b200sr_trunk_plan_create(const b200sr_net_desc* desc, b200sr_plan** out) { return net_plan_create(desc, true, false, out); }

void b200sr_plan_destroy(b200sr_plan* p) {
  if (!p) return;
  if (p->d_pack_ops) cudaFree(p->d_pack_ops);
  if (p->d_bias_ops) cudaFree(p->d_bias_ops);
  if (p->d_params) cudaFree((void*)p->d_params);
  if (p->d_unpack_ops) cudaFree(p->d_unpack_ops);
  for (int i = 0; i < b200sr_plan::kMapSlots; ++i) if (p->slots[i].d_layers) cudaFree(p->slots[i].d_layers);
  if (p->d_entries) cudaFree(p->d_entries);
  for (int k = 0; k < 3; ++k) {
    if (p->side_stream[k]) cudaStreamDestroy(p->side_stream[k]);
    if (p->ev_join[k]) cudaEventDestroy(p->ev_join[k]);
  }
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->d_layer_rec) cudaFree(p->d_layer_rec);
  if (p->d_entry_rec) cudaFree(p->d_entry_rec);
  if (p->d_counters) cudaFree(p->d_counters);
  delete p;
}

size_t b200sr_workspace_bytes(const b200sr_plan* p) { return p ? (size_t)p->ws_bytes : 0; }
size_t b200sr_packed_bytes(const b200sr_plan* p) { return p ? (size_t)p->packed_bytes : 0; }
uint64_t b200sr_pack_layout_id(const b200sr_plan* p) {
  // FNV-1a over the packing tables: two plans with equal ids produce byte-identical packed buffers from the same parameters
  if (!p) return 0;
  uint64_t h = 1469598103934665603ull;
  auto mix = [&](const void* data, size_t n) {
    const unsigned char* c = (const unsigned char*)data;
    for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; }
  };
  for (const PackOp& op : p->pack_ops) mix(&op, sizeof(op));
  for (const BiasOp& op : p->bias_ops) mix(&op, sizeof(op));
  mix(&p->total_rows, sizeof(p->total_rows));
  mix(&p->packed_bytes, sizeof(p->packed_bytes));
  return h ? h : 1;
}
int32_t b200sr_num_params(const b200sr_plan* p) { return p ? (int32_t)p->param_off.size() - 1 : 0; }
int64_t b200sr_param_numel(const b200sr_plan* p) { return p ? p->param_off.back() : 0; }

double b200sr_flops(const b200sr_plan* p, int backward) {
  if (!p) return 0;
  if (p->is_disc) {
    // 2 x MACs of the reference graph (BSRGAN/model.py:143-167).  backward = 1: the discriminator update (every weight gradient, every
    // data gradient but conv1's); backward = 2: the generator update (data gradients only, down to the input image)
    const b200sr_disc_desc& v = p->dd;
    const double cO[10] = {64, 128, 256, 512, 256, 128, 64, 64, 64, (double)v.out_channels};
    const double cI[10] = {(double)v.in_channels, 64, 128, 256, 512, 256, 128, 64, 64, 64};
    const int cK[10] = {3, 4, 4, 4, 3, 3, 3, 3, 3, 3}, lvl[10] = {0, 1, 2, 3, 2, 1, 0, 0, 0, 0};
    double total = 0;
    for (int c = 0; c < 10; ++c) {
      const double fl = 2.0 * cK[c] * cK[c] * cO[c] * cI[c] * v.batch * (v.height >> lvl[c]) * (v.width >> lvl[c]);
      if (!backward) total += fl;
      else if (backward == 1) total += fl * (c == 0 ? 1 : 2);
      else total += fl;
    }
    return total;
  }
  const int nconv = ((int)p->param_off.size() - 1) / 2;
  const int ntrunk = p->R * 5;
  double px = (double)p->d.batch * p->d.height * p->d.width, total = 0;
  for (int c = 0; c < nconv; ++c) {
    int O, I;
    conv_dims(*p, c, &O, &I);
    double res = 1;
    if (c > ntrunk + 1) {
      const int t = c - ntrunk - 1;
      res = (t <= p->L) ? (double)(1 << (2 * t)) : (double)(1 << (2 * p->L));
    }
    const double fl = 2.0 * 9 * O * I * res * px;
    total += backward ? fl * (c < p->t0 ? 1 : 2) : fl;  // (conv1 has no data gradient; every trunk conv has one)
  }
  return total;
}

// ordered-sum launches behind a step (deterministic plans: one per weight- or bias-gradient launch)
static int det_sums(const b200sr_plan& P, const Step& s) { return P.det && (s.type == ST_WGRAD || s.type == ST_BIASGRAD) ? 1 : 0; }

int32_t b200sr_num_launches(const b200sr_plan* p, int backward) {
  if (!p) return 0;
  const std::vector<Step>& v = backward ? p->bwd : p->fwd;
  // kernel launches of one pass.  backward = 1: no gradient-bucket callback, the per-bucket unpack steps collapse into one
  // launch; backward = 2: with a callback (data-parallel training), one unpack launch per bucket.
  int n = 0, unpacks = 0;
  for (const Step& s : v) {
    n += (s.type != ST_MEMSET && !s.needs_dx) + det_sums(*p, s);
    unpacks += (s.type == ST_UNPACK);
  }
  if (backward == 1 && unpacks > 1) n -= unpacks - 1;
  return n;
}

int b200sr_pack_weights(b200sr_plan* p, const float* const* params, void* packed, b200sr_stream stream) {
  if (!p || !params || !packed) return fail(B200SR_ERR_INVALID, "null argument");
  int rc = runtime_init();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int np = (int)p->param_off.size() - 1;
  if (!p->d_pack_ops) {
    CUDA_TRY(cudaMalloc(&p->d_pack_ops, p->pack_ops.size() * sizeof(PackOp)));
    CUDA_TRY(cudaMalloc(&p->d_bias_ops, p->bias_ops.size() * sizeof(BiasOp)));
    CUDA_TRY(cudaMalloc((void**)&p->d_params, np * sizeof(float*)));
    CUDA_TRY(cudaMemcpyAsync(p->d_pack_ops, p->pack_ops.data(), p->pack_ops.size() * sizeof(PackOp), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(p->d_bias_ops, p->bias_ops.data(), p->bias_ops.size() * sizeof(BiasOp), cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(cudaMemcpyAsync((void*)p->d_params, params, np * sizeof(float*), cudaMemcpyHostToDevice, st));
  const long long total = p->total_rows * 64;
  pack_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p->d_pack_ops, (int)p->pack_ops.size(), p->d_params,
                                                                      (__nv_bfloat16*)packed, p->total_rows);
  CUDA_TRY(cudaGetLastError());
  const long long bias_base = align_up(p->total_rows * 128, 1024);
  pack_bias_kernel<<<(unsigned)p->bias_ops.size(), 64, 0, st>>>(p->d_bias_ops, (int)p->bias_ops.size(), p->d_params,
                                                               (float*)((char*)packed + bias_base));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int b200sr_forward(b200sr_plan* p, const void* x, int x_dtype, const int64_t* x_strides, const void* packed, void* workspace,
                   float* y, b200sr_stream stream) {
  if (!p || !x || !x_strides || !packed || !workspace || !y) return fail(B200SR_ERR_INVALID, "null argument");
  int rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  Bases b{workspace, (void*)packed, y, nullptr, nullptr};
  return run_steps(*p, p->fwd, b, x, x_dtype, x_strides, nullptr, nullptr, (cudaStream_t)stream);
}

int b200sr_backward(b200sr_plan* p, const float* dy, const void* packed, void* workspace, float* flat_grads, float* dx_or_null,
                    b200sr_bucket_cb cb, void* user, b200sr_stream stream) {
  if (!flat_grads) return fail(B200SR_ERR_INVALID, "null argument");
  return b200sr_backward_select(p, dy, packed, workspace, flat_grads, dx_or_null, nullptr, cb, user, stream);
}

// mask_or_null / grads / dx as in b200sr_backward_select; *out: nullptr when everything is wanted (the full backward)
static int select_for(const b200sr_plan* p, const uint8_t* mask, bool grads, bool dx, GradSelect* g, const GradSelect** out) {
  const int nconv = ((int)p->param_off.size() - 1) / 2;
  if (!grads && mask)
    for (int c = 0; c < nconv; ++c)
      if (mask[c]) return fail(B200SR_ERR_INVALID, "conv %d is wanted but no gradient buffer was given", c);
  *out = nullptr;
  if (grads && !mask) return 0;
  if (p->is_vgg || p->is_disc) return fail(B200SR_ERR_INVALID, "a gradient selection needs a generator plan");
  *g = make_select(*p, mask, grads, dx);
  if (grads && std::all_of(g->want.begin(), g->want.end(), [](uint8_t w) { return w != 0; })) return 0;  // all ones = full backward
  *out = g;
  return 0;
}

int32_t b200sr_backward_launches(const b200sr_plan* p, const uint8_t* conv_wanted_or_null, int with_dx, int with_cb) {
  if (!p || !p->d.training || p->is_vgg || p->is_disc) return 0;
  GradSelect g;
  const GradSelect* sel = nullptr;
  select_for(p, conv_wanted_or_null, true, with_dx != 0, &g, &sel);  // cannot fail for a generator plan with a gradient buffer
  if (sel && !with_dx && !sel->any(0, (int)sel->want.size())) return 0;
  // counted as b200sr_num_launches counts: memsets are not launches, the unpack steps merge into one without a callback
  int n = 0;
  for (const Step& s : p->bwd) {
    if (s.type == ST_MEMSET) continue;
    if (s.needs_dx) { n += with_dx != 0; continue; }
    if (s.type == ST_CHAIN) { n += chain_layers(*p, s, sel) > 0; continue; }
    if (s.type == ST_UNPACK && !with_cb && s.i0 != 0) continue;
    n += step_selected(s, sel, true, with_dx != 0, with_cb != 0) * (1 + det_sums(*p, s));
  }
  return n;
}

int b200sr_backward_select(b200sr_plan* p, const float* dy, const void* packed, void* workspace, float* flat_grads_or_null,
                           float* dx_or_null, const uint8_t* conv_wanted_or_null, b200sr_bucket_cb cb, void* user,
                           b200sr_stream stream) {
  if (!p || !dy || !packed || !workspace) return fail(B200SR_ERR_INVALID, "null argument");
  if (!p->d.training) return fail(B200SR_ERR_INVALID, "plan was created with training=0");
  GradSelect g;
  const GradSelect* sel = nullptr;
  int rc = select_for(p, conv_wanted_or_null, flat_grads_or_null != nullptr, dx_or_null != nullptr, &g, &sel);
  if (rc) return rc;
  if (sel && !dx_or_null && !sel->any(0, (int)sel->want.size())) {  // nothing to compute: every wanted entry is zero
    if (flat_grads_or_null) CUDA_TRY(cudaMemsetAsync(flat_grads_or_null, 0, (size_t)p->param_off.back() * 4, (cudaStream_t)stream));
    return 0;
  }
  rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  if (!p->d_unpack_ops) {
    CUDA_TRY(cudaMalloc(&p->d_unpack_ops, p->unpack_ops.size() * sizeof(UnpackOp)));
    CUDA_TRY(cudaMemcpyAsync(p->d_unpack_ops, p->unpack_ops.data(), p->unpack_ops.size() * sizeof(UnpackOp), cudaMemcpyHostToDevice,
                             (cudaStream_t)stream));
  }
  Bases b{workspace, (void*)packed, dx_or_null, dy, flat_grads_or_null};
  return run_steps(*p, p->bwd, b, nullptr, 0, nullptr, cb, user, (cudaStream_t)stream, sel);
}

// ------------------------------------------------------------------------------------------ single-layer helpers
static int pick_ncols(int cout, int* n_cols, int* grid_y) {
  if (cout % 32 != 0 || cout < 32 || cout > 256) return fail(B200SR_ERR_INVALID, "cout must be a multiple of 32 in [32, 256] (got %d)", cout);
  *n_cols = (cout % 64 == 0) ? 64 : 32;
  *grid_y = cout / *n_cols;
  return 0;
}

size_t b200sr_conv3x3_scratch_bytes(int cin, int cout) {
  const long long chunks = (cin + 63) / 64;
  return (size_t)(align_up(chunks * 9 * cout * 128, 1024) + align_up(cout * 4, 1024) + 4096 + 1024);
}

static int single_conv(int mode, const void* x, int n, int h, int w, int cin, int x_stride, const float* wt, const float* bias, int cout, int act,
                       void* y, int y_stride, int y_coff, void* scratch, cudaStream_t st) {
  // mode kPackFwd: y[.., cout] = conv(x[.., cin]);  kPackDgrad: "cin" = channels of the incoming gradient (= conv Cout),
  // "cout" = channels of the produced input gradient (= conv Cin); wt is always the forward OIHW tensor.
  int rc = runtime_init();
  if (rc) return rc;
  int n_cols, grid_y;
  rc = pick_ncols(cout, &n_cols, &grid_y);
  if (rc) return rc;
  if (cin % 16 != 0) return fail(B200SR_ERR_INVALID, "cin must be a multiple of 16");
  const int chunks = (cin + 63) / 64;
  const long long rows = (long long)chunks * 9 * cout;
  char* sc = (char*)scratch;
  const long long bias_off = align_up(rows * 128, 1024);
  const long long tab_off = bias_off + align_up(cout * 4, 1024);
  PackOp op; memset(&op, 0, sizeof(op));
  op.row0 = 0; op.n_total = cout; op.n_cols = n_cols; op.n_valid = cout; op.num_chunks = chunks; op.mode = mode; op.nseg = 1;
  if (mode == kPackFwd) op.seg[0] = seg(0, cin, 0, cout, cin, 0, 0, 0);
  else                  op.seg[0] = seg(0, cin, 0, cin, cout, 0, 0, 0);
  BiasOp bo; bo.off = 0; bo.n = cout; bo.b_index = bias ? 1 : -1; bo.n_valid = cout; bo.rep = 0;
  const float* ptrs[2] = {wt, bias};
  CUDA_TRY(cudaMemcpyAsync(sc + tab_off, &op, sizeof(op), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(sc + tab_off + 1024, &bo, sizeof(bo), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(sc + tab_off + 2048, ptrs, sizeof(ptrs), cudaMemcpyHostToDevice, st));
  pack_weights_kernel<<<(unsigned)((rows * 64 + 255) / 256), 256, 0, st>>>((const PackOp*)(sc + tab_off), 1, (const float* const*)(sc + tab_off + 2048),
                                                                          (__nv_bfloat16*)sc, rows);
  CUDA_TRY(cudaGetLastError());
  pack_bias_kernel<<<1, 64, 0, st>>>((const BiasOp*)(sc + tab_off + 1024), 1, (const float* const*)(sc + tab_off + 2048), (float*)(sc + bias_off));
  CUDA_TRY(cudaGetLastError());
  CUtensorMap tmA;
  rc = encode_act_map(&tmA, (void*)x, cin, x_stride, n, h, w, kABoxRows);
  if (rc) return rc;
  LayerDesc L;
  L.tmA = tmA;
  L.p = base_conv_params(n, h, w, chunks, (cin - 64 * (chunks - 1)) / 16, 0, 1 << 20, 0, n_cols, cout);
  L.p.epi.act = act;
  L.p.epi.ob_stride = y_stride; L.p.epi.ob_coff = y_coff;
  L.p.epi.bias = (const float*)(sc + bias_off);
  L.p.epi.out_bf16 = (__nv_bfloat16*)y;
  const uint8_t* pw = (const uint8_t*)sc;
  CUDA_TRY(cudaMemcpyAsync(sc + tab_off + 3072, &L, sizeof(L), cudaMemcpyHostToDevice, st));
  EntryDesc ent; memset(&ent, 0, sizeof(ent));
  ent.layer = 0; ent.tile_lo = 0; ent.tile_hi = L.p.num_tiles; ent.dep = -1; ent.rot = 0;
  CUDA_TRY(cudaMemcpyAsync(sc + tab_off + 3072 + 512, &ent, sizeof(ent), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(sc + tab_off + 3072 + 640, 0, 64, st));
  const int work = L.p.num_tiles * L.p.col_groups;
  int grid = work < g_num_sms ? work : g_num_sms;
  const LayerDesc* layers = (const LayerDesc*)(sc + tab_off + 3072);
  const EntryDesc* entries = (const EntryDesc*)(sc + tab_off + 3072 + 512);
  int ne = 1, dbg = g_debug;
  unsigned int* ctr = (unsigned int*)(sc + tab_off + 3072 + 640);
  float* ydyn = nullptr;
  uint4 lrec[2], erec = make_entry_rec(ent);
  make_layer_rec(L.p, lrec, sc);
  CUDA_TRY(cudaMemcpyToSymbolAsync(c_layer_rec, lrec, sizeof(lrec), 0, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyToSymbolAsync(c_entry_rec, &erec, sizeof(erec), 0, cudaMemcpyHostToDevice, st));
  int layer0 = 0;
  void* args[] = {(void*)&layers, (void*)&entries, (void*)&ne, (void*)&pw, (void*)&ctr, (void*)&ydyn, (void*)&dbg, (void*)&layer0};
  const void* fn = dbg ? (const void*)conv3x3_chain_kernel<1, 0> : (const void*)conv3x3_chain_kernel<0, 0>;
  CUDA_TRY(cudaLaunchKernel(fn, dim3(grid), dim3(kConvThreads), args, (size_t)conv_smem_bytes(1), st));
  (void)grid_y;
  return 0;
}

int b200sr_conv3x3_fwd(const void* x, int n, int h, int w_, int cin, int x_stride, const float* w, const float* bias, int cout, int act,
                       void* y, int y_stride, int y_coff, void* scratch, b200sr_stream stream) {
  if (!x || !w || !y || !scratch) return fail(B200SR_ERR_INVALID, "null argument");
  return single_conv(kPackFwd, x, n, h, w_, cin, x_stride, w, bias, cout, act, y, y_stride, y_coff, scratch, (cudaStream_t)stream);
}

int b200sr_conv3x3_dgrad(const void* dy, int n, int h, int w_, int cout, int dy_stride, const float* w, int cin, void* dx, int dx_stride,
                         int dx_coff, void* scratch, b200sr_stream stream) {
  if (!dy || !w || !dx || !scratch) return fail(B200SR_ERR_INVALID, "null argument");
  return single_conv(kPackDgrad, dy, n, h, w_, cout, dy_stride, w, nullptr, cin, 0, dx, dx_stride, dx_coff, scratch, (cudaStream_t)stream);
}

size_t b200sr_conv3x3_wgrad_scratch_bytes(int cin, int cout) {
  return (size_t)(align_up(9LL * cin * align_up(cout, 4) * 4, 1024) + 1024);
}

int b200sr_conv3x3_wgrad(const void* x, int n, int h, int w_, int cin, int x_stride, const void* dy, int cout, int dy_stride, float* dw,
                         void* scratch, b200sr_stream stream) {
  if (!x || !dy || !dw || !scratch) return fail(B200SR_ERR_INVALID, "null argument");
  int rc = runtime_init();
  if (rc) return rc;
  if (cin > 128 || cout > 160 || cout % 16 != 0) return fail(B200SR_ERR_INVALID, "wgrad: cin <= 128, cout <= 160, cout %% 16 == 0");
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tmX, tmDY;
  rc = encode_act_map(&tmX, (void*)x, cin, x_stride, n, h, w_, kWgXRows);
  if (rc) return rc;
  rc = encode_act_map(&tmDY, (void*)dy, cout, dy_stride, n, h, w_, kWgTileH);
  if (rc) return rc;
  const long long stage_bytes = align_up(9LL * cin * cout * 4, 1024);
  float* staging = (float*)scratch;
  CUDA_TRY(cudaMemsetAsync(staging, 0, (size_t)stage_bytes, st));
  WgradBatch wb; memset(&wb, 0, sizeof(wb));
  wb.N = n; wb.H = h; wb.W = w_;
  wb.tiles_x = (w_ + kTileW - 1) / kTileW; wb.tiles_y = (h + kWgTileH - 1) / kWgTileH; wb.num_tiles = n * wb.tiles_x * wb.tiles_y;
  wb.num_problems = 1;
  WgradParams& wp = wb.prob[0];
  wp.b_c0 = 0; wp.n_cols = cout; wp.n_blocks = (cout + 63) / 64; wgrad_set_a(wp, 0, (cin > 64) ? 2 : 1);
  wp.num_seg = 1;
  wp.seg[0].col_begin = 0; wp.seg[0].col_end = cout; wp.seg[0].out = staging; wp.seg[0].ci_total = cin; wp.seg[0].ci0 = 0; wp.seg[0].co_pad = cout;
  int splits = g_num_sms / 3;
  if (splits > wb.num_tiles) splits = wb.num_tiles;
  wp.splits = splits;
  wb.cta_begin[0] = 0; wb.cta_begin[1] = splits * 3;
  wgrad3x3_kernel<false><<<dim3(splits * 3), kWgThreads, kWgSmemBytes, st>>>(tmX, tmDY, wb);
  CUDA_TRY(cudaGetLastError());
  UnpackOp u;
  u.src_off = 0; u.dst_off = 0; u.co = cout; u.ci = cin; u.co_pad = cout; u.fold = 0; u.block0 = 0;
  u.nblocks = ((cout + 31) / 32) * ((cin + 31) / 32);
  UnpackOp* d_u = (UnpackOp*)((char*)scratch + stage_bytes);
  CUDA_TRY(cudaMemcpyAsync(d_u, &u, sizeof(u), cudaMemcpyHostToDevice, st));
  unpack_wgrad_kernel<<<u.nblocks, 256, 0, st>>>(d_u, 0, 1, staging, dw);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------ fused optimizer
int b200sr_fused_adam_ema(const void* tensor_table, const int32_t* block_tensor, int n_tensors, int64_t total_blocks, float lr, float beta1,
                          float beta2, float eps, float weight_decay, float* step, float ema_decay, int ema_copy, const float* grad_scale,
                          const float* found_inf, b200sr_stream stream) {
  if (!tensor_table || !block_tensor || !step || n_tensors < 1 || total_blocks < 1) return fail(B200SR_ERR_INVALID, "bad argument");
  AdamEmaHyper h;
  h.lr = lr; h.beta1 = beta1; h.beta2 = beta2; h.eps = eps; h.weight_decay = weight_decay;
  h.ema_decay = ema_decay; h.ema_copy = ema_copy; h.grad_scale = grad_scale; h.found_inf = found_inf;
  h.step = step; h.block_tensor = block_tensor;
  fused_adam_ema_kernel<<<(unsigned)total_blocks, kOptBlock, 0, (cudaStream_t)stream>>>((const OptTensor*)tensor_table, n_tensors, h);
  CUDA_TRY(cudaGetLastError());
  adam_step_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step, found_inf);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------ evaluation epilogue
// blocks of the two IQA launches for an n x hc x wc cropped batch (fixed by the shape)
static long long iqa_psnr_blocks(int hc, int wc) { return std::min<long long>(((long long)hc * wc + 255) / 256, 1024); }
static dim3 iqa_ssim_grid(int n, int hc, int wc) { return dim3((unsigned)((wc - 10 + 15) / 16), (unsigned)((hc - 10 + 15) / 16), (unsigned)n); }

static int iqa_sums(const float* raw, const float* dst, int n, int h, int w, int crop_border, const double* window11,
                    double* psnr_sqerr_sum, double* ssim_map_sum, double* det_scratch, cudaStream_t st) {
  if (!raw || !dst || !window11 || (!psnr_sqerr_sum && !ssim_map_sum)) return fail(B200SR_ERR_INVALID, "null argument");
  if (n < 1 || crop_border < 0 || h - 2 * crop_border < 11 || w - 2 * crop_border < 11)
    return fail(B200SR_ERR_INVALID, "frame %dx%d with crop %d is smaller than the 11x11 SSIM window", h, w, crop_border);
  IqaParams p;
  p.raw = raw; p.dst = dst; p.N = n; p.H = h; p.W = w; p.crop = crop_border;
  for (int i = 0; i < 11; ++i) p.win[i] = window11[i];
  p.psnr_sum = psnr_sqerr_sum; p.ssim_sum = ssim_map_sum;
  const int hc = h - 2 * crop_border, wc = w - 2 * crop_border;
  const long long pblocks = iqa_psnr_blocks(hc, wc);
  const dim3 sgrid = iqa_ssim_grid(n, hc, wc);
  if (det_scratch) {
    // deterministic: [blocks][n] partial sums of each launch, then one ordered sum per metric
    SumJob<double> jobs[2];
    int nj = 0;
    double* part = det_scratch;
    if (psnr_sqerr_sum) {
      p.psnr_sum = part;
      iqa_psnr_y_kernel<true><<<dim3((unsigned)pblocks, (unsigned)n), 256, 0, st>>>(p);
      CUDA_TRY(cudaGetLastError());
      jobs[nj++] = sum_rows(psnr_sqerr_sum, part, (int)pblocks, n, n);
      part += pblocks * n;
    }
    if (ssim_map_sum) {
      p.ssim_sum = part;
      iqa_ssim_y_kernel<true><<<sgrid, dim3(16, 16), 0, st>>>(p);
      CUDA_TRY(cudaGetLastError());
      jobs[nj++] = sum_rows(ssim_map_sum, part, (int)(sgrid.x * sgrid.y), n, n);
    }
    return launch_ordered_sum(jobs, nj, st);
  }
  if (psnr_sqerr_sum) {
    CUDA_TRY(cudaMemsetAsync(psnr_sqerr_sum, 0, sizeof(double) * n, st));
    iqa_psnr_y_kernel<false><<<dim3((unsigned)pblocks, (unsigned)n), 256, 0, st>>>(p);
    CUDA_TRY(cudaGetLastError());
  }
  if (ssim_map_sum) {
    CUDA_TRY(cudaMemsetAsync(ssim_map_sum, 0, sizeof(double) * n, st));
    iqa_ssim_y_kernel<false><<<sgrid, dim3(16, 16), 0, st>>>(p);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

int b200sr_iqa_psnr_ssim_y(const float* raw, const float* dst, int n, int h, int w, int crop_border, const double* window11,
                           double* psnr_sqerr_sum, double* ssim_map_sum, b200sr_stream stream) {
  return iqa_sums(raw, dst, n, h, w, crop_border, window11, psnr_sqerr_sum, ssim_map_sum, nullptr, (cudaStream_t)stream);
}

size_t b200sr_iqa_det_scratch_bytes(int n, int h, int w) {
  if (n < 1 || h < 11 || w < 11) return 0;
  const dim3 g = iqa_ssim_grid(n, h, w);
  return sizeof(double) * (size_t)n * (size_t)(iqa_psnr_blocks(h, w) + (long long)g.x * g.y);
}

int b200sr_iqa_psnr_ssim_y_det(const float* raw, const float* dst, int n, int h, int w, int crop_border, const double* window11,
                               double* psnr_sqerr_sum, double* ssim_map_sum, double* scratch, b200sr_stream stream) {
  if (!scratch) return fail(B200SR_ERR_INVALID, "null argument");
  return iqa_sums(raw, dst, n, h, w, crop_border, window11, psnr_sqerr_sum, ssim_map_sum, scratch, (cudaStream_t)stream);
}

int b200sr_tensor_to_image_u8(const float* x, int c, int h, int w, int range_norm, int half, uint8_t* out_hwc, b200sr_stream stream) {
  if (!x || !out_hwc || c < 1 || c > 4 || h < 1 || w < 1) return fail(B200SR_ERR_INVALID, "bad argument");
  const long long plane = (long long)h * w;
  tensor_to_image_u8_kernel<<<(unsigned)((plane + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, c, h, w, range_norm, half, out_hwc);
  CUDA_TRY(cudaGetLastError());
  return 0;
}


// ------------------------------------------------------------------------------------------------ U-Net discriminator
int b200sr_disc_plan_create(const b200sr_disc_desc* desc, b200sr_plan** out) {
  if (!desc || !out) return fail(B200SR_ERR_INVALID, "null argument");
  b200sr_plan* p = new b200sr_plan();
  p->dd = *desc;
  p->det = desc->deterministic != 0;
  int rc = build_disc_plan(*p);
  if (rc) { delete p; return rc; }
  *out = p;
  return 0;
}

int b200sr_disc_forward(b200sr_plan* p, const void* x, int x_dtype, const int64_t* x_strides, const void* packed, void* workspace,
                        float* y, b200sr_stream stream) {
  if (!p || !p->is_disc || !x || !x_strides || !packed || !workspace || !y) return fail(B200SR_ERR_INVALID, "bad argument");
  int rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  Bases b{workspace, (void*)packed, y, nullptr, nullptr};
  return run_steps(*p, p->fwd, b, x, x_dtype, x_strides, nullptr, nullptr, (cudaStream_t)stream);
}

int b200sr_disc_backward(b200sr_plan* p, const float* dy, const void* packed, void* workspace, float* flat_grads_or_null,
                         float* dx_or_null, b200sr_stream stream) {
  if (!p || !p->is_disc || !dy || !packed || !workspace) return fail(B200SR_ERR_INVALID, "bad argument");
  if (!p->dd.training) return fail(B200SR_ERR_INVALID, "plan was created with training=0");
  int rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  if (!p->d_unpack_ops) {
    CUDA_TRY(cudaMalloc(&p->d_unpack_ops, p->unpack_ops.size() * sizeof(UnpackOp)));
    CUDA_TRY(cudaMemcpyAsync(p->d_unpack_ops, p->unpack_ops.data(), p->unpack_ops.size() * sizeof(UnpackOp), cudaMemcpyHostToDevice,
                             (cudaStream_t)stream));
  }
  Bases b{workspace, (void*)packed, dx_or_null, dy, flat_grads_or_null};
  return run_steps(*p, p->bwd, b, nullptr, 0, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ VGG19 features
int b200sr_vgg_plan_create(const b200sr_vgg_desc* desc, b200sr_plan** out) {
  if (!desc || !out) return fail(B200SR_ERR_INVALID, "null argument");
  b200sr_plan* p = new b200sr_plan();
  p->vd = *desc;
  p->det = desc->deterministic != 0;
  int rc = build_vgg_plan(*p);
  if (rc) { delete p; return rc; }
  *out = p;
  return 0;
}

int b200sr_vgg_forward(b200sr_plan* p, const float* x, const int64_t* x_strides, const void* packed, void* workspace, b200sr_stream stream) {
  if (!p || !p->is_vgg || !x || !x_strides || !packed || !workspace) return fail(B200SR_ERR_INVALID, "bad argument");
  int rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  Bases b{workspace, (void*)packed, nullptr, nullptr, nullptr};
  return run_steps(*p, p->fwd, b, x, B200SR_F32, x_strides, nullptr, nullptr, (cudaStream_t)stream);
}

int b200sr_vgg_feature_l1(b200sr_plan* p, const void* workspace, int conv_index, int pairs, double* out_sum, b200sr_stream stream) {
  if (!p || !p->is_vgg || !workspace || !out_sum) return fail(B200SR_ERR_INVALID, "bad argument");
  if (conv_index < 0 || conv_index > p->vd.last_conv || !p->o_vgg_feat[conv_index]) return fail(B200SR_ERR_INVALID, "conv %d has no feature buffer in this plan", conv_index);
  if (2 * pairs != p->vd.batch) return fail(B200SR_ERR_INVALID, "pairs must be half of the plan's batch");
  const long long half = (long long)pairs * p->vgg_h[conv_index] * p->vgg_w[conv_index] * kVggCout[conv_index];
  cudaStream_t st = (cudaStream_t)stream;
  long long blocks = (half / 4 + 255) / 256;
  if (blocks > kVggL1MaxBlocks) blocks = kVggL1MaxBlocks;
  const float* f = (const float*)((const char*)workspace + p->o_vgg_feat[conv_index] - 1);
  if (p->det) {
    double* partial = (double*)((char*)const_cast<void*>(workspace) + p->o_det);
    vgg_l1_pair_sum_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(f, half, partial);
    CUDA_TRY(cudaGetLastError());
    SumJob<double> j = sum_rows(out_sum, partial, (int)blocks, 1, 1);
    return launch_ordered_sum(&j, 1, st);
  }
  CUDA_TRY(cudaMemsetAsync(out_sum, 0, sizeof(double), st));
  vgg_l1_pair_sum_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(f, half, out_sum);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int b200sr_vgg_backward(b200sr_plan* p, const float* upstream, const void* packed, void* workspace, float* dx, b200sr_stream stream) {
  if (!p || !p->is_vgg || !upstream || !packed || !workspace || !dx) return fail(B200SR_ERR_INVALID, "bad argument");
  const int gc = p->vd.grad_conv, nb = p->vd.grad_images;
  if (gc < 0 || nb < 1 || 2 * nb != p->vd.batch || !p->o_vgg_feat[gc]) return fail(B200SR_ERR_INVALID, "plan was created without a gradient request");
  int rc = runtime_init();
  if (rc) return rc;
  rc = ensure_maps(*p, workspace, (void*)packed, (cudaStream_t)stream);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long half = (long long)nb * p->vgg_h[gc] * p->vgg_w[gc] * kVggCout[gc];
  const int post_relu = gc < p->vd.last_conv;  // the node's feature was stored after its ReLU (build_vgg_plan, mask_relu bit 1)
  vgg_l1_grad_kernel<<<(unsigned)((half / 4 + 255) / 256), 256, 0, st>>>((const float*)((char*)workspace + p->o_vgg_feat[gc] - 1), half, upstream,
                                                                         post_relu, (__nv_bfloat16*)((char*)workspace + p->o_vgg_g[gc] - 1));
  CUDA_TRY(cudaGetLastError());
  Bases b{workspace, (void*)packed, dx, nullptr, nullptr};
  return run_steps(*p, p->bwd, b, nullptr, 0, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
