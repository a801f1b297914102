// bf16 tensor-core ResNet path for sm_100a (tcgen05.mma, TMEM accumulators, TMA / bulk copies): the host-side plans
// and dispatch of the two whole-network kernels, the weight-packing kernels, and the conv_0 pre-pass of the packed
// strips.
//
//   resnet_tc_sweep_kernel  (resnet_sweep.cuh)   column sweep: the 128 MMA lanes are 128 rows of one map column
//   resnet_tc_fused_kernel  (resnet_fused.cuh)   position major: halo tiles of a planar-8 map
//
// Each runs conv_0 -> every C->C layer -> global mean -> Linear for a whole batch in one launch, in plain bf16 and in
// the split-bf16 ("bf16x3") mode.  Both precisions pick the kernel by one rule: the sweep plan if it can stage the
// map, else the position-major plan, else KWS_ERR_UNSUPPORTED.
#include "tc.cuh"
#include "ptx.cuh"
#include <cuda.h>
#include <cstdlib>
#include <cstring>
#include <tuple>
#include <vector>

namespace kws {

constexpr int kTcIssuers = 3;      // MMA-issuing warps (M-tiles dealt round-robin)
// warp 0 TMA, warps 1-3 MMA, then 4*NKC epilogue warps: warp e owns TMEM lane quarter (warp % 4) and the
// 16-channel group e / 4 (two planar-8 planes) of EVERY M-tile
__host__ __device__ constexpr int tc_epi_warps(int NKC) { return 4 * NKC; }
__host__ __device__ constexpr int tc_threads(int NKC) { return 32 * (1 + kTcIssuers + tc_epi_warps(NKC)); }
constexpr int kTcMaxMt = 8;       // upper bound of M-tiles per tile (tc_max_mt)
constexpr int kAccCols = 256;     // TMEM columns per accumulator buffer
constexpr int kMaxStages = 8;
// ---------------------------------------------------------------------------------------------
struct TcGeom {
  int H, W, d, dpad, Wp, R, tiles_per_utt;
  int Hpad;                            // rows per plane in memory (rows >= H are kept zero)
  int phase, chunks_per_phase;         // phase tiling: a tile = rows p, p+d, p+2d, ... (R of them) of phase p
  int rows_box, n_boxes, box_stride;   // bytes between row-block boxes inside a slab
  int h_start[3];                      // first input row of box bx relative to the tile's h0
  int tap_off[3];                      // byte offset inside a slab of tap row dh = -1, 0, +1
  int slab_bytes, stage_bytes, n_stages, side_taps;
  int smem_w_off, smem_ring_off, smem_total;
};

}  // namespace kws
#include "resnet_fused.cuh"
#include "resnet_sweep.cuh"
namespace kws {

// torch [C][C][3][3] fp32 -> [9][NKC][2][CP][8] bf16 (tap, 16-ch chunk, K half, cout, 8 cin)
// `in_scale` (nullable): BN scale 1/sigma of the PREVIOUS layer, folded into the input-channel axis
// (exact: the convolution is linear and zero padding stays zero; SURVEY appendix E).
// `out_lo` (nullable): the residual v - float(bf16(v)) in the same layout (the lo weight set of the split-bf16 mode).
__global__ void pack_conv3x3_tc_kernel(const float* __restrict__ w, const float* __restrict__ in_scale,
                                       __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo, int C, int NKC) {
  const int CP = 16 * NKC;
  const int total = 9 * NKC * 2 * CP * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i & 7;
    int t = i >> 3;
    const int co = t % CP; t /= CP;
    const int half = t & 1; t >>= 1;
    const int kc = t % NKC;
    const int tap = t / NKC;
    const int ci = kc * 16 + half * 8 + e;
    float v = (co < C && ci < C) ? w[((int64_t)co * C + ci) * 9 + tap] : 0.f;
    if (in_scale != nullptr && ci < C) v *= in_scale[ci];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[i] = hi;
    if (out_lo != nullptr) out_lo[i] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// torch [C][C][3][3] fp32 -> [NKC][3 dh][2 K halves][3 blocks][CP][8] bf16 for the column-sweep kernel
// (resnet_sweep.cuh): block k of a (16-channel chunk, height tap) slab holds the width tap dw = 2 - k, so that
// one N = 3*CP MMA on input column w feeds output columns w-d, w, w+d.  `in_scale` as above.
__global__ void pack_conv3x3_sw_kernel(const float* __restrict__ w, const float* __restrict__ in_scale,
                                       __nv_bfloat16* __restrict__ out, __nv_bfloat16* __restrict__ out_lo, int C, int NKC) {
  const int CP = 16 * NKC;
  const int total = NKC * 3 * 2 * 3 * CP * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i & 7;
    int t = i >> 3;
    const int co = t % CP; t /= CP;
    const int blk = t % 3; t /= 3;
    const int half = t & 1; t >>= 1;
    const int dh = t % 3;
    const int kc = t / 3;
    const int ci = kc * 16 + half * 8 + e;
    const int tap = dh * 3 + (2 - blk);
    float v = (co < C && ci < C) ? w[((int64_t)co * C + ci) * 9 + tap] : 0.f;
    if (in_scale != nullptr && ci < C) v *= in_scale[ci];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[i] = hi;
    if (out_lo != nullptr) out_lo[i] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// conv_0 weights [C][1][3][3] fp32 -> one-chunk sweep slab set [3 dh][2 K halves][3 blocks][CP][8] bf16: the staged
// "activation" of the conv_0 pseudo-layer carries the bf16 high and low parts of the feature in channels 0 and 1, so
// the weight sits in both positions (k = 0, 1 of K half 0) and everything else is zero.  split != 0 (bf16x3): channel 2
// carries the feature's high part again and k = 2 holds the weight's residual w - float(bf16(w)).
__global__ void pack_conv0_sw_kernel(const float* __restrict__ w0, __nv_bfloat16* __restrict__ out, int C, int CP, int split) {
  const int total = 3 * 2 * 3 * CP * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i & 7;
    int t = i >> 3;
    const int co = t % CP; t /= CP;
    const int blk = t % 3; t /= 3;
    const int half = t & 1; t >>= 1;
    const int dh = t;
    const int tap = dh * 3 + (2 - blk);
    const float w = (half == 0 && e < 3 && co < C) ? w0[co * 9 + tap] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(w);
    out[i] = e < 2 ? hi : (split && e == 2) ? __float2bfloat16_rn(w - __bfloat162float(hi)) : __float2bfloat16_rn(0.f);
  }
}

// Per-layer epilogue constants.  The activation stored by layer i is z_i = x_i - mean_i (the 1/sigma
// factor is folded into layer i+1's weights).  The skip tensor x_{i-2} of an even layer is not stored:
// it is z_{i-2} + mean_{i-2}, so z_i = ReLU(conv) + z_{i-2} + (mean_{i-2} - mean_i)   (resnet.py:49-55).
// `skip_mean` is nullptr for odd layers and for layer 2 (whose skip is the un-normalised conv_0 output).
__global__ void pad_bn_kernel(const float* __restrict__ scale, const float* __restrict__ mean,
                              const float* __restrict__ skip_mean, float* __restrict__ scale_p,
                              float* __restrict__ kconst_p, int C, int CP) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < CP) {
    scale_p[c] = c < C ? scale[c] : 0.f;
    kconst_p[c] = c < C ? (skip_mean != nullptr ? skip_mean[c] : 0.f) - mean[c] : 0.f;
  }
}

// rows [H, Hpad) of every plane are read by the phase-tiled TMA boxes and must be zero
__global__ void zero_pad_rows_kernel(uint4* __restrict__ buf, int64_t planes, int H, int Hpad, int W) {
  const int64_t per_plane = (int64_t)(Hpad - H) * W;
  const int64_t total = planes * per_plane;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pl = i / per_plane;
    buf[pl * (int64_t)Hpad * W + (int64_t)H * W + (i - pl * per_plane)] = make_uint4(0, 0, 0, 0);
  }
}

// ---------------------------------------------------------------------------------------------
// host side

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

struct TcResNet {
  kws_resnet_config cfg{};
  int NKC = 0, CP = 0, NP = 0;
  bool supported = false;
  int n_sms = 148;
  void* blob = nullptr;
  // per layer; every packed weight array is [hi set][lo set] (the lo set = residuals, read by the split-bf16 mode only)
  std::vector<__nv_bfloat16*> wpack;        // position-major layout
  std::vector<__nv_bfloat16*> wpack_sw;     // column-sweep layout (resnet_sweep.cuh)
  std::vector<float*> scale_p, shift_p;     // per layer, padded to CP: BN 1/sigma and the epilogue constant
  float* conv0_w = nullptr;                 // [C][9]
  __nv_bfloat16* conv0_wb = nullptr;        // conv_0 as a one-chunk sweep slab set (pack_conv0_sw_kernel)
  __nv_bfloat16* conv0_wb3 = nullptr;       // same for the split-bf16 mode
  float* out_w = nullptr;
  float* out_b = nullptr;
  // whole-network persistent kernel (resnet_fused.cuh): device copies of the layer table and tensor maps,
  // rebuilt when the input shape or the workspace changes
  void* fused_dev = nullptr;   // [TcLayerDesc x n_layers][pad][CUtensorMap x n_layers]
  std::tuple<int, int, const void*, int> fused_key{-1, -1, nullptr, 0};
  TcFusedParams fused_prm{};
  int fused_smem = 0;
  // column-sweep whole-network kernel (resnet_sweep.cuh), preferred when the map is tall enough
  // (HONK2_TC_SWEEP=0: the position-major kernel instead; the tests use it as the reference for sweep shapes)
  bool sweep_enabled = true;
};

static int tc_max_mt(int CP) {
  // M-tiles per tile, as many as the TMEM accumulator buffer holds (measured on B200: larger tiles win even though
  // 5 M-tiles do not divide evenly over 3 issuer warps)
  return std::min(kTcMaxMt, kAccCols / CP);
}

// Phase tiling pays when the dilation is large: a tile of R consecutive rows needs R + 2d (or 3R) input
// rows, a tile of R rows spaced d apart needs R + 2.
static bool tc_use_phase(int H, int d) { return d >= 8 && d <= 32 && 2 * d <= H; }

// Rows per plane in memory: H rounded up to the largest phase-tiled dilation of the network.
static int tc_hpad(const kws_resnet_config& c, int H) {
  int m = 1;
  for (int i = 1; i <= c.n_layers; ++i) {
    const int d = resnet_dilation(c, i);
    if (tc_use_phase(H, d)) m = std::max(m, d);
  }
  return round_up(H, m);
}

// Tile geometry of one layer of the position-major kernel.  Returns false if the layer cannot be tiled.
static bool tc_geom(int NKC, int H, int Hpad, int W, int d, TcGeom* g) {
  const int CP = 16 * NKC;
  g->H = H; g->W = W; g->d = d; g->Hpad = Hpad;
  g->side_taps = d < W ? 1 : 0;
  g->dpad = g->side_taps ? d : 0;
  g->Wp = W + g->dpad;
  if (g->Wp > 256) return false;
  const int max_pos = tc_max_mt(CP) * 128;
  const int w_bytes = 9 * NKC * 2 * CP * 16;
  g->smem_w_off = 256 + round_up(2 * CP * 4, 128);
  g->smem_ring_off = round_up(g->smem_w_off + w_bytes, 1024);
  const int budget = 227 * 1024 - g->smem_ring_off - 4096;
  g->phase = (tc_use_phase(H, d) && Hpad % d == 0) ? 1 : 0;
  g->chunks_per_phase = 1;
  if (g->phase) {
    // rows of one phase: p, p+d, ...; in phase-row units the convolution has dilation 1 in h
    const int rows_max = ceil_div(H, d);
    const int Rmax = std::min(rows_max, max_pos / g->Wp);
    if (Rmax < 1) return false;
    int best_R = 0, best_mt = 1 << 30;
    for (int R = Rmax; R >= 1; --R) {   // fewest issued M-tiles over all phases
      int mt = 0;
      for (int ph = 0; ph < d; ++ph) {
        const int n = ceil_div(H - ph, d);
        mt += (n / R) * ceil_div(R * g->Wp, 128) + ceil_div((n % R) * g->Wp, 128);
      }
      if (mt < best_mt) { best_mt = mt; best_R = R; }
    }
    const int R = best_R;
    g->R = R;
    g->chunks_per_phase = ceil_div(rows_max, R);
    g->tiles_per_utt = d * g->chunks_per_phase;
    g->n_boxes = 1;
    g->rows_box = R + 3;   // one halo row above and below + the spill row
    g->box_stride = round_up(g->rows_box * g->Wp * 16, 128);
    g->slab_bytes = g->box_stride;
    g->stage_bytes = 2 * g->slab_bytes;
    for (int k = 0; k < 3; ++k) {
      g->h_start[k] = -1;
      g->tap_off[k] = k * g->Wp * 16;
    }
    g->n_stages = std::min(kMaxStages, budget / g->stage_bytes);
    if (g->n_stages < 2) return false;
  } else {
    const int Rmax = std::min(H, max_pos / g->Wp);
    if (Rmax < 1) return false;
    // pick the rows-per-tile that issues the fewest 128-position M-tiles per utterance among those whose
    // staged input fits shared memory with >= 2 stages
    int best_R = 0, best_mt = 1 << 30, best_stages = 0;
    for (int R = Rmax; R >= 1; --R) {
      const int full = H / R, rem = H - full * R;
      const int mt = full * ceil_div(R * g->Wp, 128) + ceil_div(rem * g->Wp, 128);
      if (mt >= best_mt) continue;
      const bool dense = d <= R;
      const int rows_box = dense ? R + 2 * d + 1 : R + 1;
      if (rows_box > 256) continue;
      const int slab = (dense ? 1 : 3) * round_up(rows_box * g->Wp * 16, 128);
      if (slab >= (1 << 18)) continue;
      const int stages = std::min(kMaxStages, budget / (2 * slab));
      if (stages < 2) continue;
      best_R = R; best_mt = mt; best_stages = stages;
    }
    if (best_R == 0) return false;
    const int R = best_R;
    const bool dense = d <= R;
    g->R = R;
    g->tiles_per_utt = ceil_div(H, R);
    g->n_boxes = dense ? 1 : 3;
    g->rows_box = dense ? R + 2 * d + 1 : R + 1;
    g->box_stride = round_up(g->rows_box * g->Wp * 16, 128);
    g->slab_bytes = g->n_boxes * g->box_stride;
    g->stage_bytes = 2 * g->slab_bytes;
    for (int k = 0; k < 3; ++k) {
      g->h_start[k] = dense ? -d : (k - 1) * d;
      g->tap_off[k] = dense ? k * d * g->Wp * 16 : k * g->box_stride;
    }
    g->n_stages = best_stages;
  }
  g->smem_total = g->smem_ring_off + g->n_stages * g->stage_bytes + 4096;
  if (g->smem_total < 120 * 1024) g->smem_total = 120 * 1024;   // one CTA per SM (it owns all 512 TMEM columns)
  return true;
}

int tc_resnet_create(const kws_resnet_config& cfg, TcResNet** out) {
  TcResNet* p = new TcResNet();
  p->cfg = cfg;
  const int C = cfg.n_maps;
  p->NKC = ceil_div(C, 16);
  p->CP = 16 * p->NKC;
  p->NP = 2 * p->NKC;
  p->supported = p->NKC >= 1 && p->NKC <= 4 && get_encode_fn() != nullptr;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&p->n_sms, cudaDevAttrMultiProcessorCount, dev);
  if (p->supported) {
    const int n = cfg.n_layers;
    // one weight set is a multiple of 256 bytes (CP is a multiple of 16), so [hi set][lo set] is contiguous
    const size_t w_bytes = 2 * (size_t)9 * p->NKC * 2 * p->CP * 16;
    const size_t v_bytes = round_up<size_t>(p->CP * sizeof(float), 256);
    const size_t c0_bytes = round_up<size_t>((size_t)3 * 2 * 3 * p->CP * 16, 256);
    const size_t total = n * (2 * w_bytes + 2 * v_bytes) + 2 * c0_bytes + round_up<size_t>(C * 9 * 4, 256) +
                         round_up<size_t>((size_t)cfg.n_labels * C * 4, 256) + round_up<size_t>(cfg.n_labels * 4, 256);
    if (cudaMalloc(&p->blob, total) != cudaSuccess) {
      set_error("tc_resnet_create: cudaMalloc(%zu) failed", total);
      delete p;
      return KWS_ERR_CUDA;
    }
    char* b = static_cast<char*>(p->blob);
    for (int i = 0; i < n; ++i) {
      p->wpack.push_back(reinterpret_cast<__nv_bfloat16*>(b)); b += w_bytes;
      p->wpack_sw.push_back(reinterpret_cast<__nv_bfloat16*>(b)); b += w_bytes;
      p->scale_p.push_back(reinterpret_cast<float*>(b)); b += v_bytes;
      p->shift_p.push_back(reinterpret_cast<float*>(b)); b += v_bytes;
    }
    p->conv0_wb = reinterpret_cast<__nv_bfloat16*>(b); b += c0_bytes;
    p->conv0_wb3 = reinterpret_cast<__nv_bfloat16*>(b); b += c0_bytes;
    p->conv0_w = reinterpret_cast<float*>(b); b += round_up<size_t>(C * 9 * 4, 256);
    p->out_w = reinterpret_cast<float*>(b); b += round_up<size_t>((size_t)cfg.n_labels * C * 4, 256);
    p->out_b = reinterpret_cast<float*>(b);
    // read once per model handle (DESIGN.md section 4)
    const char* e = std::getenv("HONK2_TC_SWEEP");
    p->sweep_enabled = !e || std::atoi(e) != 0;
  }
  *out = p;
  return KWS_OK;
}

void tc_resnet_destroy(TcResNet* p) {
  if (!p) return;
  if (p->blob) cudaFree(p->blob);
  if (p->fused_dev) cudaFree(p->fused_dev);
  delete p;
}

int tc_resnet_set_weights(TcResNet* p, const kws_resnet_weights& w, float* const* bn_scale, float* const* bn_shift,
                          cudaStream_t st) {
  if (!p->supported) return KWS_OK;
  const int C = p->cfg.n_maps, n = p->cfg.n_layers, L = p->cfg.n_labels;
  for (int i = 0; i < n; ++i) {
    const int set_elems = 9 * p->NKC * 2 * p->CP * 8;   // one weight set; the lo set follows it
    pack_conv3x3_tc_kernel<<<ceil_div(set_elems, 256), 256, 0, st>>>(
        w.conv_w[i], i > 0 ? bn_scale[i - 1] : nullptr, p->wpack[i], p->wpack[i] + set_elems, C, p->NKC);
    KWS_CUDA(cudaGetLastError());
    pack_conv3x3_sw_kernel<<<ceil_div(set_elems, 256), 256, 0, st>>>(
        w.conv_w[i], i > 0 ? bn_scale[i - 1] : nullptr, p->wpack_sw[i], p->wpack_sw[i] + set_elems, C, p->NKC);
    KWS_CUDA(cudaGetLastError());
    // layer number i+1 is even and > 2  <=>  its skip comes from a normalised layer (i-1 in 0-based terms)
    const float* skip_mean = ((i + 1) % 2 == 0 && i >= 3) ? w.bn_mean[i - 2] : nullptr;
    pad_bn_kernel<<<1, 64, 0, st>>>(bn_scale[i], w.bn_mean[i], skip_mean, p->scale_p[i], p->shift_p[i], C, p->CP);
    KWS_CUDA(cudaGetLastError());
  }
  KWS_CUDA(cudaMemcpyAsync(p->conv0_w, w.conv0_w, sizeof(float) * C * 9, cudaMemcpyDeviceToDevice, st));
  pack_conv0_sw_kernel<<<ceil_div(3 * 2 * 3 * p->CP * 8, 256), 256, 0, st>>>(w.conv0_w, p->conv0_wb, C, p->CP, 0);
  KWS_CUDA(cudaGetLastError());
  pack_conv0_sw_kernel<<<ceil_div(3 * 2 * 3 * p->CP * 8, 256), 256, 0, st>>>(w.conv0_w, p->conv0_wb3, C, p->CP, 1);
  KWS_CUDA(cudaGetLastError());
  KWS_CUDA(cudaMemcpyAsync(p->out_w, w.out_w, sizeof(float) * L * C, cudaMemcpyDeviceToDevice, st));
  KWS_CUDA(cudaMemcpyAsync(p->out_b, w.out_b, sizeof(float) * L, cudaMemcpyDeviceToDevice, st));
  return KWS_OK;
}

static bool tc_layers_ok(const TcResNet* p, int H, int W) {
  TcGeom g;
  const int Hpad = tc_hpad(p->cfg, H);
  for (int i = 1; i <= p->cfg.n_layers; ++i) {
    const int d = resnet_dilation(p->cfg, i);
    if (!tc_geom(p->NKC, H, Hpad, W, d, &g)) return false;
  }
  return true;
}

// Input tensor map of one layer: dims 8 channels, W, rows (of one phase), phases, planes.  Plain tiling is the
// 1-phase case.
static int tc_encode_map(const void* base, int64_t planes, int H, int W, const TcGeom& g, CUtensorMap* out) {
  const cuuint64_t row_stride = (cuuint64_t)W * 16, plane_stride = (cuuint64_t)g.Hpad * W * 16;
  cuuint64_t dims[5], strides[4];
  dims[0] = 8; dims[1] = (cuuint64_t)W; dims[4] = (cuuint64_t)planes;
  strides[0] = 16; strides[3] = plane_stride;
  if (g.phase) {
    dims[2] = (cuuint64_t)(g.Hpad / g.d); dims[3] = (cuuint64_t)g.d;
    strides[1] = row_stride * g.d; strides[2] = row_stride;
  } else {
    dims[2] = (cuuint64_t)H; dims[3] = 1;
    strides[1] = row_stride; strides[2] = plane_stride;
  }
  const cuuint32_t box[5] = {8, (cuuint32_t)g.Wp, (cuuint32_t)g.rows_box, 1, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = get_encode_fn()(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for W=%d H=%d planes=%lld box=%dx%d phase=%d", (int)r, W, H,
              (long long)planes, g.Wp, g.rows_box, g.phase);
    return KWS_ERR_CUDA;
  }
  return KWS_OK;
}

// ---- whole-network persistent kernel: geometry, shared-memory plan, device tables ----------------
struct TcFusedPlan {
  bool ok = false, split = false;
  int Hpad = 0, n_slots = 0, smem_total = 0, n_stages = 0;
  int w_off[2] = {0, 0}, ring_off = 0, slot_bytes = 0;
  std::vector<TcGeom> geoms;
};

static TcFusedPlan tc_fused_plan(const TcResNet* p, int H, int W, bool split) {
  TcFusedPlan f;
  const kws_resnet_config& c = p->cfg;
  if (c.n_layers < 1 || c.n_layers > kFusedMaxLayers) return f;
  f.Hpad = tc_hpad(c, H);
  f.n_slots = p->n_sms;
  f.split = split;
  const int w_bytes = (split ? 2 : 1) * 9 * p->NKC * 2 * p->CP * 16;
  f.w_off[0] = 6144;   // control block: barriers, constants, layer descriptors, conv_0 weights, pooled sums
  f.w_off[1] = split ? f.w_off[0] : f.w_off[0] + round_up(w_bytes, 128);   // (split: one buffer for both weight sets)
  f.ring_off = round_up(f.w_off[1] + w_bytes, 1024);
  for (int i = 1; i <= c.n_layers; ++i) {
    TcGeom g;
    const int d = resnet_dilation(c, i);
    // (tc_geom picks the tile rows against a budget of one resident weight set; this kernel's ring is sized below)
    if (!tc_geom(p->NKC, H, f.Hpad, W, d, &g)) return f;
    f.slot_bytes = std::max(f.slot_bytes, round_up(g.stage_bytes, 128));
    f.geoms.push_back(g);
  }
  // as many ring slots as fit (large dilations stage three row-blocks per tile: fewer, larger slots)
  f.n_stages = std::min(kFusedStages, (227 * 1024 - 4096 - f.ring_off) / std::max(f.slot_bytes, 1));
  f.smem_total = f.ring_off + f.n_stages * f.slot_bytes + 4096;
  f.ok = f.n_stages >= 2;
  return f;
}

static size_t tc_fused_ws_bytes(const TcResNet* p, const TcFusedPlan& f, int W, size_t* buf_out) {
  const size_t buf = round_up<size_t>((size_t)f.n_slots * (f.split ? 2 : 1) * p->NP * f.Hpad * W * 16, 1024);
  if (buf_out) *buf_out = buf;
  return 2 * buf;
}

template <int NKC, bool SPLIT>
static int tc_launch_fused_v(const TcFusedParams& prm, int grid, int smem, cudaStream_t st) {
  KWS_CUDA(cudaFuncSetAttribute(resnet_tc_fused_kernel<NKC, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  resnet_tc_fused_kernel<NKC, SPLIT><<<grid, tc_threads(NKC), smem, st>>>(prm);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}
template <int NKC>
static int tc_launch_fused(const TcFusedParams& prm, bool split, int grid, int smem, cudaStream_t st) {
  return split ? tc_launch_fused_v<NKC, true>(prm, grid, smem, st) : tc_launch_fused_v<NKC, false>(prm, grid, smem, st);
}

static int tc_fused_forward(TcResNet* p, const TcFusedPlan& f, const float* feat, int64_t B, int T, int F, int H, int W,
                            float* logits, void* ws, LaunchProfiler* prof, cudaStream_t st) {
  const kws_resnet_config& c = p->cfg;
  size_t buf = 0;
  tc_fused_ws_bytes(p, f, W, &buf);
  __nv_bfloat16* P = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws));
  __nv_bfloat16* Q = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws) + buf);
  const auto key = std::make_tuple(T, F, (const void*)ws, f.split ? 1 : 0);
  if (p->fused_key != key) {
    // (re)build the device tables: layer descriptors + one input tensor map per layer
    const int n = c.n_layers;
    const size_t maps_off = round_up<size_t>(sizeof(TcLayerDesc) * n, 64);
    const size_t total = maps_off + sizeof(CUtensorMap) * n;
    std::vector<unsigned char> host(total, 0);
    for (int i = 1; i <= n; ++i) {
      TcLayerDesc L{};
      L.g = f.geoms[i - 1];
      L.wpack = p->wpack[i - 1];
      L.kconst = p->shift_p[i - 1];
      L.has_skip = (i % 2 == 0) ? 1 : 0;
      L.in_buf = L.has_skip ? 1 : 0;
      L.last = (i == n) ? 1 : 0;
      memcpy(host.data() + sizeof(TcLayerDesc) * (i - 1), &L, sizeof(L));
      CUtensorMap m;
      KWS_TRY(tc_encode_map(L.in_buf ? Q : P, (int64_t)f.n_slots * (f.split ? 2 : 1) * p->NP, H, W, L.g, &m));
      memcpy(host.data() + maps_off + sizeof(CUtensorMap) * (i - 1), &m, sizeof(m));
    }
    if (p->fused_dev) { KWS_CUDA(cudaStreamSynchronize(st)); KWS_CUDA(cudaFree(p->fused_dev)); p->fused_dev = nullptr; }
    KWS_CUDA(cudaMalloc(&p->fused_dev, total));
    KWS_CUDA(cudaMemcpyAsync(p->fused_dev, host.data(), total, cudaMemcpyHostToDevice, st));
    KWS_CUDA(cudaStreamSynchronize(st));   // `host` goes out of scope; this happens once per shape
    TcFusedParams& q = p->fused_prm;
    q = TcFusedParams{};
    q.layers = reinterpret_cast<const TcLayerDesc*>(p->fused_dev);
    q.maps = reinterpret_cast<const CUtensorMap*>(static_cast<char*>(p->fused_dev) + maps_off);
    q.conv0_w = p->conv0_w;
    q.last_scale = p->scale_p[n - 1];
    q.out_w = p->out_w;
    q.out_b = p->out_b;
    q.P = P; q.Q = Q;
    q.n_layers = n; q.C = c.n_maps; q.n_labels = c.n_labels; q.T = T; q.F = F;
    const auto [ph, pw] = resnet_pool(c);
    q.ph = ph; q.pw = pw;
    q.H = H; q.W = W; q.Hpad = f.Hpad;
    q.smem_w_off[0] = f.w_off[0]; q.smem_w_off[1] = f.w_off[1];
    q.smem_ring_off = f.ring_off; q.ring_slot_bytes = f.slot_bytes; q.n_stages = f.n_stages;
    p->fused_smem = f.smem_total;
    p->fused_key = key;
  }
  if (prof) prof->tick(1, st);
  if (f.Hpad > H) {
    for (__nv_bfloat16* bp : {P, Q}) {
      zero_pad_rows_kernel<<<256, 256, 0, st>>>(reinterpret_cast<uint4*>(bp), (int64_t)f.n_slots * (f.split ? 2 : 1) * p->NP, H, f.Hpad, W);
      KWS_CHECK_LAUNCH();
    }
  }
  if (prof) prof->tick(0, st);   // the whole network is one launch: it IS the dominant kernel
  TcFusedParams prm = p->fused_prm;
  prm.feat = feat;
  prm.logits = logits;
  prm.B = B;
  const int grid = (int)std::min<int64_t>(f.n_slots, B);
  static const bool dbg_on = [] { const char* e = std::getenv("HONK2_TC_DEBUG"); return e && std::atoi(e) != 0; }();
  static long long* dbg_buf = nullptr;
  if (dbg_on) {
    if (!dbg_buf) cudaMalloc(&dbg_buf, 16 * sizeof(long long));
    prm.debug = dbg_buf;
  }
  struct DbgPrint {
    long long* buf; cudaStream_t st;
    ~DbgPrint() {
      if (!buf) return;
      long long h[16];
      cudaStreamSynchronize(st);
      cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
      const double tot = (double)(h[0] + h[1] + h[2] + h[3] + h[4] + h[5]);
      fprintf(stderr, "[fused dbg] issuer 0 of CTA 0, %lld utterances, cycles: conv_0 wait %.1f%%, layer barrier (drain) %.1f%%, "
              "accumulator-free wait %.1f%%, TMA-data wait %.1f%%, issuing MMAs %.1f%% (total %.0f, %.0f per utterance)\n",
              h[6], 100 * h[0] / tot, 100 * h[1] / tot, 100 * h[2] / tot, 100 * h[3] / tot, 100 * h[4] / tot, tot, tot / (double)h[6]);
    }
  } dbg_print{dbg_on ? dbg_buf : nullptr, st};
  switch (p->NKC) {
    case 1: return tc_launch_fused<1>(prm, f.split, grid, p->fused_smem, st);
    case 2: return tc_launch_fused<2>(prm, f.split, grid, p->fused_smem, st);
    case 3: return tc_launch_fused<3>(prm, f.split, grid, p->fused_smem, st);
    default: return tc_launch_fused<4>(prm, f.split, grid, p->fused_smem, st);
  }
}

// ---- column-sweep whole-network kernel (resnet_sweep.cuh): plan, launch ------------------------------
struct TcSweepPlan {
  bool ok = false;
  int n_slots = 0, n_strips = 0, smem_total = 0, n_stages = 0;
  int c0w_off = 0, w_off[2] = {0, 0}, skip_off = 0, ring_off = 0, slot_bytes = 0, slack_bytes = 0;
  int dmax = 1, chunk_rows = 0;
  bool k32 = false, split = false;
  // packed strips (short maps): pack_n utterances stacked in one strip of Hst rows, conv_0 (+ pool) by the pre-pass kernel
  int pack_n = 1, pack_pitch = 0, Hst = 0, pool_off = 0;
  bool packed = false;
};

// (PH, PW) pooling windows the pre-pass kernel of the packed-strip mode is instantiated for
static bool tc_pack_pool_ok(int ph, int pw) { return (ph == 1 && pw == 1) || (ph == 2 && pw == 2) || (ph == 4 && pw == 3); }

// An unpooled map that fills less than this share (%) of its 128-row strips is packed; a single packed map that still
// fills less than it stays on the position-major kernel.
constexpr int kSwMinStripPct = 60;

static TcSweepPlan tc_sweep_plan(const TcResNet* p, int H, int W, bool split) {
  TcSweepPlan f;
  const int H_map = H;
  (void)H_map;
  const kws_resnet_config& c = p->cfg;
  // (no label bound: both kernels' tails loop over every label kws_resnet_create accepts, 1..1024)
  if (!p->sweep_enabled || c.n_layers < 1 || c.n_layers > kFusedMaxLayers) return f;
  if (W < 1 || W > kSwMaxW || H < 1) return f;
  if (p->NKC > 3) return f;   // 64 maps: 640 threads leave 96 registers, the epilogue spills (position-major kernel instead)
  if ((1 + c.n_layers) * p->CP * 4 > kSwKcBytes) return f;   // per-layer epilogue constants live in shared memory
  int dmax = 1;
  for (int i = 1; i <= c.n_layers; ++i) {
    const int d = resnet_dilation(c, i);
    if (d > 64) return f;   // (a staged column of 128 + 2d rows per plane would no longer leave room for three stages)
    dmax = std::max(dmax, d);
  }
  const auto [ph, pw] = resnet_pool(c);
  const bool pooled = ph > 1 || pw > 1;
  // The 128 lanes of an MMA are 128 rows of one column.  Short maps (res8 / res26 after pooling, short clips) are
  // PACKED: several utterances share a strip, stacked along the rows with dmax zero rows between them, and conv_0
  // (+ ReLU + AvgPool) is computed by a CUDA-core pre-pass (the sweep's own conv_0 pseudo-layer works on the unpooled map).
  const bool is_short = H * 100 < ceil_div(H, 128) * 128 * kSwMinStripPct;
  if (pooled || is_short) {
    const int pitch = H + dmax;
    const int n = (128 + dmax) / pitch;
    if (n < 1 || !tc_pack_pool_ok(ph, pw)) return f;
    f.packed = true;
    f.pack_n = n;
    f.pack_pitch = pitch;
    f.Hst = n * pitch - dmax;
    if (f.Hst * 100 < 128 * kSwMinStripPct && n == 1) return f;   // a single short map gains nothing here
  }
  if (f.packed) H = f.Hst;   // from here on the "map" is the stack
  f.n_strips = ceil_div(H, 128);
  f.n_slots = p->n_sms;
  f.dmax = dmax;
  f.split = split;
  // single-strip maps: 16 channels per row, [w][K chunk][h][32 B] in HBM, swizzle-32B operand in shared memory, one bulk
  // copy per step; taller maps: the planar layout
  f.k32 = f.n_strips == 1;
  if (split && !f.k32) return f;   // the split-bf16 mode is built on the 32-byte-row layout
  const int set_bytes = 9 * p->NKC * 2 * p->CP * 16;           // one weight set
  const int w_bytes = (split ? 2 : 1) * set_bytes;
  f.c0w_off = kSwCtrlBytes;
  f.w_off[0] = f.c0w_off + round_up(3 * 2 * 3 * p->CP * 16, 128);
  f.w_off[1] = split ? f.w_off[0] : f.w_off[0] + round_up(w_bytes, 128);   // (split: one buffer, see the kernel)
  f.skip_off = round_up(f.w_off[1] + w_bytes, 1024);
  // one skip slot per epilogue warp group: a planar strip column, [NP][128 rows][16 B], or a k32 column, NKC x H rows x 32 B
  f.pool_off = f.skip_off + (split ? 0 : sw_groups(p->NKC) * p->NP * 2048);
  f.ring_off = f.pool_off + (f.packed ? round_up(f.pack_n * sw_epi_warps(p->NKC) * p->CP * 4, 1024) : 0);   // packed: pooled sums per stacked utterance
  if (f.k32) {
    // a stage is [dmax guard rows][NA chunks x H rows][to a multiple of 8 rows: stages stay 256-byte aligned, the phase
    // of the 32-byte swizzle].  The MMA of chunk kc, tap dh reads 128 rows from dmax + kc H + (dh - 1) d: the last
    // chunk's lanes past the map read up to dmax + (NA - 1) H + dmax + 128 rows, into the next stage or, behind the
    // last stage, into the slack.
    const int na = (split ? 2 : 1) * p->NKC;
    const int slot_rows = round_up(dmax + na * H, 8);
    f.chunk_rows = H;
    f.slot_bytes = slot_rows * 32;
    f.slack_bytes = round_up(std::max(0, dmax + (na - 1) * H + dmax + 128 - slot_rows), 8) * 32;
  } else {
    // planar: dmax zero rows above and below the strip's 128 rows, in every plane
    f.chunk_rows = (128 + 2 * dmax + 7) & ~7;
    f.slot_bytes = p->NP * f.chunk_rows * 16;
    f.slack_bytes = 0;
  }
  f.n_stages = std::min(kSwMaxStages, (227 * 1024 - f.slack_bytes - f.ring_off) / f.slot_bytes);
  if (f.n_stages < 3) return f;
  f.smem_total = f.ring_off + f.n_stages * f.slot_bytes + f.slack_bytes;
  f.ok = true;
  return f;
}

// packed strips: utterances per pre-pass + sweep launch pair (a multiple of the group size)
static int64_t tc_pack_chunk(const TcSweepPlan& f, int64_t B, int chunk_cfg) {
  int64_t c = chunk_cfg > 0 ? chunk_cfg : 4096;
  c = round_up<int64_t>(c, f.pack_n);
  return std::min<int64_t>(c, round_up<int64_t>(std::max<int64_t>(B, 1), f.pack_n));
}

static size_t tc_sweep_ws_bytes(const TcResNet* p, const TcSweepPlan& f, int H, int W, int64_t B, int chunk_cfg,
                                size_t* buf_out, size_t* ext_group_out = nullptr) {
  const int Hs = f.packed ? f.Hst : H;
  const size_t buf = round_up<size_t>((size_t)f.n_slots * (f.split ? 2 : 1) * p->NP * Hs * W * 16, 1024);
  if (buf_out) *buf_out = buf;
  size_t ext = 0;
  if (f.packed) {
    const size_t per_group = (size_t)(f.split ? 2 : 1) * p->NP * Hs * W * 16;
    if (ext_group_out) *ext_group_out = per_group;
    ext = round_up<size_t>((size_t)(tc_pack_chunk(f, B, chunk_cfg) / f.pack_n) * per_group, 1024);
  }
  return 2 * buf + ext;
}

// conv_0 (1 -> C, 3x3, pad 1) + ReLU + AvgPool(PH, PW) (resnet.py:40-44) for the packed-strip mode of the sweep kernel:
// writes the bf16 activations of a group of `pack_n` stacked utterances exactly as the sweep kernel's epilogue would
// ([w][K chunk][stacked row][16 ch = 32 B], halves of chunk kc swapped where ((dmax + kc Hst + row) >> 2) & 1, zero rows
// between the utterances; split: the lo parts in chunks NKC .. 2 NKC-1).  One thread = one (column, stacked row) position of a group;
// a group's W * Hst positions are dealt to blocks of 128 threads column by column (rows fastest: 32-byte stores coalesce).
template <int PH, int PW>
__global__ void __launch_bounds__(128)
conv0_pool_pack_kernel(const float* __restrict__ feat, const float* __restrict__ w0, uint4* __restrict__ ext, int64_t B_utt,
                       int T, int F, int C, int NKC, int W, int Hs, int pitch, int pack_n, int Hst, int dmax, int split,
                       int64_t ext_stride) {
  __shared__ __align__(16) float s_w[64 * 12];
  const int CP = 16 * NKC;
  for (int i = threadIdx.x; i < CP * 12; i += blockDim.x) {
    const int c = i / 12, k = i - c * 12;
    s_w[i] = (k < 9 && c < C) ? w0[c * 9 + k] : 0.f;
  }
  __syncthreads();
  const int tiles = (W * Hst + 127) >> 7;
  const int64_t g = blockIdx.x / tiles;
  const int item = (blockIdx.x - (int)(g * tiles)) * 128 + threadIdx.x;
  if (item >= W * Hst) return;
  const int wo = item / Hst, row = item - wo * Hst;
  const int u = row / pitch, ho = row - u * pitch;
  const int64_t b = g * pack_n + u;
  const bool live = ho < Hs && u < pack_n && b < B_utt;
  float patch[PH + 2][PW + 2];
#pragma unroll
  for (int a = 0; a < PH + 2; ++a)
#pragma unroll
    for (int e = 0; e < PW + 2; ++e) {
      const int hh = ho * PH - 1 + a, ww = wo * PW - 1 + e;
      patch[a][e] = (live && hh >= 0 && hh < T && ww >= 0 && ww < F) ? __ldg(feat + (b * T + hh) * (int64_t)F + ww) : 0.f;
    }
  constexpr float inv = 1.f / (float)(PH * PW);
  const int NA = split ? 2 * NKC : NKC;
  auto swl_of = [&](int kc) { return ((dmax + kc * Hst + row) >> 2) & 1; };
  // (a warp whose 32 items are all gap rows / past the batch only stores zeros; the pad channels C .. CP-1 are zeros too)
  const bool warp_live = __any_sync(0xffffffffu, live);
  for (int kc = 0; kc < NKC; ++kc) {
    float out[16];
#pragma unroll
    for (int cl = 0; cl < 16; ++cl) {
      if (!warp_live || 16 * kc + cl >= C) { out[cl] = 0.f; continue; }
      const float* wc = s_w + (16 * kc + cl) * 12;
      const float4 wa = *reinterpret_cast<const float4*>(wc);
      const float4 wb = *reinterpret_cast<const float4*>(wc + 4);
      const float w8 = wc[8];
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < PH; ++i)
#pragma unroll
        for (int j = 0; j < PW; ++j) {
          float v = patch[i][j] * wa.x;
          v = fmaf(patch[i][j + 1], wa.y, v); v = fmaf(patch[i][j + 2], wa.z, v);
          v = fmaf(patch[i + 1][j], wa.w, v); v = fmaf(patch[i + 1][j + 1], wb.x, v); v = fmaf(patch[i + 1][j + 2], wb.y, v);
          v = fmaf(patch[i + 2][j], wb.z, v); v = fmaf(patch[i + 2][j + 1], wb.w, v); v = fmaf(patch[i + 2][j + 2], w8, v);
          acc += fmaxf(v, 0.f);
        }
      out[cl] = live ? acc * inv : 0.f;
    }
    uint4 hi[2], lo[2];
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      __nv_bfloat162* hb = reinterpret_cast<__nv_bfloat162*>(&hi[hf]);
      __nv_bfloat162* lb = reinterpret_cast<__nv_bfloat162*>(&lo[hf]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float a = out[8 * hf + 2 * e], c2 = out[8 * hf + 2 * e + 1];
        hb[e] = __floats2bfloat162_rn(a, c2);
        const float2 fh = __bfloat1622float2(hb[e]);
        lb[e] = __floats2bfloat162_rn(a - fh.x, c2 - fh.y);
      }
    }
    uint4* dst = ext + g * ext_stride + ((int64_t)(wo * NA + kc) * Hst + row) * 2;
    const int swl = swl_of(kc);
    dst[swl] = hi[0];
    dst[swl ^ 1] = hi[1];
    if (split) {
      uint4* dl = ext + g * ext_stride + ((int64_t)(wo * NA + NKC + kc) * Hst + row) * 2;
      const int swl_lo = swl_of(NKC + kc);
      dl[swl_lo] = lo[0];
      dl[swl_lo ^ 1] = lo[1];
    }
  }
}

static int tc_launch_conv0_pack(int ph, int pw, const float* feat, const float* w0, uint4* ext, int64_t B_utt, int64_t groups,
                                int T, int F, int C, int NKC, int W, int Hs, const TcSweepPlan& f, int64_t ext_stride,
                                cudaStream_t st) {
  const int64_t blocks = groups * ceil_div(W * f.Hst, 128);
  KWS_REQUIRE(blocks < (int64_t)2147483647, "conv_0 pre-pass: batch too large for one launch");
#define KWS_C0P(PH, PW)                                                                                                  \
  conv0_pool_pack_kernel<PH, PW><<<(unsigned)blocks, 128, 0, st>>>(feat, w0, ext, B_utt, T, F, C, NKC, W, Hs, f.pack_pitch,    \
                                                                   f.pack_n, f.Hst, f.dmax, f.split ? 1 : 0, ext_stride)
  if (ph == 1 && pw == 1) KWS_C0P(1, 1);
  else if (ph == 2 && pw == 2) KWS_C0P(2, 2);
  else if (ph == 4 && pw == 3) KWS_C0P(4, 3);
  else { set_error("conv_0 pre-pass: pooling %dx%d is not instantiated", ph, pw); return KWS_ERR_UNSUPPORTED; }
#undef KWS_C0P
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

template <int NKC, bool DBG, bool K32, bool SPLIT, bool PACK>
static int tc_launch_sweep_v(const SwParams& prm, int grid, int smem, cudaStream_t st) {
  KWS_CUDA(cudaFuncSetAttribute(resnet_tc_sweep_kernel<NKC, DBG, K32, SPLIT, PACK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  resnet_tc_sweep_kernel<NKC, DBG, K32, SPLIT, PACK><<<grid, sw_threads(NKC), smem, st>>>(prm);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

template <int NKC>
static int tc_launch_sweep(const SwParams& prm, bool k32, bool split, int grid, int smem, cudaStream_t st) {
  if (prm.ext_in != nullptr)   // packed strips (always the 32-byte-row layout; no cycle-accounting build)
    return split ? tc_launch_sweep_v<NKC, false, true, true, true>(prm, grid, smem, st)
                 : tc_launch_sweep_v<NKC, false, true, false, true>(prm, grid, smem, st);
  if (split) return tc_launch_sweep_v<NKC, false, true, true, false>(prm, grid, smem, st);
  if (prm.debug != nullptr)
    return k32 ? tc_launch_sweep_v<NKC, true, true, false, false>(prm, grid, smem, st) : tc_launch_sweep_v<NKC, true, false, false, false>(prm, grid, smem, st);
  return k32 ? tc_launch_sweep_v<NKC, false, true, false, false>(prm, grid, smem, st) : tc_launch_sweep_v<NKC, false, false, false, false>(prm, grid, smem, st);
}

static int tc_sweep_launch(TcResNet* p, const TcSweepPlan& f, const float* feat, int64_t B, int64_t B_utt, int T, int F, int H,
                           int W, float* logits, void* ws, size_t buf, const uint4* ext, int64_t ext_stride, int sub_h,
                           LaunchProfiler* prof, cudaStream_t st);

static int tc_sweep_forward(TcResNet* p, const TcSweepPlan& f, const float* feat, int64_t B, int T, int F, int H, int W,
                            float* logits, void* ws, int chunk_cfg, LaunchProfiler* prof, cudaStream_t st) {
  const kws_resnet_config& c = p->cfg;
  size_t buf = 0, ext_group = 0;
  tc_sweep_ws_bytes(p, f, H, W, B, chunk_cfg, &buf, &ext_group);
  const int n = c.n_layers;
  if (f.packed) {
    // packed strips: conv_0 + pool by the pre-pass kernel, then the sweep over groups of pack_n stacked utterances,
    // one launch pair per sub-batch.  The rows between stacked utterances are never stored: zero both buffers once.
    KWS_CUDA(cudaMemsetAsync(ws, 0, 2 * buf, st));
    const int64_t chunk = tc_pack_chunk(f, B, chunk_cfg);
    const auto [ph, pw] = resnet_pool(c);
    uint4* ext = reinterpret_cast<uint4*>(static_cast<char*>(ws) + 2 * buf);
    for (int64_t b0 = 0; b0 < B; b0 += chunk) {
      const int64_t nb = std::min(chunk, B - b0);
      const int64_t groups = ceil_div<int64_t>(nb, f.pack_n);
      if (prof) prof->tick(1, st);
      KWS_TRY(tc_launch_conv0_pack(ph, pw, feat + b0 * (int64_t)T * F, p->conv0_w, ext, nb, groups, T, F, c.n_maps, p->NKC, W,
                                   H, f, (int64_t)(ext_group / 16), st));
      KWS_TRY(tc_sweep_launch(p, f, nullptr, groups, nb, T, F, f.Hst, W, logits + b0 * c.n_labels, ws, buf, ext,
                              (int64_t)(ext_group / 16), H, prof, st));
    }
    return KWS_OK;
  }
  return tc_sweep_launch(p, f, feat, B, B, T, F, H, W, logits, ws, buf, nullptr, 0, H, prof, st);
}

// one launch of the sweep kernel: B units (utterances, or groups of stacked utterances when ext != nullptr)
static int tc_sweep_launch(TcResNet* p, const TcSweepPlan& f, const float* feat, int64_t B, int64_t B_utt, int T, int F, int H,
                           int W, float* logits, void* ws, size_t buf, const uint4* ext, int64_t ext_stride, int sub_h,
                           LaunchProfiler* prof, cudaStream_t st) {
  const kws_resnet_config& c = p->cfg;
  const int n = c.n_layers;
  // (no device-side tables: every per-layer quantity is derived from these parameters inside the kernel, so a change
  // of batch size, shape or workspace costs nothing)
  SwParams prm{};
  prm.wpack0 = reinterpret_cast<const unsigned char*>(p->wpack_sw[0]);
  prm.kconst0 = reinterpret_cast<const unsigned char*>(p->shift_p[0]);
  prm.layer_stride = n > 1 ? (int64_t)(reinterpret_cast<const unsigned char*>(p->wpack_sw[1]) - prm.wpack0) : 0;
  prm.use_dilation = c.use_dilation ? 1 : 0;
  prm.conv0_wb = reinterpret_cast<const unsigned char*>(f.split ? p->conv0_wb3 : p->conv0_wb);
  prm.last_scale = p->scale_p[n - 1];
  prm.out_w = p->out_w;
  prm.out_b = p->out_b;
  prm.P = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws));
  prm.Q = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws) + buf);
  prm.n_layers = n; prm.C = c.n_maps; prm.n_labels = c.n_labels; prm.T = T; prm.F = F;
  prm.H = H; prm.W = W; prm.n_strips = f.n_strips;
  prm.smem_c0w_off = f.c0w_off;
  prm.smem_skip_off = f.skip_off;
  prm.dmax = f.dmax;
  prm.chunk_rows = f.chunk_rows;
  prm.ring_slack_bytes = f.slack_bytes;
  prm.discard_q = f.n_strips == 1 && !f.split && !f.packed;   // (packed: the zero rows inside a column must survive)
  prm.ext_in = ext; prm.ext_stride = ext_stride;
  prm.pack_n = f.packed ? f.pack_n : 1; prm.pack_h = sub_h; prm.pack_pitch = f.packed ? f.pack_pitch : H;
  prm.smem_pool_off = f.pool_off;
  prm.B_utt = B_utt;
  prm.smem_w_off[0] = f.w_off[0]; prm.smem_w_off[1] = f.w_off[1];
  prm.smem_ring_off = f.ring_off; prm.ring_slot_bytes = f.slot_bytes; prm.n_stages = f.n_stages;
  prm.feat = feat;
  prm.logits = logits;
  prm.B = B;
  if (prof) prof->tick(0, st);   // the whole network is one launch: it IS the dominant kernel
  const int grid = (int)std::min<int64_t>(f.n_slots, B);
  static const bool dbg_on = [] { const char* e = std::getenv("HONK2_TC_DEBUG"); return e && std::atoi(e) != 0; }();
  static long long* dbg_buf = nullptr;
  if (dbg_on && !f.split && !f.packed) {
    if (!dbg_buf) cudaMalloc(&dbg_buf, 16 * sizeof(long long));
    prm.debug = dbg_buf;
  }
  static const bool trace_on = [] { const char* e = std::getenv("HONK2_TC_TRACE"); return e && std::atoi(e) != 0; }();
  static long long* trace_buf = nullptr;
  if (prm.debug != nullptr && trace_on) {
    if (!trace_buf) { cudaMalloc(&trace_buf, 8 * kSwTraceLen * sizeof(long long)); }
    cudaMemsetAsync(trace_buf, 0, 8 * kSwTraceLen * sizeof(long long), st);
    prm.trace = trace_buf;
  }
  struct DbgPrint {
    long long* buf; cudaStream_t st; long long* trace;
    ~DbgPrint() {
      if (!buf) return;
      long long h[16];
      cudaStreamSynchronize(st);
      cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
      if (trace) {   // event timestamps of CTA 0 -> HONK2_TC_TRACE_FILE (one row per event kind)
        std::vector<long long> t(8 * kSwTraceLen);
        cudaMemcpy(t.data(), trace, t.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        const char* fn = std::getenv("HONK2_TC_TRACE_FILE");
        if (FILE* f = fopen(fn ? fn : "sweep_trace.csv", "w")) {
          fprintf(f, "idx,producer_copy,issuer_start,issuer_after_tempty,issuer_after_full,issuer_after_issue,epi0_tfull,epi0_done,epi7_done\n");
          for (int i = 0; i < kSwTraceLen; ++i) {
            fprintf(f, "%d", i);
            for (int r = 0; r < 8; ++r) fprintf(f, ",%lld", t[(size_t)r * kSwTraceLen + i]);
            fprintf(f, "\n");
          }
          fclose(f);
        }
      }
      const double ptot = (double)(h[13] + h[14] + h[15] + h[7]);
      fprintf(stderr, "[sweep dbg] producer of CTA 0: waiting for the previous layer's column %.1f%%, for a free stage %.1f%%, building "
              "conv_0 columns %.1f%%, issuing copies / weights / bookkeeping %.1f%% (total %.0f)\n",
              100 * h[13] / ptot, 100 * h[14] / ptot, 100 * h[15] / ptot, 100 * h[7] / ptot, ptot);
      h[7] = 0;
      const double tot = (double)(h[0] + h[1] + h[2] + h[3] + h[5] + h[6] + h[7]);
      fprintf(stderr, "[sweep dbg] issuer 0 of CTA 0, %lld utterances, cycles: weights wait %.1f%%, accumulator-free wait %.1f%%, "
              "TMA-data wait %.1f%%, utterance boundary (tail + conv_0 + first load) %.1f%%, issuing own steps %.1f%%, first loop top after an own step %.1f%%, counting along %.1f%% "
              "(total %.0f, %.0f per utterance)\n",
              h[4], 100 * h[0] / tot, 100 * h[1] / tot, 100 * h[2] / tot, 100 * h[5] / tot, 100 * h[3] / tot, 100 * h[7] / tot, 100 * h[6] / tot, tot,
              tot / (double)std::max(1ll, h[4]));
      const double et = (double)(h[8] + h[9] + h[10] + h[11] + h[12]);
      fprintf(stderr, "[sweep dbg] epilogue warp 0 of CTA 0: waiting for accumulators %.1f%%, TMEM load + re-zero %.1f%%, publishing the "
              "previous column %.1f%%, math + stores (+ guard, tail) %.1f%%, conv_0 %.1f%% (total %.0f)\n",
              100 * h[8] / et, 100 * h[9] / et, 100 * h[10] / et, 100 * h[11] / et, 100 * h[12] / et, et);
    }
  } dbg_print{prm.debug, st, prm.trace};
  switch (p->NKC) {
    case 1: return tc_launch_sweep<1>(prm, f.k32, f.split, grid, f.smem_total, st);
    case 2: return tc_launch_sweep<2>(prm, f.k32, f.split, grid, f.smem_total, st);
    default: return tc_launch_sweep<3>(prm, f.k32, f.split, grid, f.smem_total, st);
  }
}

// One rule for both precisions: the column-sweep kernel if its plan can stage the map, else the position-major
// kernel, else unsupported (workspace 0).
size_t tc_resnet_workspace_bytes(const TcResNet* p, int64_t B, int T, int F, int chunk, bool split) {
  if (!p || !p->supported) return 0;
  int H, W;
  resnet_map(p->cfg, T, F, &H, &W);
  if (H < 1 || W < 1 || W > 256 || !tc_layers_ok(p, H, W)) return 0;
  const TcSweepPlan sp = tc_sweep_plan(p, H, W, split);
  if (sp.ok) return tc_sweep_ws_bytes(p, sp, H, W, B, chunk, nullptr);
  const TcFusedPlan f = tc_fused_plan(p, H, W, split);
  return f.ok ? tc_fused_ws_bytes(p, f, W, nullptr) : 0;
}

const char* tc_resnet_kernel_path(const TcResNet* p, int T, int F, bool split) {
  if (!p || !p->supported) return "unsupported";
  int H, W;
  resnet_map(p->cfg, T, F, &H, &W);
  if (H < 1 || W < 1 || W > 256 || !tc_layers_ok(p, H, W)) return "unsupported";
  if (tc_sweep_plan(p, H, W, split).ok) return "resnet_tc_sweep_kernel";
  if (tc_fused_plan(p, H, W, split).ok) return "resnet_tc_fused_kernel";
  return "unsupported";
}

int tc_resnet_forward(TcResNet* p, const float* feat, int64_t B, int T, int F, float* logits, void* ws,
                      size_t ws_bytes, int chunk_cfg, bool split, LaunchProfiler* prof, cudaStream_t st) {
  if (!p->supported) {
    set_error("bf16 tensor-core path supports 1..64 feature maps (got %d) and needs cuTensorMapEncodeTiled",
              p->cfg.n_maps);
    return KWS_ERR_UNSUPPORTED;
  }
  int H, W;
  resnet_map(p->cfg, T, F, &H, &W);
  KWS_REQUIRE(H >= 1 && W >= 1, "ResNet: input %dx%d is smaller than the pooling window", T, F);
  const size_t need = tc_resnet_workspace_bytes(p, B, T, F, chunk_cfg, split);
  if (need == 0) {
    set_error("%s tensor-core path cannot tile a %dx%d map", split ? "split-bf16" : "bf16", H, W);
    return KWS_ERR_UNSUPPORTED;
  }
  if (ws == nullptr || ws_bytes < need) {
    set_error("ResNet bf16 forward needs %zu bytes of workspace, got %zu", need, ws_bytes);
    return KWS_ERR_WORKSPACE;
  }
  const TcSweepPlan sp = tc_sweep_plan(p, H, W, split);
  if (sp.ok) return tc_sweep_forward(p, sp, feat, B, T, F, H, W, logits, ws, chunk_cfg, prof, st);
  return tc_fused_forward(p, tc_fused_plan(p, H, W, split), feat, B, T, F, H, W, logits, ws, prof, st);
}

}  // namespace kws
