// bf16 tensor-core (tcgen05 / TMEM) path of model.CNN for the cnn-trad-fpool3 shape family
// (/root/reference/model/cnn.py:79-107, config/cnn/cnn-trad-fpool3.json:5-49):
//
//   conv_0 (1 -> 64, KH0 x KW0<=8) + ReLU + MaxPool(1,3) + conv_1 (64 -> 64, KH1 x KW1, output width 8) + ReLU
//       one persistent whole-utterance kernel, `cnn_tc_fused_kernel`: the pooled conv_0 output never leaves the SM
//   x.view(B,-1) -> first Linear (<= 32 outputs)      `cnn_lin0_kernel` (split-K bf16 mma.sync over the stored conv_1
//                                                      output: HBM-bound, 75 KB per utterance read once)
//   remaining Linear layers                            `cnn_mlp_kernel` (fp32, sums the split-K partials first)
//
// Formulation of the two convolutions as implicit GEMMs with M = output positions, N = 64 output maps:
//
// * conv_0 has ONE input channel, so the K dimension must come from the taps.  A K chunk (8 bf16 = 16 bytes) is the
//   KW0 width taps of one kernel row: x[oh+kh][ow .. ow+7].  For output column ow = 3j + e (pool group j, member e)
//   the producer warps keep three arrays A_e[t][j] = bf16(x[t][3j+e .. 3j+e+7]) in shared memory (a width-only
//   im2col: 53 KB).  With rows n = t*WP + j (WP = pooled width) the operand of M-tile [128 i, 128 i+128), kernel rows
//   (kh, kh+1) is the canonical K-major SWIZZLE_NONE layout at start address A_e + (128 i + kh*WP)*16, LBO = WP*16:
//   a kernel-row shift is a start-address offset, no data is moved.  The three pool members of a group are the SAME
//   row n of three accumulators, so the epilogue thread that owns TMEM lane n does max(e) + bias + ReLU in registers
//   and writes pooled row n = oh*WP + j -- which is exactly the layout conv_1 reads.
// * conv_1: the pooled map lives in shared memory as eight 8-channel planes [plane][oh*WP + j][16 B] (115 KB).  The
//   output is 8 wide, so one 8-row core-matrix group is one output row: M index m = oh*8 + ow maps to address
//   (oh*WP + ow)*16 with SBO = WP*16, and tap (kh, kw) is the start offset (kh*WP + kw)*16.  All ceil(H1/16) M-tiles
//   (<= 5 x 64 TMEM columns) accumulate while the 320 KB of weights stream through a ring of 8 KB (kh, kw) units,
//   once per utterance, from L2.
//
// Warp roles (512 threads, one CTA per SM, persistent over its share of the batch): 0, 1, 3 MMA issuers (3 also owns the
// TMEM allocation), 2 weight-ring producer, 4-7 A_e builders, 8-15 epilogue.  Every accumulator is written by ONE issuer
// (bit-reproducible); every MMA accumulates and the epilogue zeroes what it has read (`tcgen05.st`).
// conv_0 accumulators: buffer 0 = TMEM columns [320, 512), buffer 1 = [0, 192) (the columns conv_1's tiles 0-2 use;
// conv_1 is a fifth "use" of buffer 1 per utterance in the empty/full bookkeeping).
#include "tc.cuh"
#include "ptx.cuh"
#include <algorithm>
#include <cstdlib>

namespace kws {

constexpr int kCnnC = 64;             // maps of conv_0 and conv_1
constexpr int kCnnIssuers = 3;
constexpr int kCnnWorkers = 16;          // worker warps: A_e builder + epilogue
constexpr int kCnnThreads = 32 * (4 + kCnnWorkers);   // warps 0, 1, 3 issue, warp 2 streams conv_1's weights
constexpr int kCnnRingUnit = 4 * 2 * kCnnC * 16;   // one (kh, kw) tap of conv_1: 4 K chunks x 2 halves x 64 x 16 B = 8 KB
constexpr int kCnnMaxRing = 8;
constexpr int kLin0Split = kTcCnnLin0Split;   // split-K factor of the first Linear
constexpr int kLin0Warps = 4;         // warps (16 utterances each) per CTA of the first Linear
constexpr int kLin0N = 32;            // padded outputs of the first Linear

struct TcCnnParams {
  const float* feat;            // [B][T][F]
  const __nv_bfloat16* w0;      // [ks0][2][64][8]
  const __nv_bfloat16* w1;      // [KH1*KW1][4][2][64][8]
  const float* b0;              // [64]
  const float* b1;              // [64]
  __nv_bfloat16* act;           // [B][4 channel groups][H1*8 positions][16]: a worker warp (32 positions x 16 channels) stores 1 KB
                                //   contiguous; the first Linear's weights are permuted to this order
  int64_t B;
  TcCnnGeom g;
  long long* debug;   // optional [16] cycle counters of CTA 0 (HONK2_TC_DEBUG=1), nullptr = off
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&v);
}
// bf16x2 {lo = relu(a), hi = relu(b)} in one instruction
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float a, float b) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

__global__ void __launch_bounds__(kCnnThreads, 1)
cnn_tc_fused_kernel(const TcCnnParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const TcCnnGeom& g = p.g;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 384);
  float* s_b0 = reinterpret_cast<float*>(smem + 512);
  float* s_b1 = reinterpret_cast<float*>(smem + 768);
  const uint32_t bar0 = smem_u32(bars);
  const uint32_t a_full = bar0, a_free = bar0 + 8, pool_full = bar0 + 16, c1_done = bar0 + 24;
  auto acc_full = [&](int b) { return bar0 + 32u + 8u * b; };
  auto acc_empty = [&](int b) { return bar0 + 48u + 8u * b; };
  auto s_full = [&](int s) { return bar0 + 64u + 8u * s; };
  auto s_empty = [&](int s) { return bar0 + 64u + 8u * (kCnnMaxRing + s); };

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(a_full, kCnnWorkers);
    mbar_init(a_free, kCnnIssuers);
    mbar_init(pool_full, kCnnWorkers);
    mbar_init(c1_done, kCnnIssuers);
    for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), kCnnIssuers); mbar_init(acc_empty(b), kCnnWorkers); }
    for (int s = 0; s < g.n_ring; ++s) { mbar_init(s_full(s), 1); mbar_init(s_empty(s), kCnnIssuers); }
    fence_barrier_init();
  }
  if (warp == 3) tmem_alloc(smem_u32(tmem_slot), 512);
  // conv_0 weights (resident), biases, zero rows of the A_e arrays
  {
    const uint4* src = reinterpret_cast<const uint4*>(p.w0);
    uint4* dst = reinterpret_cast<uint4*>(smem + g.off_w0);
    for (int i = threadIdx.x; i < g.ks0 * 128; i += kCnnThreads) dst[i] = src[i];
    if (threadIdx.x < kCnnC) { s_b0[threadIdx.x] = p.b0[threadIdx.x]; s_b1[threadIdx.x] = p.b1[threadIdx.x]; }
    for (int e = 0; e < 3; ++e) {
      uint4* a = reinterpret_cast<uint4*>(smem + g.off_a + e * g.a_bytes);
      for (int i = g.T * g.WP + threadIdx.x; i < g.a_rows; i += kCnnThreads) a[i] = make_uint4(0, 0, 0, 0);
    }
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const uint32_t w0_s = smem_u32(smem + g.off_w0);
  const uint32_t a_s = smem_u32(smem + g.off_a);
  const uint32_t pool_s = smem_u32(smem + g.off_pool);
  const uint32_t ring_s = smem_u32(smem + g.off_ring);
  constexpr uint32_t idesc = umma_idesc(128, kCnnC);
  constexpr uint32_t hi_128 = (128u >> 4) | (1u << 14);   // SBO = 128 B (8 rows x 16 B contiguous)

  if (warp < 2 || warp == 3) {
    // ===================================== MMA issuers =====================================
    // Three issuing threads keep the pipe fed (one thread sustains an MMA per ~55 cycles at best; an N = 64 MMA takes 48).
    // Every accumulator has ONE owner, so the order of the fp32 additions is fixed and the result is reproducible bit for
    // bit: issuer w owns pool member e = w of every conv_0 tile and the conv_1 M-tiles t = w, w+3; its first MMA into an
    // accumulator overwrites it.  All issuers work on the same conv_0 tile; tiles alternate between the two TMEM buffers,
    // so the epilogue of tile t overlaps the MMAs of tile t+1.
    const int w = warp == 3 ? 2 : warp;
    const bool leader = elect_one();
    const uint32_t hi_pool = ((uint32_t)(g.WP * 16) >> 4) | (1u << 14);   // SBO = one pooled row of 8 outputs
    const uint32_t lbo_w = (uint32_t)(kCnnC * 16 >> 4) << 16;             // weights: K halves 64 rows apart
    const uint32_t a0_base = (((a_s + (uint32_t)(w * g.a_bytes)) >> 4) & 0x3FFFu) | ((uint32_t)g.WP << 16);   // LBO = WP rows
    const uint32_t b0_base = ((w0_s >> 4) & 0x3FFFu) | lbo_w;
    const uint32_t a1_base = ((pool_s >> 4) & 0x3FFFu) | (((uint32_t)g.plane_bytes >> 4) << 16);               // LBO = next plane
    const uint32_t plane2 = (uint32_t)(2 * g.plane_bytes) >> 4;
    const int t1a = w, t1b = w + 3;                                        // this issuer's conv_1 tiles
    const bool has_b = t1b < g.tiles1, has_a = t1a < g.tiles1;
    uint32_t use[2] = {0, 0};   // uses of the two conv_0 accumulator buffers so far
    int stage = 0; uint32_t sphase = 0;
    uint32_t it = 0;
    const bool dbg = p.debug != nullptr && blockIdx.x == 0 && w == 0;
    long long d_afull = 0, d_aempty = 0, d_i0 = 0, d_pool = 0, d_sfull = 0, d_i1 = 0, d_t = clock64();
#define CNN_DBG(var) if (dbg) { const long long t_ = clock64(); var += t_ - d_t; d_t = t_; }
    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x, ++it) {
      // ---- conv_0
      mbar_wait_lean(a_full, it & 1);
      tc_fence_after();
      CNN_DBG(d_afull)
      for (int t = 0; t < g.tiles0; ++t) {
        const int buf = t & 1;
        mbar_wait_lean(acc_empty(buf), (use[buf] & 1) ^ 1);
        ++use[buf];
        tc_fence_after();
        CNN_DBG(d_aempty)
        if (leader) {
          const uint32_t d = tmem_base + (buf == 0 ? 320u : 0u) + 64u * w;
          const uint32_t a_t = a0_base + (uint32_t)(128 * t);
          umma_f16_lohi<false>(d, a_t, b0_base, hi_128, idesc);
#pragma unroll 3
          for (int ks = 1; ks < g.ks0; ++ks)
            umma_f16_lohi<true>(d, a_t + (uint32_t)(2 * ks * g.WP), b0_base + (uint32_t)(ks * 128), hi_128, idesc);
          umma_commit(acc_full(buf));
        }
        __syncwarp();
        CNN_DBG(d_i0)
      }
      if (leader) umma_commit(a_free);   // all conv_0 MMAs of this issuer have read the A_e arrays
      __syncwarp();
      // ---- conv_1: this issuer's M-tiles, every tap and K chunk
      mbar_wait_lean(pool_full, it & 1);
      mbar_wait_lean(acc_empty(1), (use[1] & 1) ^ 1);   // conv_1's tiles 0-2 are buffer 1's columns
      ++use[1];
      tc_fence_after();
      CNN_DBG(d_pool)
      int kw = 0;
      uint32_t tap = 0;                                           // (kh * WP + kw) rows
      for (int u = 0; u < g.units1; ++u) {
        mbar_wait_lean(s_full(stage), sphase);
        tc_fence_after();
        CNN_DBG(d_sfull)
        if (leader) {
          const uint32_t b_u = (((ring_s + (uint32_t)stage * kCnnRingUnit) >> 4) & 0x3FFFu) | lbo_w;
          if (has_a) {
            const uint32_t a_t = a1_base + tap + (uint32_t)(16 * t1a * g.WP);
            umma_f16_lohi2_rt(tmem_base + 64u * t1a, a_t, hi_pool, b_u, hi_128, idesc, u != 0);
#pragma unroll
            for (int kc = 1; kc < 4; ++kc)
              umma_f16_lohi2<true>(tmem_base + 64u * t1a, a_t + kc * plane2, hi_pool, b_u + kc * 128u, hi_128, idesc);
          }
          if (has_b) {
            const uint32_t a_t = a1_base + tap + (uint32_t)(16 * t1b * g.WP);
            umma_f16_lohi2_rt(tmem_base + 64u * t1b, a_t, hi_pool, b_u, hi_128, idesc, u != 0);
#pragma unroll
            for (int kc = 1; kc < 4; ++kc)
              umma_f16_lohi2<true>(tmem_base + 64u * t1b, a_t + kc * plane2, hi_pool, b_u + kc * 128u, hi_128, idesc);
          }
          umma_commit(s_empty(stage));
        }
        __syncwarp();
        CNN_DBG(d_i1)
        if (++kw == g.KW1) { kw = 0; tap += (uint32_t)(g.WP - g.KW1 + 1); } else { ++tap; }
        if (++stage == g.n_ring) { stage = 0; sphase ^= 1; }
      }
      if (leader) umma_commit(c1_done);
      __syncwarp();
    }
    if (dbg && lane == 0) {
      p.debug[0] = d_afull; p.debug[1] = d_aempty; p.debug[2] = d_i0; p.debug[3] = d_pool; p.debug[4] = d_sfull;
      p.debug[5] = d_i1; p.debug[6] = (long long)it;
    }
#undef CNN_DBG
  } else if (warp == 2) {
    // ===================================== conv_1 weight ring =====================================
    // (this warp has nothing else to do: it spins on the barrier instead of parking, a parked warp wakes up late)
    int stage = 0; uint32_t sphase = 0;
    const uint64_t pol = l2_policy_evict_last();
    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
      for (int u = 0; u < g.units1; ++u) {
        mbar_wait(s_empty(stage), sphase ^ 1);
        if (lane == 0) {
          mbar_expect_tx(s_full(stage), kCnnRingUnit);
          bulk_load_hint(ring_s + (uint32_t)stage * kCnnRingUnit,
                         reinterpret_cast<const unsigned char*>(p.w1) + (size_t)u * kCnnRingUnit, kCnnRingUnit,
                         s_full(stage), pol);
        }
        __syncwarp();
        if (++stage == g.n_ring) { stage = 0; sphase ^= 1; }
      }
    }
  } else {
    // ===================================== workers: A_e builder + epilogue =====================================
    // 16 warps: TMEM lane quarter q = warp % 4, 16-channel group cg = (warp - 4) / 4.  Per utterance: conv_0 epilogue
    // (8 tiles) -> build the next utterance's A_e arrays (conv_1 is running: these warps would idle) -> conv_1 epilogue.
    const int q = warp & 3, cg = (warp - 4) >> 2;
    const int wt = threadIdx.x - 128;                 // 0 .. 511
    const int lane_row = 32 * q + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * q) << 16) + 16u * cg;
    const int n_items = g.T * g.WP;
    auto build = [&](int64_t b) {
      const float* x = p.feat + b * (int64_t)g.T * g.F;
      for (int item = wt; item < n_items; item += 32 * kCnnWorkers) {
        const int t = item / g.WP, j = item - t * g.WP;
        const float* row = x + t * g.F + 3 * j;
        float v[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) v[i] = (3 * j + i < g.F) ? __ldg(row + i) : 0.f;
#pragma unroll
        for (int e = 0; e < 3; ++e) {
          uint4 o;
          o.x = pack_bf16x2(v[e], v[e + 1]);
          o.y = pack_bf16x2(v[e + 2], v[e + 3]);
          o.z = pack_bf16x2(v[e + 4], v[e + 5]);
          o.w = pack_bf16x2(v[e + 6], v[e + 7]);
          *reinterpret_cast<uint4*>(smem + g.off_a + e * g.a_bytes + item * 16) = o;
        }
      }
      fence_async_smem();   // generic-proxy stores -> visible to the MMA's async-proxy reads
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full);
    };
    uint32_t fullp[2] = {0, 0};
    uint32_t it = 0;
    const bool dbg = p.debug != nullptr && blockIdx.x == 0 && warp == 4;
    long long d_accfull = 0, d_e0 = 0, d_bld = 0, d_c1 = 0, d_e1 = 0, d_t = clock64();
#define CNN_DBG(var) if (dbg) { const long long t_ = clock64(); var += t_ - d_t; d_t = t_; }
    if ((int64_t)blockIdx.x < p.B) build(blockIdx.x);
    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x, ++it) {
      // ---- conv_0 tiles: max over the pool members + bias + ReLU -> pooled rows in shared memory
      for (int t = 0; t < g.tiles0; ++t) {
        const int buf = t & 1;
        mbar_wait_lean(acc_full(buf), fullp[buf]);
        fullp[buf] ^= 1;
        tc_fence_after();
        CNN_DBG(d_accfull)
        const int n = 128 * t + lane_row;
        const uint32_t col0 = lane_addr + (buf == 0 ? 320u : 0u);
        uint32_t v0[16], v1[16], v2[16];
        tmem_ld16(col0, v0);
        tmem_ld16(col0 + 64u, v1);
        tmem_ld16(col0 + 128u, v2);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty(buf));      // the accumulator is in registers: the next tile may overwrite it
        if (n < g.n0) {
          uint32_t o[8];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 bb = *reinterpret_cast<const float4*>(s_b0 + 16 * cg + 4 * i);
            o[2 * i] = pack_relu_bf16x2(max3(__uint_as_float(v0[4 * i]), __uint_as_float(v1[4 * i]), __uint_as_float(v2[4 * i])) + bb.x,
                                        max3(__uint_as_float(v0[4 * i + 1]), __uint_as_float(v1[4 * i + 1]), __uint_as_float(v2[4 * i + 1])) + bb.y);
            o[2 * i + 1] = pack_relu_bf16x2(max3(__uint_as_float(v0[4 * i + 2]), __uint_as_float(v1[4 * i + 2]), __uint_as_float(v2[4 * i + 2])) + bb.z,
                                            max3(__uint_as_float(v0[4 * i + 3]), __uint_as_float(v1[4 * i + 3]), __uint_as_float(v2[4 * i + 3])) + bb.w);
          }
          unsigned char* dst = smem + g.off_pool + (2 * cg) * g.plane_bytes + n * 16;
          *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<uint4*>(dst + g.plane_bytes) = make_uint4(o[4], o[5], o[6], o[7]);
        }
        CNN_DBG(d_e0)
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(pool_full);
      // ---- the next utterance's A_e arrays (this utterance's conv_0 MMAs have retired: a_free)
      if (b + gridDim.x < p.B) {
        mbar_wait_lean(a_free, it & 1);
        build(b + gridDim.x);
      }
      CNN_DBG(d_bld)
      // ---- conv_1 tiles: bias + ReLU -> bf16 activations [position][64] in global memory
      mbar_wait_lean(c1_done, it & 1);
      tc_fence_after();
      CNN_DBG(d_c1)
      __nv_bfloat16* act = p.act + b * (int64_t)(g.H1 * 8 * kCnnC) + (int64_t)cg * (g.H1 * 8 * 16);
      const uint32_t c1col = tmem_base + ((uint32_t)(32 * q) << 16) + 16u * cg;
      for (int t = 0; t < g.tiles1; t += 2) {
        uint32_t va[16], vb[16];
        const bool two = t + 1 < g.tiles1;
        tmem_ld16(c1col + 64u * t, va);
        if (two) tmem_ld16(c1col + 64u * (t + 1), vb);
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int oh = 16 * (t + h) + (lane_row >> 3), ow = lane_row & 7;
          if ((h == 0 || two) && oh < g.H1) {
            const uint32_t* v = h == 0 ? va : vb;
            uint32_t o[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 bb = *reinterpret_cast<const float4*>(s_b1 + 16 * cg + 4 * i);
              o[2 * i] = pack_relu_bf16x2(__uint_as_float(v[4 * i]) + bb.x, __uint_as_float(v[4 * i + 1]) + bb.y);
              o[2 * i + 1] = pack_relu_bf16x2(__uint_as_float(v[4 * i + 2]) + bb.z, __uint_as_float(v[4 * i + 3]) + bb.w);
            }
            uint4* dst = reinterpret_cast<uint4*>(act + (int64_t)(oh * 8 + ow) * 16);
            dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
            dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty(1));
      CNN_DBG(d_e1)
    }
    if (dbg && lane == 0) { p.debug[8] = d_accfull; p.debug[9] = d_e0; p.debug[10] = d_c1; p.debug[11] = d_e1; p.debug[12] = d_bld; }
#undef CNN_DBG
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// =============================================================================================
// First Linear over the stored conv_1 output: partial[s][b][n] = sum_{k in split s} act[b][k] * w[n][k].
// One warp = 16 utterances x 32 outputs, mma.sync m16n8k16 bf16; each thread loads 16 bytes (8 consecutive k) of its two
// rows and of its weight row, and the SAME k permutation is applied to both operands, so the products pair up.
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ROWS says where row r's activations are (DenseActRows, LiveActRows, RaggedActRows: tc.cuh).
template <typename ROWS>
__global__ void __launch_bounds__(32 * kLin0Warps)
cnn_lin0_kernel(const ROWS rows, const __nv_bfloat16* __restrict__ w, float* __restrict__ partial,
                int64_t B, int K, int k_per_split) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gq = lane >> 2, tq = lane & 3;
  const int64_t row0 = ((int64_t)blockIdx.x * kLin0Warps + warp) * 16;
  if (row0 >= B) return;
  const int split = blockIdx.y;
  const int k0 = split * k_per_split, k1 = min(K, k0 + k_per_split);
  const int64_t ra = min(row0 + gq, B - 1), rb = min(row0 + gq + 8, B - 1);
  const typename ROWS::Cursor pa = rows.row(ra, K, tq), pb = rows.row(rb, K, tq);
  const uint4* pw[4];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) pw[nt] = reinterpret_cast<const uint4*>(w + (int64_t)(8 * nt + gq) * K) + tq;
  float c[4][4];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) c[nt][i] = 0.f;
#pragma unroll 4
  for (int k = k0; k < k1; k += 32) {
    const int o = k >> 3;
    const uint4 a = __ldcs(pa.at(o)), bq = __ldcs(pb.at(o));
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const uint4 wv = __ldg(pw[nt] + o);
      mma_bf16_16816(c[nt], a.x, bq.x, a.y, bq.y, wv.x, wv.y);
      mma_bf16_16816(c[nt], a.z, bq.z, a.w, bq.w, wv.z, wv.w);
    }
  }
  float* out = partial + (int64_t)split * B * kLin0N;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    if (row0 + gq < B) *reinterpret_cast<float2*>(out + (row0 + gq) * kLin0N + 8 * nt + 2 * tq) = make_float2(c[nt][0], c[nt][1]);
    if (row0 + gq + 8 < B) *reinterpret_cast<float2*>(out + (row0 + gq + 8) * kLin0N + 8 * nt + 2 * tq) = make_float2(c[nt][2], c[nt][3]);
  }
}

// Remaining Linear layers in fp32 (cnn.py:95-106): sums the split-K partials of the first layer in a fixed order,
// adds its bias, then up to three more layers.  One CTA handles 8 utterances; thread = output.
struct MlpLayer { const float* w; const float* b; int in, out; };
struct MlpParams {
  const float* partial;   // [kLin0Split][B][kLin0N]
  const float* bias_first;
  int first_out;
  MlpLayer layer[3];
  int n_layers;
  float* logits;          // [B][n_labels] (n_labels = out of the last layer, or first_out)
  int64_t B;
};
constexpr int kMlpUtt = 8, kMlpMax = 512;

__global__ void __launch_bounds__(256)
cnn_mlp_kernel(const MlpParams p) {
  __shared__ float h[2][kMlpUtt][kMlpMax];
  const int64_t b0 = (int64_t)blockIdx.x * kMlpUtt;
  const int nu = (int)(p.B - b0 < kMlpUtt ? p.B - b0 : kMlpUtt);
  for (int i = threadIdx.x; i < nu * p.first_out; i += blockDim.x) {
    const int u = i / p.first_out, n = i - u * p.first_out;
    float v = 0.f;
    for (int s = 0; s < kLin0Split; ++s) v += p.partial[((int64_t)s * p.B + b0 + u) * kLin0N + n];
    v += __ldg(p.bias_first + n);
    if (p.n_layers == 0) p.logits[(b0 + u) * p.first_out + n] = v;
    else h[0][u][n] = v;
  }
  int cur = 0;
  for (int l = 0; l < p.n_layers; ++l) {
    __syncthreads();
    const MlpLayer& L = p.layer[l];
    const bool last = l == p.n_layers - 1;
    for (int n = threadIdx.x; n < L.out; n += blockDim.x) {
      float acc[kMlpUtt];
      const float bias = __ldg(L.b + n);
#pragma unroll
      for (int u = 0; u < kMlpUtt; ++u) acc[u] = bias;
      const float* wr = L.w + (int64_t)n * L.in;
      for (int k = 0; k < L.in; ++k) {
        const float wv = __ldg(wr + k);
#pragma unroll
        for (int u = 0; u < kMlpUtt; ++u) acc[u] = fmaf(wv, h[cur][u][k], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < kMlpUtt; ++u) {
        if (u < nu) {
          if (last) p.logits[(b0 + u) * L.out + n] = acc[u];
          else h[cur ^ 1][u][n] = acc[u];
        }
      }
    }
    cur ^= 1;
  }
}

// =============================================================================================
// weight packing (once per load_state_dict)

__global__ void pack_cnn_w0_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int KH0, int KW0, int ks0) {
  const int total = ks0 * 2 * kCnnC * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int kw = i & 7, co = (i >> 3) & 63, half = (i >> 9) & 1, ks = i >> 10;
    const int kh = 2 * ks + half;
    out[i] = __float2bfloat16((kh < KH0 && kw < KW0) ? w[(co * KH0 + kh) * KW0 + kw] : 0.f);
  }
}

__global__ void pack_cnn_w1_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int KH1, int KW1) {
  const int total = KH1 * KW1 * 4 * 2 * kCnnC * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i & 7, co = (i >> 3) & 63, half = (i >> 9) & 1, kc = (i >> 10) & 3, u = i >> 12;
    const int kh = u / KW1, kw = u - kh * KW1;
    const int ci = 16 * kc + 8 * half + e;
    out[i] = __float2bfloat16(w[((int64_t)(co * kCnnC + ci) * KH1 + kh) * KW1 + kw]);
  }
}

// torch [out][c*M + m] -> bf16 [kLin0N][(c/16)*M*16 + m*16 + c%16] (the order the fused kernel stores), rows >= out are zero
__global__ void pack_cnn_lin0_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int n_out, int M) {
  const int64_t K = (int64_t)M * kCnnC, total = K * kLin0N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i / K);
    const int64_t r = i - n * K;
    const int cg = (int)(r / ((int64_t)M * 16));
    const int64_t r2 = r - (int64_t)cg * M * 16;
    const int m = (int)(r2 / 16), c = 16 * cg + (int)(r2 - (int64_t)m * 16);
    out[i] = __float2bfloat16(n < n_out ? w[(int64_t)n * K + (int64_t)c * M + m] : 0.f);
  }
}

// =============================================================================================
// host side

struct TcCnn {
  kws_cnn_config cfg{};
  bool supported = false;
  const char* why = "";
  TcCnnGeom g{};
  int first = -1;              // index (0 lin_0, 1 dnn_0, 2 dnn_1, 3 lin_1) of the first Linear
  int lin_in[4] = {0, 0, 0, 0}, lin_out[4] = {0, 0, 0, 0};
  unsigned char* blob = nullptr;
  size_t blob_bytes = 0;
  __nv_bfloat16 *w0 = nullptr, *w1 = nullptr, *wl = nullptr;
  float *b0 = nullptr, *b1 = nullptr;
  float* lin_w[4] = {nullptr, nullptr, nullptr, nullptr};
  float* lin_b[4] = {nullptr, nullptr, nullptr, nullptr};
  long long* debug = nullptr;   // HONK2_TC_DEBUG=1: device counters printed after every launch (synchronises)
};

static bool cnn_tc_plan(TcCnn* p) {
  const kws_cnn_config& c = p->cfg;
  TcCnnGeom& g = p->g;
  auto no = [&](const char* why) { p->why = why; return false; };
  if (c.conv0_out != kCnnC || c.conv1_out != kCnnC) return no("conv_0 and conv_1 must have 64 maps");
  if (c.conv0_sh != 1 || c.conv0_sw != 1 || c.conv1_sh != 1 || c.conv1_sw != 1) return no("strided convolutions");
  if (c.pool0_kh != 1 || c.pool0_kw != 3 || c.pool1_kh != 1 || c.pool1_kw != 1) return no("pooling other than (1,3) / (1,1)");
  if (c.conv0_kw > 8 || c.conv0_kw < 1) return no("conv_0 wider than 8 taps");
  g.T = c.time; g.F = c.freq; g.KH0 = c.conv0_kh; g.KW0 = c.conv0_kw;
  g.H0 = c.time - c.conv0_kh + 1;
  const int W0 = c.freq - c.conv0_kw + 1;
  if (g.H0 < 1 || W0 < 3) return no("input smaller than conv_0 / pool_0");
  g.WP = W0 / 3;
  g.KH1 = c.conv1_kh; g.KW1 = c.conv1_kw;
  g.H1 = g.H0 - g.KH1 + 1;
  if (g.H1 < 1 || g.WP - g.KW1 + 1 != 8) return no("conv_1 output must be 8 wide");
  g.n0 = g.H0 * g.WP;
  g.tiles0 = ceil_div(g.n0, 128);
  g.ks0 = ceil_div(g.KH0, 2);
  g.tiles1 = ceil_div(g.H1, 16);
  if (g.tiles1 > 5) return no("conv_1 output taller than 80 rows (TMEM columns)");
  g.units1 = g.KH1 * g.KW1;
  g.a_rows = g.T * g.WP + g.WP;
  g.off_w0 = 1024;
  g.off_a = g.off_w0 + g.ks0 * 2048;
  g.a_bytes = g.a_rows * 16;
  g.off_pool = g.off_a + 3 * g.a_bytes;
  g.plane_bytes = g.n0 * 16;
  g.off_ring = g.off_pool + 8 * g.plane_bytes;
  // operand over-reads (rows of M-tiles past the map) must stay inside the CTA's shared memory window
  const int a_reach = (128 * g.tiles0 + (2 * g.ks0 - 1) * g.WP) * 16 + 2 * g.a_bytes;       // furthest A_e byte read
  const int p_reach = 7 * g.plane_bytes + ((16 * g.tiles1 + g.KH1 - 1) * g.WP + g.KW1 + 7) * 16;
  const int cap = 227 * 1024;
  int ring = (cap - g.off_ring) / kCnnRingUnit;
  if (ring > kCnnMaxRing) ring = kCnnMaxRing;
  if (ring > g.units1) ring = g.units1;
  if (ring < 2) return no("shared memory (pooled map + operands leave no room for the weight ring)");
  g.n_ring = ring;
  g.smem_bytes = g.off_ring + ring * kCnnRingUnit;
  if (g.off_a + a_reach > g.smem_bytes || g.off_pool + p_reach > g.smem_bytes) return no("operand over-read");
  if ((g.plane_bytes >> 4) > 0x3FFF) return no("pooled plane too large for the descriptor");
  // linear stack
  const int outs[4] = {c.lin0_out, c.dnn0_out, c.dnn1_out, c.n_labels};
  int in = kCnnC * g.H1 * 8;
  for (int i = 0; i < 4; ++i) {
    if (outs[i] <= 0) continue;
    if (p->first < 0) p->first = i;
    p->lin_in[i] = in; p->lin_out[i] = outs[i];
    in = outs[i];
  }
  if (p->first < 0 || p->lin_out[p->first] > kLin0N) return no("first Linear wider than 32 outputs");
  for (int i = p->first + 1; i < 4; ++i)
    if (p->lin_out[i] > kMlpMax || (p->lin_out[i] > 0 && p->lin_in[i] > kMlpMax)) return no("Linear layer wider than 512");
  return true;
}

int tc_cnn_create(const kws_cnn_config& cfg, TcCnn** out) {
  TcCnn* p = new TcCnn();
  p->cfg = cfg;
  p->supported = cnn_tc_plan(p);
  *out = p;
  if (!p->supported) return KWS_OK;
  const char* dbg_env = getenv("HONK2_TC_DEBUG");
  const bool want_debug = dbg_env != nullptr && atoi(dbg_env) != 0;
  const TcCnnGeom& g = p->g;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += round_up<size_t>(bytes, 256); return o; };
  const size_t o_w0 = take((size_t)g.ks0 * 2048), o_w1 = take((size_t)g.units1 * kCnnRingUnit);
  const size_t o_wl = take((size_t)kLin0N * kCnnC * g.H1 * 8 * 2), o_b0 = take(256), o_b1 = take(256);
  size_t o_lw[4] = {0, 0, 0, 0}, o_lb[4] = {0, 0, 0, 0};
  for (int i = 0; i < 4; ++i)
    if (p->lin_out[i] > 0) {
      o_lb[i] = take(sizeof(float) * p->lin_out[i]);
      if (i != p->first) o_lw[i] = take(sizeof(float) * (size_t)p->lin_out[i] * p->lin_in[i]);
    }
  p->blob_bytes = off;
  cudaError_t e = cudaMalloc(&p->blob, off);
  if (e != cudaSuccess) {
    set_error("tc_cnn_create: cudaMalloc(%zu) failed: %s", off, cudaGetErrorString(e));
    delete p;
    *out = nullptr;
    return KWS_ERR_CUDA;
  }
  if (want_debug && cudaMalloc(&p->debug, 16 * sizeof(long long)) != cudaSuccess) p->debug = nullptr;
  p->w0 = reinterpret_cast<__nv_bfloat16*>(p->blob + o_w0);
  p->w1 = reinterpret_cast<__nv_bfloat16*>(p->blob + o_w1);
  p->wl = reinterpret_cast<__nv_bfloat16*>(p->blob + o_wl);
  p->b0 = reinterpret_cast<float*>(p->blob + o_b0);
  p->b1 = reinterpret_cast<float*>(p->blob + o_b1);
  for (int i = 0; i < 4; ++i)
    if (p->lin_out[i] > 0) {
      p->lin_b[i] = reinterpret_cast<float*>(p->blob + o_lb[i]);
      if (i != p->first) p->lin_w[i] = reinterpret_cast<float*>(p->blob + o_lw[i]);
    }
  e = raise_dynamic_smem(cnn_tc_fused_kernel, g.smem_bytes);
  if (e != cudaSuccess) {
    set_error("tc_cnn_create: raising the shared memory limit to %d failed: %s", g.smem_bytes, cudaGetErrorString(e));
    cudaFree(p->blob);
    delete p;
    *out = nullptr;
    return KWS_ERR_CUDA;
  }
  return KWS_OK;
}

void tc_cnn_destroy(TcCnn* p) {
  if (!p) return;
  if (p->blob) cudaFree(p->blob);
  if (p->debug) cudaFree(p->debug);
  delete p;
}

bool tc_cnn_supported(const TcCnn* p, const char** why) {
  if (why) *why = p ? p->why : "no plan";
  return p && p->supported;
}

int tc_cnn_set_weights(TcCnn* p, const kws_cnn_weights& w, cudaStream_t st) {
  if (!p || !p->supported) return KWS_OK;
  const TcCnnGeom& g = p->g;
  pack_cnn_w0_kernel<<<ceil_div(g.ks0 * 1024, 256), 256, 0, st>>>(w.conv0_w, p->w0, g.KH0, g.KW0, g.ks0);
  KWS_CUDA(cudaGetLastError());
  pack_cnn_w1_kernel<<<ceil_div(g.units1 * 4096, 256), 256, 0, st>>>(w.conv1_w, p->w1, g.KH1, g.KW1);
  KWS_CUDA(cudaGetLastError());
  KWS_CUDA(cudaMemcpyAsync(p->b0, w.conv0_b, sizeof(float) * kCnnC, cudaMemcpyDeviceToDevice, st));
  KWS_CUDA(cudaMemcpyAsync(p->b1, w.conv1_b, sizeof(float) * kCnnC, cudaMemcpyDeviceToDevice, st));
  const float* lw[4] = {w.lin0_w, w.dnn0_w, w.dnn1_w, w.lin1_w};
  const float* lb[4] = {w.lin0_b, w.dnn0_b, w.dnn1_b, w.lin1_b};
  for (int i = 0; i < 4; ++i) {
    if (p->lin_out[i] <= 0) continue;
    KWS_REQUIRE(lw[i] && lb[i], "tc_cnn_set_weights: linear layer %d tensors are null", i);
    KWS_CUDA(cudaMemcpyAsync(p->lin_b[i], lb[i], sizeof(float) * p->lin_out[i], cudaMemcpyDeviceToDevice, st));
    if (i == p->first) {
      pack_cnn_lin0_kernel<<<1024, 256, 0, st>>>(lw[i], p->wl, p->lin_out[i], g.H1 * 8);
      KWS_CUDA(cudaGetLastError());
    } else {
      KWS_CUDA(cudaMemcpyAsync(p->lin_w[i], lw[i], sizeof(float) * (size_t)p->lin_out[i] * p->lin_in[i],
                               cudaMemcpyDeviceToDevice, st));
    }
  }
  return KWS_OK;
}

static int64_t cnn_tc_chunk(const TcCnn* p, int64_t B, int chunk) {
  int64_t c = chunk > 0 ? chunk : 8192;   // one launch per 8192 utterances measured best (612 MB of conv_1 output; 2048-utterance
                                         // sub-batches keep it closer to the L2 but pay three more launch ramps: 2.18 vs 2.44 M utt/s)
  if (c > B) c = B;
  if (c < 1) c = 1;
  return c;
}

size_t tc_cnn_workspace_bytes(const TcCnn* p, int64_t B, int T, int F, int chunk) {
  if (!p || !p->supported || T != p->g.T || F != p->g.F) return 0;
  const int64_t c = cnn_tc_chunk(p, B, chunk);
  return round_up<size_t>((size_t)c * p->g.H1 * 8 * kCnnC * 2, 256) + round_up<size_t>((size_t)kLin0Split * c * kLin0N * 4, 256);
}

int tc_cnn_forward(TcCnn* p, const float* feat, int64_t B, int T, int F, float* logits, void* ws, size_t ws_bytes,
                   int chunk, LaunchProfiler* prof, cudaStream_t st) {
  KWS_REQUIRE(p != nullptr && p->supported, "CNN: no tensor-core path for this configuration (%s)", p ? p->why : "no plan");
  const TcCnnGeom& g = p->g;
  KWS_REQUIRE(T == g.T && F == g.F, "CNN: input is %dx%d but the model was built for %dx%d (cnn.py:16-17)", T, F, g.T, g.F);
  const size_t need = tc_cnn_workspace_bytes(p, B, T, F, chunk);
  if (ws == nullptr || ws_bytes < need) {
    set_error("CNN bf16 forward needs %zu bytes of workspace, got %zu", need, ws_bytes);
    return KWS_ERR_WORKSPACE;
  }
  const int64_t c = cnn_tc_chunk(p, B, chunk);
  const int K = g.H1 * 8 * kCnnC;
  __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(ws);
  float* partial = reinterpret_cast<float*>(static_cast<char*>(ws) + round_up<size_t>((size_t)c * K * 2, 256));
  int n_labels = 0;
  for (int i = 0; i < 4; ++i) if (p->lin_out[i] > 0) n_labels = p->lin_out[i];
  for (int64_t b0 = 0; b0 < B; b0 += c) {
    const int64_t nb = std::min<int64_t>(c, B - b0);
    TcCnnParams prm;
    prm.feat = feat + b0 * (int64_t)T * F;
    prm.w0 = p->w0; prm.w1 = p->w1; prm.b0 = p->b0; prm.b1 = p->b1;
    prm.act = act; prm.B = nb; prm.g = g; prm.debug = p->debug;
    if (p->debug) cudaMemsetAsync(p->debug, 0, 16 * sizeof(long long), st);
    if (prof) prof->tick(0, st);
    const unsigned grid = (unsigned)std::min<int64_t>(nb, kNumSMs);
    cnn_tc_fused_kernel<<<grid, kCnnThreads, g.smem_bytes, st>>>(prm);
    KWS_CHECK_LAUNCH();
    if (p->debug) {
      long long h[16];
      if (cudaMemcpyAsync(h, p->debug, sizeof(h), cudaMemcpyDeviceToHost, st) == cudaSuccess &&
          cudaStreamSynchronize(st) == cudaSuccess && h[6] > 0)
        fprintf(stderr, "[cnn_tc] CTA 0, %lld utterances, cycles per utterance: issuer 0 waits a_full %lld acc_empty %lld "
                        "pool_full %lld s_full %lld, issues conv_0 %lld conv_1 %lld | worker warp waits acc_full %lld "
                        "c1_done %lld, works conv_0 %lld build %lld conv_1 %lld\n",
                h[6], h[0] / h[6], h[1] / h[6], h[3] / h[6], h[4] / h[6], h[2] / h[6], h[5] / h[6], h[8] / h[6], h[10] / h[6],
                h[9] / h[6], h[12] / h[6], h[11] / h[6]);
    }
    if (prof) prof->tick(1, st);
    const int k_per = round_up(ceil_div(K, kLin0Split), 32);
    cnn_lin0_kernel<<<dim3((unsigned)ceil_div<int64_t>(nb, 16 * kLin0Warps), kLin0Split), 32 * kLin0Warps, 0, st>>>(
        DenseActRows{act}, p->wl, partial, nb, K, k_per);
    KWS_CHECK_LAUNCH();
    MlpParams mp{};
    mp.partial = partial;
    mp.bias_first = p->lin_b[p->first];
    mp.first_out = p->lin_out[p->first];
    mp.n_layers = 0;
    for (int i = p->first + 1; i < 4; ++i)
      if (p->lin_out[i] > 0) mp.layer[mp.n_layers++] = MlpLayer{p->lin_w[i], p->lin_b[i], p->lin_in[i], p->lin_out[i]};
    mp.logits = logits + b0 * n_labels;
    mp.B = nb;
    if (prof) prof->tick(1, st);
    cnn_mlp_kernel<<<(unsigned)ceil_div<int64_t>(nb, kMlpUtt), 256, 0, st>>>(mp);
    KWS_CHECK_LAUNCH();
  }
  return KWS_OK;
}

bool tc_cnn_view(const TcCnn* p, TcCnnView* v) {
  if (!p || !p->supported) return false;
  v->g = p->g;
  v->w0 = p->w0; v->w1 = p->w1; v->b0 = p->b0; v->b1 = p->b1;
  v->blob_bytes = p->blob_bytes;
  v->n_labels = 0;
  for (int i = 0; i < 4; ++i) if (p->lin_out[i] > 0) v->n_labels = p->lin_out[i];
  return true;
}

int tc_cnn_copy(const TcCnn* src, TcCnn** out, cudaStream_t st) {
  *out = nullptr;
  KWS_REQUIRE(src != nullptr && src->supported, "CNN: no tensor-core path for this configuration");
  TcCnn* p = nullptr;
  KWS_TRY(tc_cnn_create(src->cfg, &p));
  if (p->blob_bytes != src->blob_bytes) {
    tc_cnn_destroy(p);
    set_error("tc_cnn_copy: plans of one configuration differ in size");
    return KWS_ERR_INVALID;
  }
  const cudaError_t e = cudaMemcpyAsync(p->blob, src->blob, src->blob_bytes, cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) {
    tc_cnn_destroy(p);
    set_error("tc_cnn_copy: %s", cudaGetErrorString(e));
    return KWS_ERR_CUDA;
  }
  *out = p;
  return KWS_OK;
}

template <typename ROWS>
static int live_linear(const TcCnn* p, const ROWS& rows, int64_t B, float* partial, float* logits, cudaStream_t st) {
  KWS_REQUIRE(p != nullptr && p->supported, "CNN: no tensor-core path for this configuration");
  const int K = p->g.H1 * 8 * kCnnC;
  const int k_per = round_up(ceil_div(K, kLin0Split), 32);   // the batch path's split-K slices
  cnn_lin0_kernel<<<dim3((unsigned)ceil_div<int64_t>(B, 16 * kLin0Warps), kLin0Split), 32 * kLin0Warps, 0, st>>>(
      rows, p->wl, partial, B, K, k_per);
  KWS_CHECK_LAUNCH();
  MlpParams mp{};
  mp.partial = partial;
  mp.bias_first = p->lin_b[p->first];
  mp.first_out = p->lin_out[p->first];
  mp.n_layers = 0;
  for (int i = p->first + 1; i < 4; ++i)
    if (p->lin_out[i] > 0) mp.layer[mp.n_layers++] = MlpLayer{p->lin_w[i], p->lin_b[i], p->lin_in[i], p->lin_out[i]};
  mp.logits = logits;
  mp.B = B;
  cnn_mlp_kernel<<<(unsigned)ceil_div<int64_t>(B, kMlpUtt), 256, 0, st>>>(mp);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

int tc_cnn_live_linear(const TcCnn* p, const LiveActRows& rows, int64_t B, float* partial, float* logits,
                       cudaStream_t st) {
  return live_linear(p, rows, B, partial, logits, st);
}

int tc_cnn_live_linear(const TcCnn* p, const RaggedActRows& rows, int64_t B, float* partial, float* logits,
                       cudaStream_t st) {
  return live_linear(p, rows, B, partial, logits, st);
}

}  // namespace kws
