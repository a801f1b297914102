// Whole-network persistent kernel of the bf16 tensor-core ResNet path (included by conv_tc.cu).
//
// One launch runs conv_0 -> all C->C layers -> global mean -> Linear for the whole batch
// (/root/reference/model/resnet.py:38-60).  Each CTA (one per SM) owns an "utterance slot": two
// planar-8 activation buffers in global memory that it reuses for every utterance it processes, so
// the working set is n_sms x 2 x 388 KB (L2 resident) whatever the batch size, no activation ever
// makes a round trip through HBM, there is no inter-CTA synchronisation at all (utterances are
// independent), and tiles never straddle a launch boundary.
//
// Per utterance:   conv_0 (epilogue warps, CUDA cores) -> P
//                  layer i odd : TMA reads P, epilogue writes Q
//                  layer i even: TMA reads Q, epilogue adds the skip (read from P) and writes P in place
//                  last layer  : epilogue accumulates the pooled sums in shared memory -> logits
// Between layers the CTA drains: epilogue stores -> __threadfence + fence.proxy.async -> __syncthreads
// -> the producer may issue TMA loads of what was just written.  Weights of layer i+1 are bulk-copied
// into the second weight buffer while layer i runs.
//
// Activation layout ("planar-8"): [slot][NP][Hpad][W][8] bf16, NP = CP/8 planes of 8 channels,
// CP = channels padded to a multiple of 16 (45 -> 48).  One plane row is W*16 contiguous bytes,
// so a TMA box {8 ch, Wp, rows} lands in shared memory as a dense array of 16-byte "positions":
// exactly the UMMA K-major SWIZZLE_NONE canonical layout (core matrix = 8 positions x 16 B,
// SBO = 128 B), in which a pixel shift is nothing but a start-address offset.
//
// Implicit GEMM per tap (dh, dw) and 16-channel chunk kc:
//   D[128 positions x CP] += A[128 positions x 16] (shifted view of the staged tile)
//                          * B[16 x CP]            (weights, resident in shared memory)
// Positions are flat indices p = r * Wp + c into the zero-padded tile rows (Wp = W + d: the d
// left-pad columns of row r+1 double as the right padding of row r; TMA out-of-bounds fill
// supplies every zero).  Outputs at pad positions are computed and discarded.  Tile rows and
// boxes come from tc_geom (conv_tc.cu); large dilations tile by phase (rows p, p+d, p+2d, ...).
//
// Warp roles (tc_threads(NKC) threads, 1 CTA per SM; every role walks the same tile sequence):
//   warp 0             TMA producer: one ring stage = one 16-channel chunk of the haloed input tile
//   warps 1-3          MMA issuers, one elected lane each; the M-tiles of a tile are dealt round-robin
//                      (warp 1 also allocates TMEM)
//   4*NKC warps        epilogue: tcgen05.ld -> ReLU -> +skip -> BN -> bf16 planar-8 stores
//                      (last layer: pooled sums instead of stores)
// TMEM holds two accumulator buffers (up to min(8, 256 / CP) M-tiles x CP columns each) so the
// epilogue of tile i overlaps the MMAs of tile i+1.
//
// SPLIT (the "bf16x3" precision): activations and weights are carried as bf16 pairs hi + lo (planes 0 .. NP-1 hold the
// hi parts, NP .. 2 NP-1 the lo parts; the lo weight set follows the hi set) and every product is three MMAs,
// hi*hi + hi*lo + lo*hi, accumulated in fp32: fp32-grade logits at a third of the bf16 MMA rate.  The two weight sets
// of a layer share ONE buffer, loaded at the start of the layer (the CTA has just drained anyway).
#pragma once

namespace kws {

constexpr int kFusedStages = 4;     // most ring slots (the plan takes fewer, down to 2, when a layer's staged tile is large)
constexpr int kFusedMaxLayers = 64;

struct TcLayerDesc {
  TcGeom g;
  const __nv_bfloat16* wpack;
  const float* kconst;
  int in_buf;     // 0: P, 1: Q
  int has_skip;   // even layer: skip from P, output to P (in place)
  int last;       // pooling instead of a store
  int pad_;
};

struct TcFusedParams {
  const TcLayerDesc* layers;     // [n_layers]  (global memory)
  const CUtensorMap* maps;       // [n_layers]  input tensor map of every layer (global memory, 64 B aligned)
  const float* feat;             // [B][T][F]
  const float* conv0_w;          // [C][9]
  const float* last_scale;       // [CP] 1/sigma of the last BatchNorm (folded into the Linear)
  const float* out_w;            // [n_labels][C]
  const float* out_b;            // [n_labels]
  float* logits;                 // [B][n_labels]
  __nv_bfloat16* P;              // [n_slots][NP][Hpad][W][8]  (SPLIT: 2 NP planes per slot)
  __nv_bfloat16* Q;
  int64_t B;
  int n_layers, C, n_labels, T, F, ph, pw, H, W, Hpad;
  int smem_w_off[2], smem_ring_off, ring_slot_bytes;
  int n_stages;       // ring slots in use (2 .. kFusedStages)
  long long* debug;   // optional [16] cycle counters written by CTA 0's first issuer thread (nullptr = off)
};

template <int NKC, bool SPLIT>
__global__ void __launch_bounds__(tc_threads(NKC), 1)
resnet_tc_fused_kernel(const TcFusedParams p) {
  constexpr int kThreads = tc_threads(NKC);
  constexpr int kEpiWarps = tc_epi_warps(NKC);
  constexpr int CP = 16 * NKC;
  constexpr int NP = 2 * NKC;
  constexpr int NPX = SPLIT ? 2 * NP : NP;             // planes per utterance slot
  constexpr int NA = SPLIT ? 2 * NKC : NKC;            // staged 16-channel chunks per tile (SPLIT: hi chunks, then lo chunks)
  constexpr int W_HALF = CP * 16;
  constexpr int W_PART = 9 * NKC * 2 * W_HALF;         // one weight set
  constexpr int W_BYTES = (SPLIT ? 2 : 1) * W_PART;
  constexpr int MAXMT = (kAccCols / CP) < kTcMaxMt ? (kAccCols / CP) : kTcMaxMt;
  constexpr int MAXU = (MAXMT + kTcIssuers - 1) / kTcIssuers;
  extern __shared__ __align__(1024) unsigned char smem[];

  // ---- shared memory carve-up (first 6 KB: control)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);    // full[4], empty[4], tfull[2], tempty[2], wfull[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 128);
  float* s_pool = reinterpret_cast<float*>(smem + 4608);                // [4 lane quarters][CP] pooled sums of the current utterance
  float* s_kconst = reinterpret_cast<float*>(smem + 512);               // [2][CP]
  TcLayerDesc* s_layer = reinterpret_cast<TcLayerDesc*>(smem + 1024);   // [2]
  float* s_w0 = reinterpret_cast<float*>(smem + 1536);                  // [CP][12] conv_0 weights (<= 64*12*4 = 3 KB)
  unsigned char* s_ring = smem + p.smem_ring_off;
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kFusedStages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * kFusedStages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * kFusedStages + 2 + a); };
  auto wfull_bar = [&](int i) { return bar0 + 8u * (2 * kFusedStages + 4 + i); };

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_layers = p.n_layers;
  const int64_t n_my = (p.B - blockIdx.x + gridDim.x - 1) / gridDim.x;   // utterances this CTA processes
  const int64_t n_seq = n_my * n_layers;                                  // (utterance, layer) steps

  // ---- one-time setup
  if (threadIdx.x == 0) {
    for (int s = 0; s < kFusedStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), kTcIssuers); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), kTcIssuers); mbar_init(tempty_bar(a), kEpiWarps); }
    mbar_init(wfull_bar(0), 1);
    mbar_init(wfull_bar(1), 1);
    fence_barrier_init();
    if (n_seq > 0) {   // weights + descriptor of the first layer (SPLIT loads every layer's weights at its start)
      if constexpr (!SPLIT) {
        mbar_expect_tx(wfull_bar(0), W_BYTES);
        bulk_load(smem_u32(smem + p.smem_w_off[0]), p.layers[0].wpack, W_BYTES, wfull_bar(0));
      }
      s_layer[0] = p.layers[0];
    }
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  for (int i = threadIdx.x; i < CP * 12; i += kThreads) {
    const int c = i / 12, k = i - c * 12;
    s_w0[i] = (k < 9 && c < p.C) ? p.conv0_w[c * 9 + k] : 0.f;
  }
  for (int i = threadIdx.x; i < CP; i += kThreads) {
    if (n_seq > 0) s_kconst[i] = p.layers[0].kconst[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t plane_stride = (int64_t)p.Hpad * p.W;                    // 16-byte units
  const int64_t slot_base = (int64_t)blockIdx.x * NPX * plane_stride;    // this CTA's utterance slot
  uint4* bufP = reinterpret_cast<uint4*>(p.P) + slot_base;
  uint4* bufQ = reinterpret_cast<uint4*>(p.Q) + slot_base;

  // The two slot buffers of all CTAs together are about as large as the L2, so plain LRU thrashes.  P is
  // kept (evict_last): it is read as the odd layers' input, read again as the skip tensor and rewritten in
  // place.  Q streams (evict_first): written once, read once.  Each policy is created where it is used: one
  // instruction, and no register pair held for the whole kernel.

  // pipeline state (persists across layers and utterances; every role walks the same tile sequence)
  int stage = 0, acc = 0;
  uint32_t phase = 0, acc_phase = 0;

  auto tile_decode = [&](const TcGeom& g, int tix, int& ph, int& r0, int& rows) {
    if (g.phase) {
      ph = tix / g.chunks_per_phase;
      r0 = (tix - ph * g.chunks_per_phase) * g.R;
      rows = min(g.R, (g.H - ph + g.d - 1) / g.d - r0);
    } else {
      ph = 0;
      r0 = tix * g.R;
      rows = min(g.R, g.H - r0);
    }
  };

  // cycle accounting of one issuer thread (HONK2_TC_DEBUG=1).  BAR.SYNC blocks lazily, so the layer-barrier
  // wait shows up in the first bucket sampled AFTER the barrier (dbg_bar), not right behind __syncthreads.
  long long dbg_bar = 0, dbg_tempty = 0, dbg_full = 0, dbg_issue = 0, dbg_conv0 = 0, dbg_t = clock64();
  const bool dbg = p.debug != nullptr && blockIdx.x == 0 && threadIdx.x == 32;
  int64_t seq = 0;   // running (utterance, layer) counter: weight buffer = seq & 1
  for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
    // =============================== conv_0 -> P (epilogue warps) ===============================
    if (warp > kTcIssuers) {
      const int et = threadIdx.x - 32 * (1 + kTcIssuers);           // 0 .. 32 * kEpiWarps - 1
      const float* src = p.feat + b * (int64_t)p.T * p.F;
      if (p.ph == 1 && p.pw == 1) {
        // no pooling (res15): 4 consecutive pixels x all channels per item, every weight read feeds 4 FMAs
        const int groups = (p.W + 3) >> 2;
        for (int item = et; item < p.H * groups; item += 32 * kEpiWarps) {
          const int h = item / groups, w0 = (item - h * groups) * 4;
          float pch[3][6];
#pragma unroll
          for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int e = 0; e < 6; ++e) {
              const int hh = h + a - 1, ww = w0 + e - 1;
              pch[a][e] = (hh >= 0 && hh < p.T && ww >= 0 && ww < p.F) ? __ldg(src + (int64_t)hh * p.F + ww) : 0.f;
            }
          for (int pl = 0; pl < NP; ++pl) {
            float a4[4][8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const float* wc9 = s_w0 + (pl * 8 + e) * 12;
              const float4 wa = *reinterpret_cast<const float4*>(wc9);
              const float4 wb = *reinterpret_cast<const float4*>(wc9 + 4);
              const float w8 = wc9[8];
#pragma unroll
              for (int px = 0; px < 4; ++px) {
                float v = pch[0][px] * wa.x;
                v = fmaf(pch[0][px + 1], wa.y, v); v = fmaf(pch[0][px + 2], wa.z, v);
                v = fmaf(pch[1][px], wa.w, v); v = fmaf(pch[1][px + 1], wb.x, v); v = fmaf(pch[1][px + 2], wb.y, v);
                v = fmaf(pch[2][px], wb.z, v); v = fmaf(pch[2][px + 1], wb.w, v); v = fmaf(pch[2][px + 2], w8, v);
                a4[px][e] = fmaxf(v, 0.f);
              }
            }
#pragma unroll
            for (int px = 0; px < 4; ++px) {
              if (w0 + px < p.W) {
                uint4 o;
                __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
                for (int e = 0; e < 4; ++e) ob[e] = __floats2bfloat162_rn(a4[px][2 * e], a4[px][2 * e + 1]);
                uint4* dst = bufP + pl * plane_stride + (int64_t)h * p.W + w0 + px;
                st_hint(dst, o, l2_policy_evict_last());
                if constexpr (SPLIT) {   // lo part: x - float(hi)
                  uint4 o2;
                  __nv_bfloat162* ob2 = reinterpret_cast<__nv_bfloat162*>(&o2);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 fh = __bfloat1622float2(ob[e]);
                    ob2[e] = __floats2bfloat162_rn(a4[px][2 * e] - fh.x, a4[px][2 * e + 1] - fh.y);
                  }
                  st_hint(dst + NP * plane_stride, o2, l2_policy_evict_last());
                }
              }
            }
          }
        }
      } else {
      const float inv = 1.f / (float)(p.ph * p.pw);
      for (int pix = et; pix < p.H * p.W; pix += 32 * kEpiWarps) {
        const int ho = pix / p.W, wo = pix - ho * p.W;
        for (int pl = 0; pl < NP; ++pl) {
          float a8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) a8[e] = 0.f;
          for (int i = 0; i < p.ph; ++i)
            for (int j = 0; j < p.pw; ++j) {
              const int hc = ho * p.ph + i, wc = wo * p.pw + j;   // centre of the 3x3 window
              float xin[9];
#pragma unroll
              for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int e = 0; e < 3; ++e) {
                  const int hh = hc + a - 1, ww = wc + e - 1;
                  xin[a * 3 + e] = (hh >= 0 && hh < p.T && ww >= 0 && ww < p.F) ? __ldg(src + (int64_t)hh * p.F + ww) : 0.f;
                }
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const float* wc9 = s_w0 + (pl * 8 + e) * 12;
                const float4 wa = *reinterpret_cast<const float4*>(wc9);
                const float4 wb = *reinterpret_cast<const float4*>(wc9 + 4);
                float v = xin[0] * wa.x;
                v = fmaf(xin[1], wa.y, v); v = fmaf(xin[2], wa.z, v); v = fmaf(xin[3], wa.w, v);
                v = fmaf(xin[4], wb.x, v); v = fmaf(xin[5], wb.y, v); v = fmaf(xin[6], wb.z, v);
                v = fmaf(xin[7], wb.w, v); v = fmaf(xin[8], wc9[8], v);
                a8[e] += fmaxf(v, 0.f);
              }
            }
          uint4 o;
          __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
          for (int e = 0; e < 4; ++e) ob[e] = __floats2bfloat162_rn(a8[2 * e] * inv, a8[2 * e + 1] * inv);
          bufP[pl * plane_stride + pix] = o;
          if constexpr (SPLIT) {
            uint4 o2;
            __nv_bfloat162* ob2 = reinterpret_cast<__nv_bfloat162*>(&o2);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 fh = __bfloat1622float2(ob[e]);
              ob2[e] = __floats2bfloat162_rn(a8[2 * e] * inv - fh.x, a8[2 * e + 1] * inv - fh.y);
            }
            bufP[(NP + pl) * plane_stride + pix] = o2;
          }
        }
      }
      }
      __threadfence();
      fence_async_all();   // generic-proxy global writes -> visible to the TMA (async proxy) reads of layer 1
    }
    __syncthreads();
    if (dbg) { const long long t = clock64(); dbg_conv0 += t - dbg_t; dbg_t = t; }

    for (int l = 0; l < n_layers; ++l, ++seq) {
      const int cur = (int)(seq & 1);
      const TcLayerDesc& L = s_layer[cur];
      const TcGeom& g = L.g;
      const uint32_t w_smem = smem_u32(smem + p.smem_w_off[cur]);
      const int n_tiles = g.tiles_per_utt;

      if (warp == 0) {
        // ================================ TMA producer ================================
        // prefetch the next step's weights / descriptor / constants into the other buffers
        // (free: the layer that used them finished before the barrier we just passed)
        if constexpr (SPLIT) {
          // one weight buffer: this layer's two weight sets now (every MMA of the previous layer has retired: its
          // epilogue read all accumulators before the barrier we just passed)
          if (lane == 0) {
            mbar_expect_tx(wfull_bar(cur), W_BYTES);
            bulk_load(w_smem, L.wpack, W_BYTES, wfull_bar(cur));
          }
        }
        if (seq + 1 < n_seq) {
          const int nl = (l + 1 < n_layers) ? l + 1 : 0;
          const TcLayerDesc* nd = p.layers + nl;
          if (lane == 0) {
            if constexpr (!SPLIT) {
              mbar_expect_tx(wfull_bar(cur ^ 1), W_BYTES);
              bulk_load(smem_u32(smem + p.smem_w_off[cur ^ 1]), nd->wpack, W_BYTES, wfull_bar(cur ^ 1));
            }
            s_layer[cur ^ 1] = *nd;
          }
          for (int i = lane; i < CP; i += 32) s_kconst[(cur ^ 1) * CP + i] = nd->kconst[i];
        }
        if (lane == 0) {
          const CUtensorMap* map = p.maps + l;
          const uint32_t tx = (uint32_t)(2 * g.n_boxes * g.rows_box * g.Wp * 16);
          for (int tix = 0; tix < n_tiles; ++tix) {
            int ph, r0, rows;
            tile_decode(g, tix, ph, r0, rows);
            if (rows <= 0) continue;
            for (int kc = 0; kc < NA; ++kc) {
              mbar_wait(empty_bar(stage), phase ^ 1);
              mbar_expect_tx(full_bar(stage), tx);
              const uint32_t sbase = smem_u32(s_ring + (size_t)stage * p.ring_slot_bytes);
              for (int half = 0; half < 2; ++half)
                for (int bx = 0; bx < g.n_boxes; ++bx)
                  tma_load_5d_hint(sbase + half * g.slab_bytes + bx * g.box_stride, map, full_bar(stage), 0, -g.dpad,
                                   r0 + g.h_start[bx], ph, (int)blockIdx.x * NPX + 2 * kc + half,
                                   L.in_buf ? l2_policy_evict_first() : l2_policy_evict_last());
              if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      } else if (warp <= kTcIssuers) {
        // ================================ MMA issuers ================================
        const int me = warp - 1;
        constexpr uint32_t idesc = umma_idesc(128, CP);
        constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);
        const uint32_t a_lo_fields = ((uint32_t)(g.slab_bytes >> 4) & 0x3FFFu) << 16;
        const uint32_t b_lo_base = ((w_smem >> 4) & 0x3FFFu) | (((uint32_t)(W_HALF >> 4) & 0x3FFFu) << 16);
        int tap16[9];
#pragma unroll
        for (int dh = 0; dh < 3; ++dh)
#pragma unroll
          for (int dw = 0; dw < 3; ++dw) tap16[dh * 3 + dw] = (g.tap_off[dh] >> 4) + (dw - 1) * g.d;
        const bool side = g.side_taps != 0;
        const int first_tap = side ? 0 : 1;
        const bool leader = elect_one();
        mbar_wait(wfull_bar(cur), (uint32_t)((seq >> 1) & 1));   // this layer's weights have landed
        if (dbg) { const long long t = clock64(); dbg_bar += t - dbg_t; dbg_t = t; }
        for (int tix = 0; tix < n_tiles; ++tix) {
          int ph, r0, rows;
          tile_decode(g, tix, ph, r0, rows);
          if (rows <= 0) continue;
          const int n_mt = (rows * g.Wp + 127) >> 7;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1);
          tc_fence_after();
          if (dbg) { const long long t = clock64(); dbg_tempty += t - dbg_t; dbg_t = t; }
          const uint32_t d_base = tmem_base + acc * kAccCols + me * CP;
#pragma unroll
          for (int kca = 0; kca < NA; ++kca) {
            const int kc = kca < NKC ? kca : kca - NKC;   // weight chunk (SPLIT: stages NKC .. 2 NKC-1 hold the lo parts)
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            if (dbg) { const long long t = clock64(); dbg_full += t - dbg_t; dbg_t = t; }
            if (leader) {
              const uint32_t a_lo_stage =
                  (((smem_u32(s_ring + (size_t)stage * p.ring_slot_bytes) >> 4) + me * 128) & 0x3FFFu) | a_lo_fields;
#pragma unroll
              for (int tap = 0; tap < 9; ++tap) {
                if ((tap % 3) != 1 && !side) continue;
                const uint32_t a_lo = a_lo_stage + (uint32_t)tap16[tap];
                const uint32_t b_lo = b_lo_base + (uint32_t)(((tap * NKC + kc) * 2 * W_HALF) >> 4);
                if (kca == 0 && tap <= 1) {
                  const uint32_t accum = (tap == first_tap) ? 0u : 1u;
#pragma unroll
                  for (int u = 0; u < MAXU; ++u)
                    if (me + u * kTcIssuers < n_mt)
                      umma_f16_lohi_rt(d_base + u * kTcIssuers * CP, a_lo + u * kTcIssuers * 128, b_lo, desc_hi, idesc, accum);
                } else {
#pragma unroll
                  for (int u = 0; u < MAXU; ++u)
                    if (me + u * kTcIssuers < n_mt)
                      umma_f16_lohi<true>(d_base + u * kTcIssuers * CP, a_lo + u * kTcIssuers * 128, b_lo, desc_hi, idesc);
                }
                if constexpr (SPLIT) {
                  if (kca < NKC) {   // hi activations x lo weights (the lo set follows the hi set; no carry: < 256 KB)
#pragma unroll
                    for (int u = 0; u < MAXU; ++u)
                      if (me + u * kTcIssuers < n_mt)
                        umma_f16_lohi<true>(d_base + u * kTcIssuers * CP, a_lo + u * kTcIssuers * 128,
                                            b_lo + (uint32_t)(W_PART >> 4), desc_hi, idesc);
                  }
                }
              }
              umma_commit(empty_bar(stage));
              if (kca == NA - 1) umma_commit(tfull_bar(acc));
            }
            __syncwarp();
            if (dbg) { const long long t = clock64(); dbg_issue += t - dbg_t; dbg_t = t; }
            if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
          }
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        }
      } else {
        // ================================ epilogue (4*NKC warps) ================================
        // warp e: TMEM lane quarter q = warp % 4, channel group j = e / 4 (16 channels = planes 2j, 2j+1)
        const int q = warp & 3;
        const int j = (warp - (1 + kTcIssuers)) >> 2;
        const int hstep = g.phase ? g.d : 1;
        const bool has_skip = L.has_skip != 0, last = L.last != 0;
        const uint4* skip_in = bufP + (int64_t)(2 * j) * plane_stride;          // even layers read AND write P
        uint4* y_out = (has_skip ? bufP : bufQ) + (int64_t)(2 * j) * plane_stride;
        float kc_reg[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) kc_reg[c] = s_kconst[cur * CP + 16 * j + c];
        float psum[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) psum[c] = 0.f;
        for (int tix = 0; tix < n_tiles; ++tix) {
          int ph, r0, rows;
          tile_decode(g, tix, ph, r0, rows);
          if (rows <= 0) continue;
          const int n_mt = (rows * g.Wp + 127) >> 7;
          const int64_t tile_base = (int64_t)(r0 * hstep + ph) * g.W;
          auto locate = [&](int mt, bool& valid) -> int64_t {
            const int pos = mt * 128 + q * 32 + lane;
            const int r = pos / g.Wp;
            const int w = pos - r * g.Wp - g.dpad;
            valid = (w >= 0) && (r < rows) && (mt < n_mt);
            return tile_base + (int64_t)(r * hstep) * g.W + w;
          };
          constexpr int NSK = SPLIT ? 4 : 2;   // skip registers: planes 2j, 2j+1 (SPLIT: and their lo planes)
          auto load_skip = [&](int64_t b0, uint4 (&dst)[NSK]) {
            dst[0] = ld_hint(skip_in + b0, l2_policy_evict_last());
            dst[1] = ld_hint(skip_in + b0 + plane_stride, l2_policy_evict_last());
            if constexpr (SPLIT) {
              dst[2] = ld_hint(skip_in + b0 + NP * plane_stride, l2_policy_evict_last());
              dst[3] = ld_hint(skip_in + b0 + (NP + 1) * plane_stride, l2_policy_evict_last());
            }
          };
          uint4 pv_next[NSK];
          if (has_skip) {
            bool v0;
            const int64_t b0 = locate(0, v0);
            if (v0) load_skip(b0, pv_next);
          }
          mbar_wait(tfull_bar(acc), acc_phase);
          tc_fence_after();
          for (int mt = 0; mt < n_mt; ++mt) {
            bool valid;
            const int64_t base = locate(mt, valid);
            uint4 pv[NSK];
            if (has_skip) {
#pragma unroll
              for (int k = 0; k < NSK; ++k) pv[k] = pv_next[k];
              bool v2;
              const int64_t b2 = locate(mt + 1, v2);
              if (v2) load_skip(b2, pv_next);
            }
            uint32_t v[16];
            tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + acc * kAccCols + mt * CP + 16 * j, v);
            tmem_ld_wait();
            if (valid) {
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                float x[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) x[e] = fmaxf(__uint_as_float(v[8 * hf + e]), 0.f) + kc_reg[8 * hf + e];
                if (has_skip) {
                  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&pv[hf]);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 f = __bfloat1622float2(pb[e]);
                    x[2 * e] += f.x;
                    x[2 * e + 1] += f.y;
                  }
                  if constexpr (SPLIT) {
                    const __nv_bfloat162* pl2 = reinterpret_cast<const __nv_bfloat162*>(&pv[2 + hf]);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                      const float2 f = __bfloat1622float2(pl2[e]);
                      x[2 * e] += f.x;
                      x[2 * e + 1] += f.y;
                    }
                  }
                }
                if (last) {
#pragma unroll
                  for (int e = 0; e < 8; ++e) psum[8 * hf + e] += x[e];
                } else {
                  uint4 yo;
                  __nv_bfloat162* yb = reinterpret_cast<__nv_bfloat162*>(&yo);
#pragma unroll
                  for (int e = 0; e < 4; ++e) yb[e] = __floats2bfloat162_rn(x[2 * e], x[2 * e + 1]);
                  st_hint(y_out + base + hf * plane_stride, yo, has_skip ? l2_policy_evict_last() : l2_policy_evict_first());
                  if constexpr (SPLIT) {   // lo part: x - float(hi)
                    uint4 yl;
                    __nv_bfloat162* lb = reinterpret_cast<__nv_bfloat162*>(&yl);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                      const float2 fh = __bfloat1622float2(yb[e]);
                      lb[e] = __floats2bfloat162_rn(x[2 * e] - fh.x, x[2 * e + 1] - fh.y);
                    }
                    st_hint(y_out + base + (NP + hf) * plane_stride, yl, has_skip ? l2_policy_evict_last() : l2_policy_evict_first());
                  }
                }
              }
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar(acc));
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        }
        if (last) {
          // fused global mean (resnet.py:57-58): warp-reduce the 32 positions; every warp leaves its share in its own
          // slot (no atomics: the logits add the four lane quarters in a fixed order => bit-reproducible)
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            float sum = psum[c];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            if (lane == c) s_pool[q * CP + 16 * j + c] = sum;
          }
        }
        __threadfence();
        fence_async_all();   // this layer's activations -> visible to the next layer's TMA loads
      }
      // keep the non-epilogue roles' accumulator bookkeeping in step (they never touch tfull/tempty state
      // beyond what they advanced themselves: producer has none, issuers advanced per tile above)
      __syncthreads();   // layer boundary: all tiles computed and stored; next descriptor/constants published
    }

    // =============================== logits (resnet.py:59) ===============================
    if (n_layers > 0) {
      for (int lb = threadIdx.x; lb < p.n_labels; lb += kThreads) {
        const float inv = 1.f / (float)(p.H * p.W);
        float v = __ldg(p.out_b + lb);
        // s_pool holds sums of z = x - mean; the BatchNorm output mean is z_mean / sigma (resnet.py:55-58)
        for (int c = 0; c < p.C; ++c) {
          const float pooled = (s_pool[c] + s_pool[CP + c]) + (s_pool[2 * CP + c] + s_pool[3 * CP + c]);
          v = fmaf(pooled * inv * __ldg(p.last_scale + c), __ldg(p.out_w + lb * p.C + c), v);
        }
        p.logits[b * p.n_labels + lb] = v;
      }
      // (s_pool is rewritten by the last layer of the next utterance, many barriers away)
    }
  }

  if (dbg) {
    p.debug[0] = dbg_conv0; p.debug[1] = dbg_bar; p.debug[2] = dbg_tempty; p.debug[3] = dbg_full;
    p.debug[4] = dbg_issue; p.debug[5] = 0; p.debug[6] = n_my;
  }
  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace kws
