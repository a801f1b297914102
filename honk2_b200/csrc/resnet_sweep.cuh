// Column-sweep whole-network kernel of the bf16 tensor-core ResNet path (included by conv_tc.cu).
//
// Why a second formulation.  tools/umma_bench*.cu shows that a 128 x N x 16 tcgen05.mma with both
// operands in shared memory costs max(N/2, 32 + N/4) cycles: the 4 KB activation operand is re-read
// from shared memory (128 B/cycle) by every instruction, so the N = 48 MMAs of the position-major
// kernel (resnet_fused.cuh) run at 44 cycles instead of 24.  Here the three WIDTH taps of the 3x3
// convolution (/root/reference/model/resnet.py:20-26) are stacked on the N axis instead:
//
//   lanes (M = 128)  = 128 consecutive rows h of ONE map column w   ("strip")
//   one MMA          = X[rows + (dh-1) d, w, 16 ch]  x  [ W[dh][+1] | W[dh][0] | W[dh][-1] ]   (N = 3 CP = 144)
//   accumulators     = a ring of CP-column blocks in TMEM, one block per OUTPUT column; the MMA of input
//                      column w writes the three consecutive blocks of output columns w-d, w, w+d
//
// so input column w is read once and feeds all nine taps with 9 MMAs of 72 cycles (the tensor-pipe
// rate) instead of 27 MMAs of 44.  Columns are visited run by run (w = r, r+d, r+2d, ... for every
// residue r mod d), so consecutive steps always shift the accumulator window by exactly one block.
// Every MMA accumulates: the epilogue zeroes a ring block right after reading it.  A window that wraps around the
// ring is issued as two narrower MMAs (N = 96 + 48).
//
// Activation layouts, one slot (buffers P and Q) per CTA, staged by 1-D bulk copies (cp.async.bulk):
//   single-strip maps (H <= 128): [slot][W][K chunk][H][16 ch = 32 B] bf16, so that a column is NA * H * 32 contiguous
//     bytes and lands with ONE copy per step in a stage laid out as [dmax guard rows][NA chunks x H rows][slack], read
//     as a SWIZZLE_32B K-major operand (chunk pitch H rows).  Nothing in the stage is zero: the reference's zero
//     padding (resnet.py:22-24, padding = dilation) is the MMA's disable-output-lane mask instead -- the height tap that
//     reads row h - d leaves lanes 0 .. d-1 alone, the one that reads row h + d lanes H-d .. H-1 (tools/umma_bench6:
//     bit-exact, and free at the pipe rate).  The guard and the slack, and the neighbouring chunk's rows, only ever
//     feed masked lanes: lanes >= H are masked in every MMA too (their results are dropped anyway, and a disabled lane
//     saves tensor-pipe power, which under the power cap is clock);
//   taller maps ("column planar-8"): [slot][NP][W][H][8] bf16; a staged column is [NP planes][rows -d .. 128+d][8 ch]
//     = the K-major SWIZZLE_NONE canonical layout (row pitch 16 B, plane pitch = LBO), one copy per plane of the rows
//     of the strip's window that lie inside the map; rows outside the map are zero rows of the stage.
// The +-d row shift of a height tap is a descriptor start-address offset.
//
// SPLIT (the "bf16x3" precision, single-strip maps): every activation and weight is carried as a bf16 pair hi + lo
// (hi = bf16(v), lo = bf16(v - hi): 16 mantissa bits) -- chunks 0 .. NKC-1 hold the hi parts, NKC .. 2 NKC-1 the lo
// parts -- and each product is three MMAs, hi*hi + lo*hi + hi*lo, accumulated in fp32 in TMEM: the logits agree with
// the fp32 reference arithmetic to ~1e-5 instead of ~3e-3, at a third of the bf16 MMA rate.
//
// conv_0 (1 -> C, resnet.py:18) runs in the same pipeline as a pseudo-layer with ONE 16-channel chunk whose only
// live "channels" are the bf16 high and low parts of the fp32 feature (the weight slab holds w in both positions, so
// the product is fp32-feature x bf16-weight): the producer warp writes the staged column itself instead of copying
// it, three N = 3*CP MMAs per column do the rest, and the ordinary epilogue applies ReLU and stores.  There is no
// CUDA-core convolution and no pipeline drain between utterances.
//
// There is no CTA-wide barrier between layers.  Dependencies are tracked per map column with
// mbarriers: the producer loads column w of layer l+1 as soon as the epilogue has stored column w of
// layer l (col_done), the epilogue of layer l+1 starts storing only after every MMA of layer l has
// retired (layer_done: the two layers ping-pong the same buffers), weights are double buffered.
#pragma once
#include <type_traits>

namespace kws {

// Warp roles: warps 0 .. 4*NKC-1 epilogue (warp % 4 = TMEM lane quarter), then one TMA producer warp and three
// MMA issuer warps.  The front-end warps have the HIGHEST warp ids on purpose: the SM's warp arbiter prefers
// higher ids, and the epilogue warps spend half their time polling barriers; with the issuers at the low ids
// every instruction of the (latency-critical) issue loops waited behind those polls.
constexpr int kSwFrontWarps = 4;
constexpr int kSwIssuers = 3;       // issuer m owns every third step (all MMAs of one input column and its commits)
constexpr int kSwMaxStages = 12;
constexpr int kSwMaxRing = 32;
constexpr int kSwMaxW = 256;
constexpr int kSwTraceLen = 2048;   // steps / blocks recorded by the event trace
constexpr int kSwWeightStep = 12;   // producer step of a layer at which the NEXT layer's weights are requested

// Epilogue warp groups (4 warps = the four TMEM lane quarters each).  A group owns every sw_groups-th output block and handles all
// of its channels; what a group spends per block hardly depends on the channel count (barrier wait, TMEM round trips, skip
// staging, publishing), so the narrow nets (NKC = 1, 2) get three groups too: with two they were epilogue bound (ncu: tensor pipe
// 38 % active, 680 cycles per step against 336 of MMAs).
__host__ __device__ constexpr int sw_groups(int NKC) { return NKC < 3 ? 3 : NKC; }
__host__ __device__ constexpr int sw_epi_warps(int NKC) { return 4 * sw_groups(NKC); }
__host__ __device__ constexpr int sw_threads(int NKC) { return 32 * (kSwFrontWarps + sw_epi_warps(NKC)); }

// control block layout (bytes from the start of dynamic shared memory)
constexpr int kSwBarFull = 0;                                  // [kSwMaxStages]
constexpr int kSwBarEmpty = kSwBarFull + 8 * kSwMaxStages;     // [kSwMaxStages]
constexpr int kSwBarTfull = kSwBarEmpty + 8 * kSwMaxStages;    // [kSwMaxRing]
constexpr int kSwBarTempty = kSwBarTfull + 8 * kSwMaxRing;     // [kSwMaxRing]
constexpr int kSwBarWfull = kSwBarTempty + 8 * kSwMaxRing;     // [2]
constexpr int kSwBarLayer = kSwBarWfull + 16;                  // [2]  all MMAs of a layer retired
constexpr int kSwBarTurn = kSwBarLayer + 16;                   // [kSwIssuers]  the issuers' burst token
constexpr int kSwSkipSlots = 4;     // skip-tensor staging (shared memory): one slot per epilogue warp group (<= 4 groups), [NP][128 rows][8]
constexpr int kSwBarSkFull = kSwBarTurn + 8 * 4;               // [kSwSkipSlots]
constexpr int kSwBarCol = kSwBarSkFull + 8 * kSwSkipSlots;     // [2][kSwMaxW]  column stored by the owning epilogue warps
constexpr int kSwTmemSlot = kSwBarCol + 8 * 2 * kSwMaxW;       // u32
constexpr int kSwKc = round_up(kSwTmemSlot + 4, 128);          // [1 + n_layers][CP] f32 epilogue constants (row 0 = conv_0 = zeros)
constexpr int kSwKcBytes = 6144;
constexpr int kSwPool = kSwKc + kSwKcBytes;                    // [12 epilogue warps][48] f32: every warp's share of the pooled sums
constexpr int kSwCtrlBytes = round_up(kSwPool + 12 * 48 * 4, 1024);
// (epilogue warp group g = warp / 4, one warp per TMEM lane quarter, owns the blocks = g mod sw_groups(NKC))

struct SwParams {
  // Per-layer data is derived from kernel parameters only (constant bank => warp-uniform for the compiler, which
  // keeps the MMA issue loop on the uniform datapath): layer l (0-based) has dilation 2^(l/3) or 1
  // (resnet.py:21), reads Q and adds the skip tensor iff l is odd (resnet.py:51-53), and its packed weights /
  // epilogue constants sit at a fixed stride.
  const unsigned char* wpack0;  // layer 0 weights, [NKC][3 dh][2 K halves][3 blocks][CP][8] bf16; block k = width tap dw = 2 - k
                                //   (SPLIT: the hi parts in that layout, followed by the lo parts in the same layout)
  const unsigned char* kconst0; // layer 0 epilogue constants, [CP] f32 (see pad_bn_kernel)
  int64_t layer_stride;         // bytes between consecutive layers in both arrays
  int use_dilation;
  const float* feat;            // [B][T][F]
  const unsigned char* conv0_wb; // conv_0 weights as a one-chunk sweep slab set: [3 dh][2 K halves][3 blocks][CP][8] bf16
                                //   (k = 0, 1: bf16(w) against the feature's hi and lo parts; SPLIT: k = 2 holds w - bf16(w)
                                //   against a second copy of the feature's hi part)
  const float* last_scale;      // [CP]
  const float* out_w;           // [n_labels][C]
  const float* out_b;           // [n_labels]
  float* logits;                // [B][n_labels]
  __nv_bfloat16* P;             // [n_slots][NP][W][H][8]
  __nv_bfloat16* Q;
  int64_t B;
  int n_layers, C, n_labels, T, F, H, W;   // (no pooling on this path: H = T, W = F)
  int n_strips;                 // ceil(H / 128)
  int smem_c0w_off;             // conv_0 weight slabs (3 * 2 * 3*CP*16 bytes), resident for the whole kernel
  int smem_w_off[2], smem_ring_off, ring_slot_bytes, n_stages;
  int smem_skip_off;            // skip staging: one slot of NP * 2048 bytes per epilogue warp group (unused by SPLIT)
  int ring_slack_bytes;         // bytes behind the last stage that its lanes past the map read (planar: zeroed)
  int chunk_rows;               // planar: rows per plane of a staged column (a multiple of 8): data row h of the strip sits at
                                //   slot row dmax + h, the pad rows above and below are zero (zeroed once, and re-zeroed by
                                //   the producer for the strips that touch the map's top / bottom), 128 + 2 dmax.  (k32: the
                                //   chunk pitch is H)
  int dmax;                     // largest dilation of the network = the guard rows in front of a k32 stage's first chunk
  int discard_q;                // 1 = Q columns are discarded from L2 (no write-back) once the layer that reads them has consumed
                                //     them (single-strip maps, so the 32-byte-row layout only)
  long long* debug;             // optional cycle counters of CTA 0 (HONK2_TC_DEBUG=1)
  long long* trace;             // optional [8][kSwTraceLen] event timestamps of CTA 0 (HONK2_TC_TRACE=1, needs DEBUG)
  // Packed strips (short maps: res8 / res26 after pooling, short clips): `pack_n` utterances share ONE strip, stacked along
  // the rows with `pack_pitch - pack_h` >= dmax zero rows between them (never stored: they are the zero padding of both
  // neighbours).  H is then the stacked height, B counts GROUPS of pack_n utterances, and conv_0 (+ ReLU + AvgPool,
  // resnet.py:40-44) has been computed by conv0_pool_pack_kernel into `ext_in`, which the first layer reads instead of P
  // and the second layer adds as its skip tensor.
  const uint4* ext_in;          // [groups][W][NA chunks][H][32 B] (nullptr: conv_0 runs in this kernel as a pseudo-layer)
  int64_t ext_stride;           // 16-byte units per group
  int pack_n, pack_h, pack_pitch;
  int smem_pool_off;            // pack_n > 1: [pack_n][epilogue warps][CP] f32 pooled sums
  int64_t B_utt;                // utterances (packed mode: the last group may be partly empty)
};

// K32: the 32-byte-row layout of single-strip maps (above), else the planar one.  The two 16-byte halves of row h of
// chunk kc are stored swapped where ((dmax + kc H + h) >> 2) & 1, i.e. exactly as the linear copy must land them in the
// stage (stages are 256-byte aligned: the swizzle works on absolute addresses).
template <int NKC, bool DBG, bool K32, bool SPLIT, bool PACK>
__global__ void __launch_bounds__(sw_threads(NKC), 1)
resnet_tc_sweep_kernel(const SwParams p) {
  static_assert(K32 || !PACK, "packed strips are built on the 32-byte-row layout");
  static_assert(K32 || !SPLIT, "the split-bf16 mode is built on the 32-byte-row layout");
  constexpr int NA = SPLIT ? 2 * NKC : NKC;            // activation chunks staged per column (SPLIT: hi chunks, then lo chunks)
  constexpr int kEpiWarps = sw_epi_warps(NKC);
  constexpr int NG = sw_groups(NKC);
  constexpr int kEpiThreads = 32 * kEpiWarps;
  constexpr int CP = 16 * NKC;
  constexpr int NP = 2 * NKC;
  constexpr int NB = (512 / CP) < kSwMaxRing ? (512 / CP) : kSwMaxRing;   // accumulator ring, in blocks of CP columns
  constexpr int BLK_BYTES = CP * 16;                   // one [CP][8] weight block
  constexpr int W_LBO = 3 * BLK_BYTES;                 // distance between the two K halves of a weight slab
  constexpr int W_SLAB = 2 * W_LBO;                    // one (kc, dh) slab
  constexpr int W_PART = NKC * 3 * W_SLAB;             // one set of slabs (SPLIT: the lo set follows the hi set)
  constexpr int W_BYTES = (SPLIT ? 2 : 1) * W_PART;
  extern __shared__ __align__(1024) unsigned char smem[];

  const uint32_t sbase = smem_u32(smem);
  auto full_bar = [&](int s) { return sbase + kSwBarFull + 8u * s; };
  auto empty_bar = [&](int s) { return sbase + kSwBarEmpty + 8u * s; };
  auto tfull_bar = [&](int a) { return sbase + kSwBarTfull + 8u * a; };
  auto tempty_bar = [&](int a) { return sbase + kSwBarTempty + 8u * a; };
  auto wfull_bar = [&](int i) { return sbase + kSwBarWfull + 8u * i; };
  auto layer_bar = [&](int i) { return sbase + kSwBarLayer + 8u * i; };
  auto turn_bar = [&](int i) { return sbase + kSwBarTurn + 8u * i; };
  auto skfull_bar = [&](int i) { return sbase + kSwBarSkFull + 8u * i; };
  constexpr uint32_t SKIP_SLOT = NP * 128 * 16;   // bytes
  auto col_bar = [&](int par, int w) { return sbase + kSwBarCol + 8u * (par * kSwMaxW + w); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kSwTmemSlot);
  float* s_pool = reinterpret_cast<float*>(smem + (PACK ? p.smem_pool_off : kSwPool));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_layers = p.n_layers, H = p.H, W = p.W, n_strips = p.n_strips;
  const int64_t n_my = (p.B - blockIdx.x + gridDim.x - 1) / gridDim.x;
  const int64_t n_wq = n_my * n_layers;        // real (C -> C) layers this CTA runs
  const int64_t n_seq = n_wq;
  const int nl1 = n_layers + 1;                 // pseudo-layers per utterance: conv_0, then the C -> C layers
  constexpr bool ext = PACK;                    // conv_0 came from conv0_pool_pack_kernel: no conv_0 pseudo-layer here
  constexpr int ll0 = ext ? 1 : 0;

  // Activation layout in HBM (16-byte units = 8 bf16 channels of one position), one slot per CTA:
  //   k32     [w][K chunk][h][2]      (single-strip maps; SPLIT: 2 NKC chunks, the lo parts after the hi parts)
  //   planar  [plane][w][h]           (multi-strip maps)
  constexpr bool k32 = K32;   // (compile time: the two layouts' address arithmetic would not fit the epilogue's registers together)
  const int kc_stride = H * 2;                     // k32: 16-byte units between K chunks
  const int64_t col_stride = (int64_t)NA * H * 2;  // k32: 16-byte units between columns
  const int64_t plane_stride = (int64_t)W * H;    // planar: 16-byte units between planes
  const int64_t slot_base = (int64_t)blockIdx.x * ((int64_t)(SPLIT ? 2 : 1) * NP * W * H);   // this CTA's utterance slot
  uint4* bufP = reinterpret_cast<uint4*>(p.P) + slot_base;
  uint4* bufQ = reinterpret_cast<uint4*>(p.Q) + slot_base;

  // ---- one-time setup
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.n_stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < NB; ++a) { mbar_init(tfull_bar(a), kSwIssuers); mbar_init(tempty_bar(a), 4); }
    for (int i = 0; i < 2; ++i) { mbar_init(wfull_bar(i), 1); mbar_init(layer_bar(i), kSwIssuers); }
    for (int i = 0; i < kSwIssuers; ++i) mbar_init(turn_bar(i), 1);
    for (int i = 0; i < kSwSkipSlots; ++i) mbar_init(skfull_bar(i), 1);
    for (int par = 0; par < 2; ++par)
      for (int w = 0; w < W; ++w) mbar_init(col_bar(par, w), (uint32_t)(4 * n_strips));
    fence_barrier_init();
    mbar_arrive(turn_bar(0));   // issuer 0 holds the burst token first
  }
  if (warp == kEpiWarps + 1) tmem_alloc(smem_u32(tmem_slot), 512);
  {   // conv_0 weight slabs -> shared memory (generic copy; the fence below publishes it to the tensor core)
    const uint4* src = reinterpret_cast<const uint4*>(p.conv0_wb);
    uint4* dst = reinterpret_cast<uint4*>(smem + p.smem_c0w_off);
    for (int i = threadIdx.x; i < (3 * W_SLAB) / 16; i += sw_threads(NKC)) dst[i] = src[i];
  }
  {   // epilogue constants of every pseudo-layer, read from shared memory at use
      // (the host plan guarantees (1 + n_layers) * CP * 4 <= kSwKcBytes)
    float* s_kc = reinterpret_cast<float*>(smem + kSwKc);
    for (int i = threadIdx.x; i < nl1 * CP; i += sw_threads(NKC)) {
      const int ll = i / CP, c = i - ll * CP;
      s_kc[i] = ll == 0 ? 0.f : reinterpret_cast<const float*>(p.kconst0 + (ll - 1) * p.layer_stride)[c];
    }
  }
  if constexpr (!K32) {
    // planar: the pad rows above and below the map are never written again and supply the zero padding
    uint4* ring = reinterpret_cast<uint4*>(smem + p.smem_ring_off);
    const int n16 = (p.n_stages * p.ring_slot_bytes + p.ring_slack_bytes) >> 4;
    for (int i = threadIdx.x; i < n16; i += sw_threads(NKC)) ring[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  fence_async_smem();   // generic-proxy writes (conv_0 weights, planar zeros) -> visible to the tensor core's (async proxy) reads
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Every MMA accumulates (three issuer warps feed the same accumulators, in no particular order), so the ring
  // starts zeroed and the epilogue re-zeroes each block right after reading it.
  if (warp < kEpiWarps) {
    const int q = warp & 3, j = warp >> 2;
    if (j < NKC)   // (the narrow nets have more warp groups than 16-column chunks)
      for (int a = 0; a < NB; ++a) tmem_st16_zero(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * CP + 16 * j));
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // L2 policies: P (read as the odd layers' input and as the skip tensor, rewritten in place) evict_last, Q (written once,
  // read once) evict_first.  Each is created where it is used: one instruction, and no register pair held for the
  // whole kernel.

  auto layer_dil = [&](int l) { return p.use_dilation ? (1 << (l / 3)) : 1; };
  // rows per plane / chunk of a staged column = its pitch in shared memory (a multiple of 8 rows)
  const int box_rows = p.chunk_rows;
  // slot row that the height tap dh = 0 of output row 0 reads
  auto row0_of = [&](int d) { return p.dmax - d; };

  if (warp == kEpiWarps) {
    // ========================================= TMA producer =========================================
    // The whole warp walks the (warp-uniform) schedule; one elected lane issues the copies.
    const bool leader = elect_one();
    if (n_seq > 0) {
      int stage = 0;
      uint32_t sphase = 0;
      int64_t sq = 0;      // pseudo-layer counter (conv_0 included): parity of the layer / column barriers
      int64_t wq = 0;      // real-layer counter: parity of the weight buffers
      const bool pdbg = DBG && p.debug != nullptr && blockIdx.x == 0;
      const bool ptrace = DBG && p.trace != nullptr && blockIdx.x == 0;
      int pstep = 0;
      long long pd_col = 0, pd_empty = 0, pd_c0 = 0, pd_issue = 0, pd_t = DBG ? clock64() : 0;
      auto pstamp = [&](long long& bucket) {
        if constexpr (DBG) { if (pdbg) { const long long t = clock64(); bucket += t - pd_t; pd_t = t; } }
      };
      if (leader) {
        mbar_expect_tx(wfull_bar(0), W_BYTES);
        bulk_load(sbase + p.smem_w_off[0], p.wpack0, W_BYTES, wfull_bar(0));
      }
      for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
        const float* feat_b = p.feat + b * (int64_t)p.T * p.F;
        const uint4* ext_b = ext ? p.ext_in + b * p.ext_stride : nullptr;
        const bool c0_vec = (p.F & 3) == 0 && (reinterpret_cast<uintptr_t>(p.feat) & 15) == 0;
        for (int ll = ll0; ll < nl1; ++ll, ++sq) {
          const bool is_c0 = ll == 0;
          const int l = ll - 1;
          const int d = is_c0 ? 1 : layer_dil(l);
          const int n_runs = d < W ? d : W;
          const bool in_q = !is_c0 && (l & 1) != 0;
          const uint64_t pol = in_q ? l2_policy_evict_first() : l2_policy_evict_last();
          bool w_pending = !is_c0 && wq + 1 < n_wq;
          auto request_weights = [&]() {
            if constexpr (SPLIT) {
              // ONE weight buffer (hi + lo slabs of a layer are 2 x 41 KB): the next layer's weights can only be
              // requested when every MMA of THIS layer has retired -- a short bubble per layer, in a mode whose steps
              // are three times as long
              mbar_wait(layer_bar((int)(sq & 1)), (uint32_t)((sq >> 1) & 1));
            } else if (wq >= 1) {
              // buffer (wq+1)&1 was read by the MMAs of the previous real layer: wait until they have retired
              // (that layer is the previous pseudo-layer, or the one before conv_0 when this is the utterance's first)
              const int64_t sp = (l >= 1 || ext) ? sq - 1 : sq - 2;
              mbar_wait(layer_bar((int)(sp & 1)), (uint32_t)((sp >> 1) & 1));
            }
            const int nl = (l + 1 < n_layers) ? l + 1 : 0;
            const int nb = (int)((wq + 1) & 1);
            if (leader) {
              mbar_expect_tx(wfull_bar(nb), W_BYTES);
              bulk_load(sbase + p.smem_w_off[nb], p.wpack0 + nl * p.layer_stride, W_BYTES, wfull_bar(nb));
            }
            w_pending = false;
          };
          const int prev_par = (int)((sq - 1) & 1);
          const uint32_t prev_phase = (uint32_t)(((sq - 1) >> 1) & 1);
          if (is_c0) {
            // conv_0 pseudo-layer: the producer BUILDS the staged columns.  Rows 128 s - 1 .. 128 s + 128 of feature
            // column w (k32: rows 0 .. H-1), each as {hi, lo, 0 x 6} bf16 (fp32 feature split into two bf16 parts) in
            // plane 0; the MMA's second K half reads the same plane (LBO = 0) against zero weights, so nothing an earlier
            // layer left in the slot can reach this utterance.  Zero outside the map = the reference's padding.  Up to four
            // consecutive columns are built per pass from one 16-byte feature load per row: the MMAs of a conv_0 step
            // are few, so this warp's instruction count is what bounds the pseudo-layer.
            const int r0 = row0_of(1);
            // the NEXT utterance's features into L2 now, a whole utterance period before they are needed: the column
            // builder's loads otherwise wait for DRAM once per pass
            if (b + gridDim.x < p.B) {
              const char* nf = reinterpret_cast<const char*>(p.feat + (b + gridDim.x) * (int64_t)p.T * p.F);
              const int n_lines = (p.T * p.F * 4 + 127) >> 7;
              for (int i = lane; i < n_lines; i += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(nf + (size_t)i * 128));
            }
            for (int s = 0; s < n_strips; ++s)
              for (int w0 = 0; w0 < W; w0 += 4) {
                const int cnt = c0_vec ? (W - w0 < 4 ? W - w0 : 4) : 1;
                for (int w = w0; w < (W < w0 + 4 ? W : w0 + 4); w += cnt) {
                  pstamp(pd_issue);
                  // the stages of these `cnt` steps
                  int st[4]; uint32_t ph[4];
                  { int t = stage; uint32_t q2 = sphase;
#pragma unroll
                    for (int c = 0; c < 4; ++c) { st[c] = t; ph[c] = q2; if (++t == p.n_stages) { t = 0; q2 ^= 1u; } } }
#pragma unroll
                  for (int c = 0; c < 4; ++c) if (c < cnt) mbar_wait_lean(empty_bar(st[c]), ph[c] ^ 1u);
                  pstamp(pd_empty);
                  float4 fr[5];
#pragma unroll
                  for (int k = 0; k < 5; ++k) {   // all loads first
                    const int rr = lane + 32 * k;
                    const int h = s * 128 - 1 + rr;
                    fr[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (rr < 130 && h >= 0 && h < p.T) {
                      if (c0_vec) fr[k] = __ldg(reinterpret_cast<const float4*>(feat_b + (int64_t)h * p.F + w));
                      else fr[k].x = __ldg(feat_b + (int64_t)h * p.F + w);
                    }
                  }
                  pstamp(pd_col);   // (debug accounting: the feature-load latency is booked under "previous layer's column")
#pragma unroll
                  for (int k = 0; k < 5; ++k) {
                    const int rr = lane + 32 * k;
                    // k32: the map's rows only (the lane masks are the padding; a row past the map could be the next stage's)
                    if (k32 ? (rr >= 1 && rr <= H) : (rr < 130 && r0 + rr < box_rows)) {
                      const float4 f = fr[k];
                      const float fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
                      for (int c = 0; c < 4; ++c) {
                        if (c < cnt) {
                          const __nv_bfloat16 hi = __float2bfloat16_rn(fv[c]);
                          const __nv_bfloat16 lo = __float2bfloat16_rn(fv[c] - __bfloat162float(hi));
                          const uint32_t hilo = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(lo) << 16);
                          // SPLIT: channel 2 carries the hi part again, against the lo part of the weight
                          const uint32_t hi2 = SPLIT ? (uint32_t)__bfloat16_as_ushort(hi) : 0u;
                          unsigned char* slot = smem + p.smem_ring_off + (size_t)st[c] * p.ring_slot_bytes;
                          if (k32) {   // 32-byte rows: channels 0-7 in the (swizzled) first half, zeros in the other
                            const int row = r0 + rr, sw = (row >> 2) & 1;
                            *reinterpret_cast<uint4*>(slot + (size_t)row * 32 + (sw << 4)) = make_uint4(hilo, hi2, 0u, 0u);
                            *reinterpret_cast<uint4*>(slot + (size_t)row * 32 + ((sw ^ 1) << 4)) = make_uint4(0u, 0u, 0u, 0u);
                          } else
                          *reinterpret_cast<uint4*>(slot + (size_t)(r0 + rr) * 16) = make_uint4(hilo, 0u, 0u, 0u);
                        }
                      }
                    }
                  }
                  fence_async_smem();   // generic-proxy writes -> visible to the tensor core
                  __syncwarp();
                  if (leader) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) if (c < cnt) mbar_arrive(full_bar(st[c]));
                  }
                  for (int c = 0; c < cnt; ++c) {
                    if constexpr (DBG) {
                      if (ptrace && leader && pstep < kSwTraceLen) p.trace[0 * kSwTraceLen + pstep] = clock64();
                      ++pstep;
                    }
                    if (++stage == p.n_stages) { stage = 0; sphase ^= 1; }
                  }
                  pstamp(pd_c0);
                }
              }
            continue;   // (conv_0 has no weights to request and does not advance the real-layer counter)
          }
          int step = 0;
          for (int s = 0; s < n_strips; ++s)
            for (int r = 0; r < n_runs; ++r)
              for (int w = r; w < W; w += d, ++step) {
                if (!SPLIT && w_pending && step == kSwWeightStep) request_weights();
                pstamp(pd_issue);
                if (!is_c0 && !(ext && l == 0)) mbar_wait_lean(col_bar(prev_par, w), prev_phase);   // column w of the previous pseudo-layer is stored
                pstamp(pd_col);
                mbar_wait_lean(empty_bar(stage), sphase ^ 1);
                pstamp(pd_empty);
                const uint32_t dst = sbase + p.smem_ring_off + (uint32_t)stage * p.ring_slot_bytes;
                if (k32) {
                  // the whole column, NA chunks x H rows x 32 B (SPLIT: hi chunks, then lo chunks), behind the guard rows
                  if (leader) {
                    const uint32_t bytes = (uint32_t)(NA * H) * 32u;
                    mbar_expect_tx(full_bar(stage), bytes);
                    const uint4* src = ((ext && l == 0) ? ext_b : in_q ? bufQ : bufP) + (int64_t)w * col_stride;
                    bulk_load_hint(dst + (uint32_t)p.dmax * 32u, src, bytes, full_bar(stage), pol);
                  }
                } else {
                  // one contiguous H x 16 B run per 8-channel plane (a TMA box with 16-byte rows fetches a whole
                  // 32-byte sector per row: 2.6x the bytes, measured with ncu)
                  // (issued by ONE lane with warp-uniform operands: per-lane operands would make the compiler wrap every
                  // copy in a 15-instruction ELECT / R2UR loop, and this warp's instruction count is what bounds it)
                  const int win_lo = s * 128 - d, win_hi = s * 128 + 128 + d;         // rows the MMAs of this strip read
                  const int h_lo = win_lo > 0 ? win_lo : 0, h_hi = win_hi < H ? win_hi : H;
                  if (n_strips > 1 && (win_lo < 0 || win_hi > H)) {
                    // this slot last held an interior strip (data in every row): restore the zero rows of the padding
                    unsigned char* slot = smem + p.smem_ring_off + (size_t)stage * p.ring_slot_bytes;
                    const int top = win_lo < 0 ? -win_lo : 0;                       // rows above the map
                    const int bot = win_hi > H ? win_hi - H : 0;                    // rows below the map
                    const int r_top = p.dmax - d, r_bot = p.dmax + H - s * 128;     // their first slot rows
                    for (int i = lane; i < NP * (top + bot); i += 32) {
                      const int pl = i / (top + bot), k = i - pl * (top + bot);
                      const int row = k < top ? r_top + k : r_bot + (k - top);
                      *reinterpret_cast<uint4*>(slot + (size_t)(pl * box_rows + row) * 16) = make_uint4(0u, 0u, 0u, 0u);
                    }
                    fence_async_smem();
                    __syncwarp();
                  }
                  const uint32_t bytes = (uint32_t)(h_hi - h_lo) * 16u;
                  if (leader) {
                    mbar_expect_tx(full_bar(stage), bytes * NP);
                    const uint4* src = (in_q ? bufQ : bufP) + (int64_t)w * H + h_lo;
                    const uint32_t d0 = dst + (uint32_t)(p.dmax + h_lo - s * 128) * 16u;
#pragma unroll
                    for (int pl = 0; pl < NP; ++pl)
                      bulk_load_hint(d0 + (uint32_t)(pl * box_rows) * 16u, src + (int64_t)pl * plane_stride, bytes, full_bar(stage), pol);
                  }
                }
                if constexpr (DBG) {
                  if (ptrace && leader && pstep < kSwTraceLen) p.trace[0 * kSwTraceLen + pstep] = clock64();
                  ++pstep;
                }
                if (++stage == p.n_stages) { stage = 0; sphase ^= 1; }
              }
          if (w_pending) request_weights();
          if (!is_c0) ++wq;
        }
      }
      if constexpr (DBG) {
        if (pdbg && leader) { p.debug[13] = pd_col; p.debug[14] = pd_empty; p.debug[15] = pd_c0; p.debug[7] = pd_issue; }
      }
    }
    __syncwarp();
  } else if (warp > kEpiWarps) {
    // ========================================= MMA issuers (3 warps) =========================================
    // Issuer m owns every third STEP: it waits for the step's staged column and for the ring slots of the step's
    // window, issues the 3*NKC MMAs of the step (twice as many, half as wide, when the window wraps around the
    // ring) and commits; for the other two steps it only advances its counters.  While one issuer is inside its
    // burst the next one has already prepared its operands and queues right behind it.  All MMAs accumulate (the
    // ring blocks are zeroed by the epilogue), so the order in which the three warps' MMAs reach the tensor pipe
    // does not matter (tools/umma_bench2/4: concurrent accumulation from several warps into one accumulator is
    // exact and runs at the pipe rate).
    //
    // What limits this role is the INSTRUCTION COUNT of its single worker lane (ncu: ~5 cycles per instruction in
    // this branchy scalar code, the MMA instructions themselves are 3 % of its time), so the step is kept lean: ring
    // slots advance by increments (no divisions), the cycle accounting is compiled out unless DBG, barrier polls use
    // the hardware suspend hint, and the MMA burst is straight-line code without predicated-off instructions.
    //
    // An output block receives MMAs from the steps of its three neighbouring input columns, i.e. from all three
    // issuers: tfull counts three arrivals (each issuer commits on every block of its window; the run's first and
    // last block, which have only two contributing steps, get a plain arrival from the issuer of the edge step),
    // and every issuer waits for the ring slot of every block of its window to be drained, not only the fresh one,
    // because nothing orders the issuers among themselves.
    const int me = warp - kEpiWarps - 1;
    // Whole warp walks the schedule with warp-uniform values only (kernel parameters, counters, the TMEM base
    // broadcast by a shuffle), so the descriptors live in uniform registers and an MMA costs 2-3 instructions
    // instead of the 17-instruction ELECT / R2UR / branch sequence the compiler emits for per-thread operands;
    // one elected lane issues the MMAs, commits and arrivals.
    const bool leader = elect_one();
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    if (n_seq > 0) {
      int stage = 0;
      uint32_t sphase = 0;
      int owner = 0;            // issuer of the current step (global step counter mod 3)
      uint32_t turn_par = 0;    // parity of this issuer's next token
      int sl = 0;               // ring slot of the output block of the CURRENT step's own column
      uint32_t pr = 0;          // use parity of that slot
      constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);   // SBO = 128 B, descriptor version 1
      constexpr uint32_t idesc0 = umma_idesc(128, 0);
      constexpr uint32_t idesc_blk = (uint32_t)(CP >> 3) << 17;   // one more block of CP columns
      constexpr uint32_t b_lbo = ((uint32_t)(W_LBO >> 4) & 0x3FFFu) << 16;
      constexpr uint32_t blk16 = BLK_BYTES >> 4;
      long long dbg_full = 0, dbg_tempty = 0, dbg_issue = 0, dbg_w = 0, dbg_utt = 0, dbg_other = 0, dbg_t = DBG ? clock64() : 0;
      const bool dbg = DBG && p.debug != nullptr && blockIdx.x == 0 && me == 0;
      const bool itrace = DBG && p.trace != nullptr && blockIdx.x == 0;
      int gstep = 0;
      auto tr = [&](int row) {
        if constexpr (DBG) { if (itrace && leader && gstep < kSwTraceLen) p.trace[row * kSwTraceLen + gstep] = clock64(); }
      };
      auto stamp = [&](long long& bucket) {
        if constexpr (DBG) { if (dbg) { const long long t = clock64(); bucket += t - dbg_t; dbg_t = t; } }
      };
      int64_t sq = 0, wq = 0;   // pseudo-layer / real-layer counters (see the producer)
      for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
        for (int ll = ll0; ll < nl1; ++ll, ++sq) {
          const bool is_c0 = ll == 0;
          const int l = ll - 1;
          const int d = is_c0 ? 1 : layer_dil(l);
          const int n_runs = d < W ? d : W;
          const int cur = (int)(sq & 1);
          const uint32_t plane16 = (uint32_t)box_rows;                       // plane pitch in 16-byte units
          // (conv_0: both K halves read plane 0, the weights of the second half are zero)
          const uint32_t a_lbo = k32 ? (1u << 16) : is_c0 ? 0u : (plane16 & 0x3FFFu) << 16;
          // A descriptor high word: SWIZZLE_NONE, SBO = 128 B -- or SWIZZLE_32B (layout type 6), SBO = 256 B per 8 rows
          // (the swizzle is applied to absolute shared-memory addresses, so any row offset works: tools/umma_bench5)
          const uint32_t a_hi = k32 ? ((256u >> 4) | (1u << 14) | (6u << 29)) : desc_hi;
          const uint32_t row_mul = k32 ? 2u : 1u;                                    // 16-byte units per row
          const uint32_t kc_step = k32 ? (uint32_t)H * 2u : 2u * plane16;            // 16-byte units per K chunk
          const uint32_t w16 = ((sbase + (is_c0 ? p.smem_c0w_off : p.smem_w_off[wq & 1])) >> 4);
          const uint32_t row0 = (uint32_t)row0_of(d);
          // SPLIT: the lo chunks of the staged column follow the NKC hi chunks, the lo slabs follow the hi slabs
          const uint32_t a_lo_off = (uint32_t)NKC * kc_step;
          constexpr uint32_t b_lo_off = (uint32_t)(W_PART >> 4);
          // k32: the zero padding of the map's edge rows.  The tap dh = 0 reads row h - d: lanes 0 .. d-1 get nothing;
          // dh = 2 reads row h + d: lanes H-d .. H-1 get nothing.  Every tap also leaves the lanes past the map
          // (>= H, results never used) alone: the tensor pipe then draws less power, and under the power cap that is
          // clock (res15: 27 of 128 lanes, +3 % end to end on its own, NVIDIA B200 at 1000 W).
          auto lane_bits = [](int lo, int hi, int j) {   // word j of the mask of lanes lo .. hi-1
            const int a = min(max(lo - 32 * j, 0), 32), b = min(max(hi - 32 * j, 0), 32);
            return (b >= 32 ? ~0u : (1u << b) - 1u) & ~(a >= 32 ? ~0u : (1u << a) - 1u);
          };
          const uint4 m_ge = make_uint4(lane_bits(H, 128, 0), lane_bits(H, 128, 1), lane_bits(H, 128, 2), lane_bits(H, 128, 3));
          const uint4 m_top = make_uint4(lane_bits(0, d, 0) | m_ge.x, lane_bits(0, d, 1) | m_ge.y, lane_bits(0, d, 2) | m_ge.z, lane_bits(0, d, 3) | m_ge.w);
          const uint4 m_bot = make_uint4(lane_bits(H - d, 128, 0), lane_bits(H - d, 128, 1), lane_bits(H - d, 128, 2), lane_bits(H - d, 128, 3));
          // one MMA of height tap dh (compile-time after unrolling)
          auto mma = [&](int dh, uint32_t dt, uint32_t a, uint32_t b, uint32_t id) {
            if (k32) umma_f16_lohi2_mask(dt, a, a_hi, b, desc_hi, id, dh == 0 ? m_top : dh == 1 ? m_ge : m_bot);
            else umma_f16_lohi2<true>(dt, a, a_hi, b, desc_hi, id);
          };
          stamp(dbg_other);
          if (!is_c0) mbar_wait_lean(wfull_bar((int)(wq & 1)), (uint32_t)((wq >> 1) & 1));
          stamp(dbg_w);
          for (int s = 0; s < n_strips; ++s)
            for (int r = 0; r < n_runs; ++r) {
              const int Lr = (W - r + d - 1) / d;   // output columns of this run
              for (int i = 0; i < Lr; ++i) {
                if (owner == me) {
                  // window = output blocks of columns i-1 (if any), i, i+1 (if any): n blocks, ring-contiguous from p0
                  const bool lo = i > 0, hi_ = i + 1 < Lr;
                  const int s_lo = sl > 0 ? sl - 1 : NB - 1, s_hi = sl + 1 < NB ? sl + 1 : 0;
                  const uint32_t par_lo = pr ^ (sl == 0 ? 1u : 0u), par_hi = pr ^ (sl + 1 == NB ? 1u : 0u);
                  const int p0 = lo ? s_lo : sl;
                  const int n = 1 + (lo ? 1 : 0) + (hi_ ? 1 : 0);
                  const int wrap_at = NB - p0 < n ? NB - p0 : n;              // blocks before the ring wraps
                  const int blk0 = lo ? 0 : 1;                                 // weight block of the first window block
                  stamp(dbg_other);
                  tr(1);
                  // the epilogue must have drained and re-zeroed the previous use of every slot of the window
                  if (lo) mbar_wait_lean(tempty_bar(s_lo), par_lo ^ 1u);
                  mbar_wait_lean(tempty_bar(sl), pr ^ 1u);
                  if (hi_) mbar_wait_lean(tempty_bar(s_hi), par_hi ^ 1u);
                  stamp(dbg_tempty);
                  tr(2);
                  mbar_wait_lean(full_bar(stage), sphase);
                  tc_fence_after();
                  tr(3);
                  if constexpr (DBG) { if (is_c0 && s == 0 && r == 0 && i < kSwIssuers) stamp(dbg_utt); else stamp(dbg_full); }
                  // All operands of the step are computed BEFORE the burst, and the burst is straight-line code
                  // without predicated-off MMAs (separate path for the wrapped window).
                  const uint32_t a16 = ((sbase + p.smem_ring_off + (uint32_t)stage * p.ring_slot_bytes) >> 4) + row0 * row_mul;
                  const uint32_t d1 = tmem_u + (uint32_t)(p0 * CP);
                  const uint32_t id1 = idesc0 + (uint32_t)wrap_at * idesc_blk;
                  uint32_t al[3 * NKC], bl[3 * NKC];
#pragma unroll
                  for (int kc = 0; kc < NKC; ++kc)
#pragma unroll
                    for (int dh = 0; dh < 3; ++dh) {
                      al[kc * 3 + dh] = ((a16 + (uint32_t)kc * kc_step + (uint32_t)(dh * d) * row_mul) & 0x3FFFu) | a_lbo;
                      bl[kc * 3 + dh] = ((w16 + (uint32_t)(((kc * 3 + dh) * W_SLAB) >> 4) + (uint32_t)blk0 * blk16) & 0x3FFFu) | b_lbo;
                    }
                  // The burst token: bursts are issued one issuer at a time, in step order.  Without it the three
                  // issuers' bursts interleave MMA by MMA in the (blocking, shallow) issue queue, all three finish
                  // together, then all three do their commits / bookkeeping / operand preparation at the same time and
                  // the tensor pipe idles ~600 cycles per round (event trace).  With it, everything above this line
                  // and the commits below overlap the other two issuers' bursts.
                  mbar_wait_lean(turn_bar(me), turn_par);
                  turn_par ^= 1u;
                  if (!leader) {
                    // (only the elected lane issues)
                  } else if (is_c0) {
                    // conv_0: one 16-channel chunk (k = 0 .. 2 are its three height taps)
                    if (wrap_at == n) {
#pragma unroll
                      for (int k = 0; k < 3; ++k) mma(k, d1, al[k], bl[k], id1);
                    } else {
                      const uint32_t id2 = idesc0 + (uint32_t)(n - wrap_at) * idesc_blk;
                      const uint32_t bo2 = (uint32_t)wrap_at * blk16;
#pragma unroll
                      for (int k = 0; k < 3; ++k) {
                        mma(k, d1, al[k], bl[k], id1);
                        mma(k, tmem_u, al[k], bl[k] + bo2, id2);
                      }
                    }
                  } else if (wrap_at == n) {
#pragma unroll
                    for (int k = 0; k < 3 * NKC; ++k) {
                      mma(k % 3, d1, al[k], bl[k], id1);
                      if constexpr (SPLIT) {   // lo x hi, hi x lo (shared memory ends far below 256 KB: no carry out of the address fields)
                        mma(k % 3, d1, al[k] + a_lo_off, bl[k], id1);
                        mma(k % 3, d1, al[k], bl[k] + b_lo_off, id1);
                      }
                    }
                  } else {
                    // the window wraps around the ring: first wrap_at blocks at p0, the rest from slot 0
                    const uint32_t id2 = idesc0 + (uint32_t)(n - wrap_at) * idesc_blk;
                    const uint32_t bo2 = (uint32_t)wrap_at * blk16;
#pragma unroll
                    for (int k = 0; k < 3 * NKC; ++k) {
                      mma(k % 3, d1, al[k], bl[k], id1);
                      mma(k % 3, tmem_u, al[k], bl[k] + bo2, id2);   // (weights end far below 256 KB: no carry out of the address field)
                      if constexpr (SPLIT) {
                        mma(k % 3, d1, al[k] + a_lo_off, bl[k], id1);
                        mma(k % 3, tmem_u, al[k] + a_lo_off, bl[k] + bo2, id2);
                        mma(k % 3, d1, al[k], bl[k] + b_lo_off, id1);
                        mma(k % 3, tmem_u, al[k], bl[k] + b_lo_off + bo2, id2);
                      }
                    }
                  }
                  if (leader) {
                  mbar_arrive(turn_bar(me + 1 == kSwIssuers ? 0 : me + 1));   // burst issued: the next issuer's turn
                  umma_commit(empty_bar(stage));   // stage reusable once these MMAs retire
                  // this issuer's share of every block of the window; the run's edge blocks have only two
                  // contributing steps, so the issuer of the edge step stands in for the missing third
                  if (lo) umma_commit(tfull_bar(s_lo));
                  umma_commit(tfull_bar(sl));
                  if (hi_) umma_commit(tfull_bar(s_hi));
                  if (!lo) mbar_arrive(tfull_bar(sl));
                  if (!hi_) mbar_arrive(tfull_bar(sl));
                  }
                  __syncwarp();
                  stamp(dbg_issue);
                  tr(4);
                }
                ++gstep;
                if (++owner == kSwIssuers) owner = 0;
                if (++stage == p.n_stages) { stage = 0; sphase ^= 1; }
                if (++sl == NB) { sl = 0; pr ^= 1u; }
              }
            }
          if (leader) umma_commit(layer_bar(cur));   // every MMA of this pseudo-layer issued by this warp has retired
          __syncwarp();
          if (!is_c0) ++wq;
        }
      }
      if constexpr (DBG) {
        if (dbg && leader) {
          p.debug[0] = dbg_w; p.debug[1] = dbg_tempty; p.debug[2] = dbg_full; p.debug[3] = dbg_issue;
          p.debug[4] = n_my; p.debug[5] = dbg_utt; p.debug[6] = dbg_other;
        }
      }
    }
    __syncwarp();
  } else {
    // ========================================= epilogue (4*NKC warps) =========================================
    // warp e: TMEM lane quarter q = warp % 4 (rows q*32 .. q*32+31 of the strip), channel group j = e / 4
    // (16 channels = planes 2j, 2j+1).  One block = one output column of one strip.
    // Warp (q, g): TMEM lane quarter q = warp % 4 (rows q*32 .. q*32+31 of the strip), group g = warp / 4.  One block =
    // one output column of one strip.  Group g owns every block whose running index is g mod NKC and handles ALL of its
    // channels, 16 at a time: the per-visit costs (barrier wait, slot hand-back, publishing, the latency of the first
    // TMEM load) are paid once per three blocks and per 48 channels instead of once per block and per 16 (the
    // epilogue's store/math phase, not the tensor pipe, bounded the kernel: with it disabled the same schedule ran
    // 34 % faster), and the skip tensor of the next own block is prefetched a whole two block periods ahead with a
    // single register set.
    const int q = warp & 3;
    const int g = warp >> 2;
    const int et = threadIdx.x;
    int esl = 0;         // ring slot of the block the iterator stands on
    uint32_t epr = 0;    // its use parity
    int eown = 0;        // which group owns it
    uint32_t eskpar = 0; // parity of this group's skip slot (one use per own block of a skip layer)
    int64_t sq = 0;      // pseudo-layer counter (see the producer)
    // packed strips: the rows between two stacked utterances are never stored (they stay zero = both neighbours' padding)
    const bool row_ok = !PACK || ((q * 32 + lane) % p.pack_pitch) < p.pack_h;
    // cycle accounting of epilogue warp 0 of CTA 0 (HONK2_TC_DEBUG=1)
    const bool edbg = DBG && p.debug != nullptr && blockIdx.x == 0 && warp == 0;
    const bool etrace = DBG && p.trace != nullptr && blockIdx.x == 0 && (warp == 0 || warp == 7) && lane == 0;
    int gblk = 0;
    long long e_wait = 0, e_tmem = 0, e_pub = 0, e_math = 0, e_conv0 = 0, e_t = clock64();
    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
      // Block ownership restarts with every utterance: which warp group sums which columns of the last layer then does
      // not depend on how many blocks this CTA has processed before, so an utterance's pooled sums -- and logits -- are
      // bit-identical wherever it sits in the batch (tests: full-batch permutation invariance).
      eown = 0;
      for (int ll = ll0; ll < nl1; ++ll, ++sq) {
        const bool is_c0 = ll == 0;      // conv_0 + ReLU -> P (resnet.py:40-41): no skip, no constant
        const int l = ll - 1;
        // the skip tensor of the first skip layer is conv_0's output (resnet.py:44,52): P, or the packed pre-pass buffer
        const uint4* skipP = (ext && l == 1) ? p.ext_in + b * p.ext_stride : bufP;
        const int64_t seq = sq;
        const int d = is_c0 ? 1 : layer_dil(l);
        const int n_runs = d < W ? d : W;
        const int cur = (int)(sq & 1);
        const uint32_t kc_addr = sbase + kSwKc + (uint32_t)(ll * CP) * 4u;
        // The layer body is instantiated per (skip, pooling) variant so that the registers of the skip prefetch
        // and of the pooled sums are not live together.
        auto layer_body = [&](auto skip_c, auto last_c) {
          constexpr bool HAS_SKIP = decltype(skip_c)::value;   // odd l: adds the skip tensor from P, stores to P in place
          constexpr bool LAST = decltype(last_c)::value;       // pooled instead of stored
          const bool to_p = HAS_SKIP || is_c0;   // conv_0 and the skip layers write P, the others Q
          uint4* y_out = to_p ? bufP : bufQ;
          const uint64_t pol_out = to_p ? l2_policy_evict_last() : l2_policy_evict_first();
          float psum[LAST ? CP : 1];
#pragma unroll
          for (int c = 0; c < (LAST ? CP : 1); ++c) psum[c] = 0.f;
          // Before touching this layer: wait until every MMA of the previous pseudo-layer has retired.  (1) This layer
          // overwrites the buffer the previous one READS through bulk copies / TMA, so no store may precede that.
          // (2) The skip tensor prefetched below was stored two pseudo-layers ago, possibly by ANOTHER warp group that
          // this one has overtaken (block ownership rotates; with very short layers a group can have no block in a
          // layer at all); the previous layer's MMAs having retired implies that all of its inputs were copied, hence
          // that every column of the layer before it had been stored and published.  The wait is free: none of this
          // warp's blocks of this layer can be complete earlier.
          if (sq > 0) mbar_wait_sleepy(layer_bar(cur ^ 1), (uint32_t)(((seq - 1) >> 1) & 1));
          int pending_w = -1;   // column whose stores still have to be published (one visit behind)
          auto publish = [&](int wcol) {
            // generic-proxy global stores of this thread -> visible to the async proxy (the bulk copies / TMA loads of the
            // next layer, issued by this CTA's producer after it acquires the column barrier).  The all-space
            // fence.proxy.async compiles to MEMBAR.ALL.GPU and stalls the whole SM; the .global form is a view fence.
            fence_async_global();
            __syncwarp();
            if (lane == 0) mbar_arrive(col_bar(cur, wcol));
          };
          // block iterator over (strip, run, output column of the run); every warp walks all blocks, works on its own
          struct It { int s, r, o, Lr, w; bool done; };
          struct Own { int off, w, s, slot; uint32_t par; bool exists; };   // off: this lane's position inside a plane, -1 outside the map
          It it; it.s = 0; it.r = 0; it.o = 0; it.Lr = (W + d - 1) / d; it.w = 0; it.done = false;
          auto next_own = [&]() {   // advance to this group's next block (consuming it) and describe it
            Own ob; ob.exists = false; ob.off = -1; ob.w = 0; ob.s = 0; ob.slot = 0; ob.par = 0;
            while (!it.done) {
              const bool mine = eown == g;
              if (mine) {
                const int row = it.s * 128 + q * 32 + lane;
                ob.exists = true; ob.w = it.w; ob.s = it.s; ob.slot = esl; ob.par = epr;
                ob.off = (row >= H || !row_ok) ? -1 : k32 ? ((it.w * NA) * H + row) * 2 : it.w * H + row;
              }
              // step the iterator, the ring slot and the owner
              ++it.o; it.w += d;
              if (it.o == it.Lr) {
                it.o = 0;
                if (++it.r == n_runs) { it.r = 0; if (++it.s == n_strips) it.done = true; }
                it.w = it.r;
                it.Lr = (W - it.r + d - 1) / d;
              }
              if (++esl == NB) { esl = 0; epr ^= 1u; }
              if (++eown == NG) eown = 0;
              if (mine) break;
            }
            return ob;
          };
          auto process = [&](const Own& ob) {
            const bool valid = ob.off >= 0;
            mbar_wait_sleepy(tfull_bar(ob.slot), ob.par);
            tc_fence_after();
            if constexpr (DBG) { if (etrace && warp == 0 && gblk < kSwTraceLen) p.trace[5 * kSwTraceLen + gblk] = clock64(); }
            if (edbg) { const long long t = clock64(); e_wait += t - e_t; e_t = t; }
            if (pending_w >= 0) { publish(pending_w); pending_w = -1; }
            if (edbg) { const long long t = clock64(); e_pub += t - e_t; e_t = t; }
            const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ob.slot * CP);
            // this lane's row of the staged skip column: [plane][128 rows][16 B]
            const uint32_t sk_addr = sbase + p.smem_skip_off + (uint32_t)g * SKIP_SLOT + (uint32_t)(q * 32 + lane) * 16u;
            constexpr uint32_t sk_plane = 2048u;
            // k32: this lane's row, and whether the two 16-byte halves of its row of chunk kc are stored swapped
            auto swl_of = [&](int kc) { return (uint32_t)((p.dmax + kc * H + q * 32 + lane) >> 2) & 1u; };
            const uint32_t sk_addr32 = sbase + p.smem_skip_off + (uint32_t)g * SKIP_SLOT + (uint32_t)(q * 32 + lane) * 32u;
            if constexpr (HAS_SKIP) {
              // This layer READS Q (the previous layer's output), one column per step, and the MMAs of this block were
              // the last consumers of Q column w.  Nothing reads that column again before the next even layer rewrites
              // it, so its dirty lines need not ever reach HBM: discard the 128-byte lines that lie wholly inside the
              // column (lines shared with the neighbouring columns stay).  One line per lane: the column is contiguous,
              // NKC * H * 32 B <= 96 lines.
              if (k32 && p.discard_q) {
                const char* qb = reinterpret_cast<const char*>(bufQ);
                const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(qb) & 127u);
                const uint32_t col_bytes = (uint32_t)(NKC * H) * 32u;
                const uint32_t o0 = (uint32_t)ob.w * col_bytes + mis;
                const uint32_t a = ((o0 + 127u) & ~127u) + (uint32_t)(q * 32 + lane) * 128u;
                if (a + 128u <= o0 + col_bytes)
                  asm volatile("discard.global.L2 [%0], 128;" ::"l"(qb + (a - mis)) : "memory");
              }
              if constexpr (!SPLIT) { mbar_wait_sleepy(skfull_bar(g), eskpar); eskpar ^= 1u; }
            }
            // two accumulator register sets: the TMEM load of the next 16 channels is in flight during the math of these
            uint32_t v[2][16];
            tmem_ld16(tbase, v[0]);
#pragma unroll
            for (int jj = 0; jj < NKC; ++jj) {
              // SPLIT: the skip tensor (hi and lo rows of this lane's position, 32 B each) straight from L2 -- this mode's
              // steps are three times as long, the latency hides behind the accumulator wait of the other groups' blocks
              // and the shared memory of the staging slots holds the second weight set instead.  (.cg: the rows were
              // stored by other warps of this CTA two pseudo-layers ago.)
              uint4 skv[4] = {};
              if constexpr (SPLIT && HAS_SKIP) {
                if (valid) {
                  const uint4* s_hi = skipP + jj * kc_stride + ob.off;
                  const uint4* s_lo = skipP + (NKC + jj) * kc_stride + ob.off;
                  skv[0] = ld_cg(s_hi); skv[1] = ld_cg(s_hi + 1); skv[2] = ld_cg(s_lo); skv[3] = ld_cg(s_lo + 1);
                }
              }
              tmem_ld_wait();
              tmem_st16_zero(tbase + 16 * jj);   // the next user of this ring slot accumulates from zero
              if (jj + 1 < NKC) {
                tmem_ld16(tbase + 16 * (jj + 1), v[(jj + 1) & 1]);
              } else {
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(ob.slot));   // all channels are in registers / stored, the slot is zero again
              }
              if (valid) {
                uint4 ykeep = make_uint4(0u, 0u, 0u, 0u), ykeep_lo = make_uint4(0u, 0u, 0u, 0u);
                const uint32_t swl = swl_of(jj), swl_lo = SPLIT ? swl_of(NKC + jj) : 0u;   // (SPLIT: the lo chunk's rows)
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  float x[8], kc8[8];   // constants read at use (volatile: not hoisted into registers for the whole layer)
                  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(kc8[0]), "=f"(kc8[1]), "=f"(kc8[2]), "=f"(kc8[3]) : "r"(kc_addr + (uint32_t)(64 * jj + 32 * hf)));
                  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(kc8[4]), "=f"(kc8[5]), "=f"(kc8[6]), "=f"(kc8[7]) : "r"(kc_addr + (uint32_t)(64 * jj + 32 * hf + 16)));
#pragma unroll
                  for (int e = 0; e < 8; ++e) x[e] = fmaxf(__uint_as_float(v[jj & 1][8 * hf + e]), 0.f) + kc8[e];
                  if constexpr (HAS_SKIP && SPLIT) {
                    // logical half hf of a row is stored at 16-byte slot hf ^ swl; skip = hi + lo
                    const uint4 sh = (((uint32_t)hf ^ swl) != 0u) ? skv[1] : skv[0];
                    const uint4 sl = (((uint32_t)hf ^ swl_lo) != 0u) ? skv[3] : skv[2];
                    const __nv_bfloat162* ph = reinterpret_cast<const __nv_bfloat162*>(&sh);
                    const __nv_bfloat162* pl2 = reinterpret_cast<const __nv_bfloat162*>(&sl);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                      const float2 fh = __bfloat1622float2(ph[e]), fl = __bfloat1622float2(pl2[e]);
                      x[2 * e] += fh.x + fl.x;
                      x[2 * e + 1] += fh.y + fl.y;
                    }
                  } else if constexpr (HAS_SKIP) {
                    uint4 sv;   // 8 channels of the skip tensor at this position (plane 2 jj + hf)
                    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(sv.x), "=r"(sv.y), "=r"(sv.z), "=r"(sv.w)
                                 : "r"(k32 ? sk_addr32 + (uint32_t)(jj * H) * 32u + (((uint32_t)hf ^ swl) << 4)
                                           : sk_addr + (uint32_t)(2 * jj + hf) * sk_plane));
                    const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&sv);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                      const float2 f = __bfloat1622float2(pb[e]);
                      x[2 * e] += f.x;
                      x[2 * e + 1] += f.y;
                    }
                  }
                  if constexpr (LAST) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) psum[16 * jj + 8 * hf + e] += x[e];
                  } else {
                    uint4 yo;
                    __nv_bfloat162* yb = reinterpret_cast<__nv_bfloat162*>(&yo);
#pragma unroll
                    for (int e = 0; e < 4; ++e) yb[e] = __floats2bfloat162_rn(x[2 * e], x[2 * e + 1]);
                    if constexpr (SPLIT) {
                      // the residual x - float(hi), again as bf16: hi + lo carries 16 mantissa bits of x
                      uint4 yl;
                      __nv_bfloat162* lb = reinterpret_cast<__nv_bfloat162*>(&yl);
#pragma unroll
                      for (int e = 0; e < 4; ++e) {
                        const float2 fh = __bfloat1622float2(yb[e]);
                        lb[e] = __floats2bfloat162_rn(x[2 * e] - fh.x, x[2 * e + 1] - fh.y);
                      }
                      if (hf == 0) { ykeep = yo; ykeep_lo = yl; }
                      else {
                        st_hint256(y_out + jj * kc_stride + ob.off, swl ? yo : ykeep, swl ? ykeep : yo, pol_out);
                        st_hint256(y_out + (NKC + jj) * kc_stride + ob.off, swl_lo ? yl : ykeep_lo, swl_lo ? ykeep_lo : yl, pol_out);
                      }
                    } else if constexpr (k32) {
                      // both halves of this row's 32 bytes in ONE store (16-byte stores at a 32-byte stride would write
                      // every sector in two halves); which half comes first follows the row's swizzle bit
                      if (hf == 0) ykeep = yo;
                      else st_hint256(y_out + jj * kc_stride + ob.off, swl ? yo : ykeep, swl ? ykeep : yo, pol_out);
                    } else {
                      st_hint(y_out + (int64_t)(2 * jj + hf) * plane_stride + ob.off, yo, pol_out);
                    }
                  }
                }
              }
            }
            if (edbg) { const long long t = clock64(); e_math += t - e_t; e_t = t; }
            if constexpr (DBG) {
              if (etrace && gblk < kSwTraceLen) p.trace[(warp == 0 ? 6 : 7) * kSwTraceLen + gblk] = clock64();
              ++gblk;
            }
            pending_w = ob.w;
          };
          // Skip layers (odd l, resnet.py:51-53): the block of output column w adds column w of P.  That column is staged
          // in this group's shared-memory slot (k32: one bulk copy; planar: NP) issued by the group's quarter-0 warp as soon as all four
          // warps have finished reading the previous one, i.e. two block periods before it is needed: no L2 latency on
          // the epilogue's critical path and no prefetch registers (they hold a second accumulator set instead).
          auto stage_skip = [&](const Own& ob) {
            if constexpr (HAS_SKIP && !SPLIT) {
              asm volatile("bar.sync %0, 128;" ::"r"(2 + g) : "memory");   // the group's four warps are done with the slot
              if (k32) {
                if (q == 0 && ob.exists && elect_one()) {   // the whole column, [K chunk][H rows][32 B]
                  const uint32_t bytes = (uint32_t)(NKC * H) * 32u;
                  mbar_expect_tx(skfull_bar(g), bytes);
                  bulk_load_hint(sbase + p.smem_skip_off + (uint32_t)g * SKIP_SLOT, skipP + (ob.w * NKC) * H * 2, bytes,
                                 skfull_bar(g), l2_policy_evict_last());
                }
              } else if (q == 0 && ob.exists && elect_one()) {
                const int rows = H - ob.s * 128 < 128 ? H - ob.s * 128 : 128;
                mbar_expect_tx(skfull_bar(g), (uint32_t)(NP * rows * 16));
                const uint4* src = bufP + (int64_t)ob.w * H + ob.s * 128;
                const uint32_t d0 = sbase + p.smem_skip_off + (uint32_t)g * SKIP_SLOT;
#pragma unroll
                for (int pl = 0; pl < NP; ++pl)
                  bulk_load_hint(d0 + (uint32_t)pl * 2048u, src + (int64_t)pl * plane_stride, (uint32_t)(rows * 16), skfull_bar(g), l2_policy_evict_last());
              }
            }
          };
          Own ob = next_own();
          stage_skip(ob);
          while (ob.exists) {
            process(ob);
            ob = next_own();
            stage_skip(ob);
          }
          if (pending_w >= 0) publish(pending_w);
          if constexpr (LAST) {
            // fused global mean (resnet.py:57-58): warp-reduce the 32 rows; every warp leaves ITS share of every channel
            // in its own row of s_pool (no atomics: the logits below add the rows in a fixed order, so repeated
            // launches agree bit for bit)
            if constexpr (!PACK) {
#pragma unroll
              for (int c = 0; c < CP; ++c) {
                float sum = psum[c];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                if (lane == (c & 31)) s_pool[warp * CP + c] = sum;
              }
            } else {
              // packed strips: one sum per stacked utterance (this lane's row belongs to utterance `mine`, or to none)
              const int prow = q * 32 + lane;
              const int mine = (row_ok && prow < H) ? prow / p.pack_pitch : -1;
              for (int u = 0; u < p.pack_n; ++u) {
#pragma unroll
                for (int c = 0; c < CP; ++c) {
                  float sum = mine == u ? psum[c] : 0.f;
#pragma unroll
                  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                  if (lane == (c & 31)) s_pool[(u * kEpiWarps + warp) * CP + c] = sum;
                }
              }
            }
          }
        };
        const bool has_skip = !is_c0 && (l & 1) != 0, last = l == n_layers - 1;
        if (has_skip) { if (last) layer_body(std::true_type{}, std::true_type{}); else layer_body(std::true_type{}, std::false_type{}); }
        else { if (last) layer_body(std::false_type{}, std::true_type{}); else layer_body(std::false_type{}, std::false_type{}); }
      }

      // ------------------------------ logits (resnet.py:59) ------------------------------
      // One label per warp, lanes over the channels (C <= 64 on this kernel); the label's folded weights are fetched
      // BEFORE the barrier, so their L2 latency overlaps the wait for the other warps' pooled sums.  (All epilogue
      // warps stand at these two barriers between utterances while the accumulator ring fills up behind them: with
      // one thread per label walking the channels through global loads the event trace showed a ~20 000-cycle stall
      // per utterance, ~8 000 with this form.  Under the power cap the end-to-end gain is within noise.)
      // s_pool holds sums of z = x - mean; the BatchNorm output mean is z_mean / sigma (resnet.py:55-58)
      {
        const int sub_h = PACK ? p.pack_h : H;
        const float inv = 1.f / (float)(sub_h * W);
        auto fold = [&](int lb, float (&wv)[2]) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const int c = lane + 32 * k;
            wv[k] = c < p.C ? __ldg(p.last_scale + c) * inv * __ldg(p.out_w + lb * p.C + c) : 0.f;
          }
        };
        float wv[2] = {0.f, 0.f};
        if (warp < p.n_labels) fold(warp, wv);
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        if (warp < p.n_labels) {
          const int n_sub = PACK ? p.pack_n : 1;
          for (int u = 0; u < n_sub; ++u) {
            const int64_t bu = PACK ? b * p.pack_n + u : b;
            if (PACK && bu >= p.B_utt) break;
            const float* sp = s_pool + u * kEpiWarps * CP;
            float ps[2] = {0.f, 0.f};   // this lane's channels: the epilogue warps' shares, added in warp order
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const int c = lane + 32 * k;
              if (c < p.C)
                for (int e = 0; e < kEpiWarps; ++e) ps[k] += sp[e * CP + c];
            }
            for (int lb = warp; lb < p.n_labels; lb += kEpiWarps) {
              if (lb != warp || u > 0) fold(lb, wv);
              float v = fmaf(ps[0], wv[0], ps[1] * wv[1]);
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
              if (lane == 0) p.logits[bu * p.n_labels + lb] = v + __ldg(p.out_b + lb);
            }
          }
        }
      }
      // (no second barrier: s_pool is rewritten, never accumulated into, and its next writers -- the last layer of the
      // next utterance -- are a whole utterance minus one accumulator ring behind this read)
      (void)et;
      if (edbg) { const long long t = clock64(); e_math += t - e_t; e_t = t; }
    }
    if (edbg && lane == 0) {
      p.debug[8] = e_wait; p.debug[9] = e_tmem; p.debug[10] = e_pub; p.debug[11] = e_math; p.debug[12] = e_conv0;
    }
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == kEpiWarps + 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace kws
