// Micro-benchmark #6: can the zero pad rows of a staged column be replaced by tcgen05.mma's disable-output-lane mask?
//
// The column-sweep kernel reads the height tap dh of output row h from staged row h + (dh - 1) d.  Today every 16-channel
// chunk of a staged column has d zero rows above and below it, so that the taps of the map's edge rows read zeros (the
// reference's zero padding).  With a 128-bit lane mask the MMA can instead leave the edge lanes alone: the tap that
// reads row h - d must not update lanes 0 .. d-1, the tap that reads row h + d must not update lanes H-d .. H-1.  The
// chunks of a column then need no rows between them, and a column can be one contiguous bulk copy.
//
// 1. Exactness.  One 128 x 144 x 16 MMA, A = K-major SWIZZLE_32B rows of a buffer whose rows are all NONZERO (no pad
//    rows anywhere), start address shifted by -d or +d rows, B = the SWIZZLE_NONE weight layout of the sweep kernel,
//    accumulating into a TMEM block preloaded with a known pattern, mask = the edge lanes of that shift (H = 101 and
//    H = 128).  Masked lanes must be bit-unchanged, the others must equal pattern + the exact product (small integers),
//    which is what the zero rows gave for them.  The unmasked MMA is run too, to show the mask is what keeps the edge.
// 2. Rate.  The sweep's step, 148 CTAs x 3 issuer warps passing a burst token: each step is 9 MMAs (3 K chunks x 3
//    height taps) of N = 144 into a window that slides one 48-column block per step, from a ring of staged columns laid
//    out as [guard][3 chunks x H rows] (H = 101, pitch H).  Variants: no mask operand / the three edge masks of d = 1 /
//    edge masks plus lanes >= H.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/umma_bench6 tools/umma_bench6.cu
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <vector>
#include <algorithm>
#include <cstring>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) if (clock64() - t0 > 2000000000ll) __trap();
}
__device__ __forceinline__ void umma(uint32_t d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, 1;\n\t}"
      ::"r"(d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc) : "memory");
}
__device__ __forceinline__ void umma_mask(uint32_t d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint4 m) {
  asm volatile(
      "{\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, {%6, %7, %8, %9}, 1;\n\t}"
      ::"r"(d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(m.x), "r"(m.y), "r"(m.z), "r"(m.w) : "memory");
}
__device__ __forceinline__ bool elect_one_lane() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                 "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// lanes lo .. hi-1 as a disable-output-lane mask (bit i of the 128-bit value = lane i, word j = lanes 32 j .. 32 j + 31)
__host__ __device__ inline uint4 lane_mask(int lo, int hi) {
  uint32_t w[4] = {0u, 0u, 0u, 0u};
  for (int i = lo; i < hi; ++i) if (i >= 0 && i < 128) w[i >> 5] |= 1u << (i & 31);
  return make_uint4(w[0], w[1], w[2], w[3]);
}

constexpr int kN = 144, kRows = 192, kGuard = 16;     // A: kRows swizzled 32-byte rows, the MMA starts at kGuard +- d
constexpr uint32_t kAHi = (256u >> 4) | (1u << 14) | (6u << 29);   // SWIZZLE_32B, SBO = 256 B, version 1
constexpr uint32_t kBHi = (128u >> 4) | (1u << 14);                 // SWIZZLE_NONE, SBO = 128 B
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kN >> 3) << 17) | (8u << 24);

struct Case { int shift; uint4 mask; int use_mask; };

// one case per launch: D = pattern; D += A[kGuard + shift + i] * B (masked); D -> out [128][kN]
__global__ void __launch_bounds__(128, 1) exact_kernel(const float* A, const float* B, Case c, float* out) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  unsigned char* sA = smem;               // kRows * 32 B
  unsigned char* sB = smem + 8192;        // [K half][n][16 B]
  for (int i = threadIdx.x; i < kRows * 16; i += blockDim.x) {
    const int r = i / 16, k = i % 16;
    *reinterpret_cast<__nv_bfloat16*>(sA + r * 32 + (((k >> 3) ^ ((r >> 2) & 1)) << 4) + (k & 7) * 2) = __float2bfloat16(A[i]);
  }
  for (int i = threadIdx.x; i < kN * 16; i += blockDim.x) {
    const int n = i / 16, k = i % 16;
    *reinterpret_cast<__nv_bfloat16*>(sB + (k >> 3) * (kN * 16) + n * 16 + (k & 7) * 2) = __float2bfloat16(B[i]);
  }
  if (threadIdx.x == 0) { mbar_init(smem_u32(&bar), 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, row = threadIdx.x;
  const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
  for (int n0 = 0; n0 < kN; n0 += 16) {   // pattern: (row * 3 + n) % 17 - 8 (small integers, nonzero in most lanes)
    uint32_t v[16];
    for (int j = 0; j < 16; ++j) v[j] = __float_as_uint((float)((row * 3 + n0 + j) % 17 - 8));
    tmem_st16(tl + (uint32_t)n0, v);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (threadIdx.x == 0) {
    const uint32_t a_lo = ((smem_u32(sA) + (uint32_t)(kGuard + c.shift) * 32u) >> 4) & 0x3FFFu;
    const uint32_t b_lo = ((smem_u32(sB) >> 4) & 0x3FFFu) | (((uint32_t)(kN * 16) >> 4) << 16);
    if (c.use_mask) umma_mask(tmem, a_lo | (1u << 16), kAHi, b_lo, kBHi, kIdesc, c.mask);
    else umma(tmem, a_lo | (1u << 16), kAHi, b_lo, kBHi, kIdesc);
    umma_commit(smem_u32(&bar));
  }
  mbar_wait(smem_u32(&bar), 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  for (int n0 = 0; n0 < kN; n0 += 16) {
    uint32_t v[16];
    tmem_ld16(tl + (uint32_t)n0, v);
    for (int j = 0; j < 16; ++j) out[row * kN + n0 + j] = __uint_as_float(v[j]);
  }
  (void)lane;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256) : "memory");
  }
}

// ---- rate: the sweep's nine-MMA step, three issuer warps with a burst token
constexpr int kH = 101, kNA = 3, kStages = 8;
constexpr int kSlotRows = ((kGuard + kNA * kH + kGuard) + 7) & ~7;   // guard, three chunks at pitch H, slack
constexpr int kSlotBytes = kSlotRows * 32;
constexpr int kSlabBytes = 2 * 3 * 48 * 16;                          // one (kc, dh) weight slab: [K half][3 blocks][48][16 B]

template <int MODE>   // 0 = no mask operand, 1 = edge masks of d = 1, 2 = edge masks + lanes >= H
__global__ void __launch_bounds__(128, 1) rate_kernel(int steps, long long* cycles) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t turn[3], done[3];
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5;
  // random-looking bf16 data everywhere (the power drawn depends on the operands)
  for (int i = threadIdx.x; i < (kStages * kSlotBytes + 9 * kSlabBytes) / 4; i += blockDim.x) {
    const uint32_t h = (uint32_t)i * 2654435761u;
    const uint32_t lo = 0x3c00u | ((h >> 7) & 0x3FFu) | ((h & 1u) << 15), hi = 0x3c00u | ((h >> 17) & 0x3FFu) | ((h & 2u) << 14);
    reinterpret_cast<uint32_t*>(smem)[i] = (lo & 0xBFFFu) | ((hi & 0xBFFFu) << 16);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < 3; ++i) { mbar_init(smem_u32(&turn[i]), 1); mbar_init(smem_u32(&done[i]), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive(smem_u32(&turn[0]));
  }
  if (warp == 3) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = __shfl_sync(0xffffffffu, tmem_slot, 0);
  if (warp < 3) {
    const int me = warp;
    const uint32_t ring16 = smem_u32(smem) >> 4, w16 = (smem_u32(smem) + kStages * kSlotBytes) >> 4;
    const uint32_t b_lbo = ((uint32_t)(3 * 48 * 16) >> 4) << 16;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(144 >> 3) << 17) | (8u << 24);
    const int d = 1;
    const uint4 m_ge = MODE == 2 ? lane_mask(kH, 128) : make_uint4(0u, 0u, 0u, 0u);
    uint4 mk[3];
    mk[0] = lane_mask(0, d); mk[1] = make_uint4(0u, 0u, 0u, 0u); mk[2] = lane_mask(kH - d, kH);
    for (int t = 0; t < 3; ++t) { mk[t].x |= m_ge.x; mk[t].y |= m_ge.y; mk[t].z |= m_ge.z; mk[t].w |= m_ge.w; }
    uint32_t par = 0;
    int stage = me, win = me;
    const long long t0 = clock64();
    for (int s = me; s < steps; s += 3) {
      const uint32_t a16 = ring16 + (uint32_t)(stage * kSlotBytes >> 4) + (uint32_t)(kGuard - d) * 2u;
      const uint32_t dt = tmem + (uint32_t)(win * 48);
      uint32_t al[9], bl[9];
#pragma unroll
      for (int kc = 0; kc < 3; ++kc)
#pragma unroll
        for (int dh = 0; dh < 3; ++dh) {
          al[kc * 3 + dh] = ((a16 + (uint32_t)(kc * kH * 2) + (uint32_t)(dh * d * 2)) & 0x3FFFu) | (1u << 16);
          bl[kc * 3 + dh] = ((w16 + (uint32_t)(((kc * 3 + dh) * kSlabBytes) >> 4)) & 0x3FFFu) | b_lbo;
        }
      mbar_wait(smem_u32(&turn[me]), par);
      par ^= 1u;
      if (elect_one_lane()) {
#pragma unroll
        for (int k = 0; k < 9; ++k) {
          if constexpr (MODE == 0) umma(dt, al[k], kAHi, bl[k], kBHi, idesc);
          else umma_mask(dt, al[k], kAHi, bl[k], kBHi, idesc, mk[k % 3]);
        }
        mbar_arrive(smem_u32(&turn[me + 1 == 3 ? 0 : me + 1]));
      }
      __syncwarp();
      stage += 3; if (stage >= kStages) stage -= kStages;
      win += 3; if (win >= 8) win -= 8;   // windows of 144 columns at 48-column steps inside 512 columns
    }
    if (elect_one_lane()) umma_commit(smem_u32(&done[me]));
    __syncwarp();
    mbar_wait(smem_u32(&done[me]), 0);
    if ((threadIdx.x & 31) == 0) cycles[blockIdx.x * 3 + me] = clock64() - t0;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 3) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

int main() {
  // ---- 1. exactness
  std::vector<float> A(kRows * 16), B(kN * 16);
  for (int r = 0; r < kRows; ++r)
    for (int k = 0; k < 16; ++k) A[r * 16 + k] = (float)(((r * 7 + k * 3) % 13) - 6 + (((r + k) % 13) == 6 ? 1 : 0));   // no zero rows
  for (int n = 0; n < kN; ++n)
    for (int k = 0; k < 16; ++k) B[n * 16 + k] = (float)(((n * 5 + k * 11) % 9) - 4);
  float *dA, *dB, *dD;
  cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, 128 * kN * 4);
  cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
  cudaFuncSetAttribute(exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768);
  int n_fail = 0;
  printf("exactness: 128 x %d x 16 MMA, SWIZZLE_32B A without pad rows, accumulate onto a pattern\n", kN);
  for (int H : {101, 128})
    for (int d : {1, 2, 4, 8, 16})
      for (int side = 0; side < 2; ++side)
        for (int use_mask = 1; use_mask >= 0; --use_mask) {
          const int shift = side == 0 ? -d : d;
          const int m_lo = side == 0 ? 0 : H - d, m_hi = side == 0 ? d : H;
          Case c{shift, lane_mask(m_lo, m_hi), use_mask};
          cudaMemset(dD, 0, 128 * kN * 4);
          exact_kernel<<<1, 128, 32768>>>(dA, dB, c, dD);
          const cudaError_t e = cudaDeviceSynchronize();
          if (e != cudaSuccess) { printf("kernel failed: %s\n", cudaGetErrorString(e)); return 1; }
          std::vector<float> D(128 * kN);
          cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
          int bad_masked = 0, bad_live = 0, changed_masked = 0;
          for (int i = 0; i < 128; ++i) {
            const bool masked = use_mask && i >= m_lo && i < m_hi;
            for (int n = 0; n < kN; ++n) {
              const float pat = (float)((i * 3 + n) % 17 - 8);
              float dot = 0.f;
              for (int k = 0; k < 16; ++k) dot += A[(kGuard + shift + i) * 16 + k] * B[n * 16 + k];
              const float got = D[i * kN + n];
              if (masked) { if (std::memcmp(&got, &pat, 4) != 0) ++bad_masked; }
              else if (got != pat + dot) ++bad_live;
              if (!use_mask && i >= m_lo && i < m_hi && got != pat) ++changed_masked;
            }
          }
          if (use_mask) {
            printf("  H %3d d %2d %s (start %+3d rows, lanes %3d..%3d masked): masked lanes %s, live lanes %s\n", H, d,
                   side ? "bottom" : "top   ", shift, m_lo, m_hi - 1, bad_masked ? "CHANGED" : "bit-unchanged",
                   bad_live ? "WRONG" : "exact");
            n_fail += bad_masked + bad_live;
          } else {
            printf("  H %3d d %2d %s without mask: live lanes %s, edge lanes updated in %d of %d elements\n", H, d,
                   side ? "bottom" : "top   ", bad_live ? "WRONG" : "exact", changed_masked, d * kN);
            n_fail += bad_live;
          }
        }
  printf("exactness: %s\n", n_fail ? "FAILED" : "all cases exact");

  // ---- 2. rate
  long long* dcyc;
  cudaMalloc(&dcyc, 148 * 3 * sizeof(long long));
  const int smem = kStages * kSlotBytes + 9 * kSlabBytes;
  cudaFuncSetAttribute(rate_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaFuncSetAttribute(rate_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaFuncSetAttribute(rate_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  const int steps = 30000;
  const char* names[3] = {"no mask operand      ", "edge masks (d = 1)   ", "edge masks + lanes>=H"};
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  printf("rate: 148 CTAs x 3 issuers, %d steps of 9 MMAs (128 x 144 x 16) per CTA, H = %d, pitch H, 5 alternating rounds\n",
         steps, kH);
  std::vector<double> ms[3], cyc[3];
  for (int round = 0; round < 6; ++round)
    for (int mode = 0; mode < 3; ++mode) {
      cudaEventRecord(e0);
      if (mode == 0) rate_kernel<0><<<148, 128, smem>>>(steps, dcyc);
      else if (mode == 1) rate_kernel<1><<<148, 128, smem>>>(steps, dcyc);
      else rate_kernel<2><<<148, 128, smem>>>(steps, dcyc);
      cudaEventRecord(e1);
      const cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("rate kernel failed: %s\n", cudaGetErrorString(e)); return 1; }
      if (round == 0) continue;   // warm-up
      float t = 0.f;
      cudaEventElapsedTime(&t, e0, e1);
      std::vector<long long> h(148 * 3);
      cudaMemcpy(h.data(), dcyc, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
      ms[mode].push_back(t);
      cyc[mode].push_back((double)*std::max_element(h.begin(), h.end()));
    }
  for (int mode = 0; mode < 3; ++mode) {
    std::sort(ms[mode].begin(), ms[mode].end());
    std::sort(cyc[mode].begin(), cyc[mode].end());
    const double med_cyc = cyc[mode][cyc[mode].size() / 2];
    printf("  %s: %.2f cycles per MMA (median, max over CTAs), kernel %.3f ms median (min %.3f, max %.3f)\n", names[mode],
           med_cyc / (9.0 * steps), ms[mode][ms[mode].size() / 2], ms[mode].front(), ms[mode].back());
  }
  return 0;
}
