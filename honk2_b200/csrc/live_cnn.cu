// Live CNN streams (kws_live_cnn_*): a live front-end (kws_live, mfcc.cu) feeding the bf16 CNN of the cnn_tc family,
// which computes each convolution row of a stream once.
//
// Neither convolution pads in time and MaxPool(1,3) pools along frequency only, so the network is shift-equivariant
// along a stream.  Window k's frames t = 2 .. T-3 are the stream's frame-table rows k m + t (m = shift / 160); only
// its four edge frames t = 0, 1, T-2, T-1 (reflect-padded at the window's ends) are its own.  Hence
//   pooled conv_0 row r of window k = stream pooled row k m + r   unless r < 2 or r > H0 - 3,
//   conv_1 row r of window k        = stream conv_1 row k m + r   unless r < 2 or r > H1 - 3,
// and a push of n samples per stream computes n / 160 new stream rows of each convolution per stream plus four
// window-specific rows of each per window (rows 0, 1, H-2, H-1), instead of H0 + H1 rows per window.
//
// Per stream the state keeps a ring of pooled conv_0 rows (cap0 rows of WP x 64 bf16) and a ring of conv_1 rows (cap1
// rows of 1 KB, [4 channel groups][8 positions][16 channels], the order cnn_lin0_kernel's weights are packed in).
// Ring capacities (P = max_push / 160; window k0 is the push's first, k0 + K - 1 its last; K m <= P):
//   a push writes stream rows ((k0 - 1) m + H - 3, (k0 + K - 1) m + H - 3] of each ring (H = H0 or H1), K m of them,
//   and reads no stream row older than k0 m + 2 (the oldest window's first shared row; a new stream conv_1 row R >
//   (k0 - 1) m + H1 - 3 reads pooled rows from R on, and R >= k0 m + 2 whenever a window reads it).  The newest row
//   written minus the oldest row read is at most (K - 1) m + H - 5 < P + H, so with cap = P + H no row a push reads
//   is overwritten by that push, and the K m rows it writes go to distinct slots.
//
// Launches per push: append and frame-table rows (mfcc.cu), edge frames into [S K][4][n_mels], conv_0 rows, conv_1
// rows, the first Linear over ring + window-specific rows (cnn_lin0_kernel<LiveActRows>), the remaining Linear layers
// (cnn_mlp_kernel), zeroing of the warm-up slots.  Every row address is derived on the device from the stream
// counters; nothing is read back.
//
// The two convolution kernels are bf16 mma.sync (m16n8k16, fp32 accumulation) over rows gathered from any stream:
// each lane hands ldmatrix its own row address, so rows of different streams share an MMA tile without a common
// layout.  They keep cnn_tc_fused_kernel's MMA shape (K = 16 per product), K order and rounding points (features and
// pooled rows to bf16, max + bias + ReLU on the fp32 accumulators), and the first Linear keeps its split-K slices: on
// the B200 the logits are bit-identical to the batch path's on the materialised windows (tests/test_live_cnn.py).
//
// Ragged pushes (kws_live_cnn_push_ragged): stream s goes from count c to c' = c + n_s, any n_s in [0, max_push].  The
// stream rows of a convolution are a function of the counter alone: with top(c) = floor((c - W) / H) m + Hc - 3 (Hc =
// H0 or H1, the floor not clamped at 0), a push computes rows (top(c), top(c')], which for aligned counts are the rows
// the uniform push computes, so the two pushes may be mixed on one state.  During a stream's warm-up a push computes
// rows although it completes no window; window 0 reads them.  The windows the push completes are compacted as the
// front-end's ragged push lists them (window i of the push: stream s, window k), and their window-specific rows go to
// slot i of the edge buffers.  Ring capacity: DESIGN.md section 7, "Ragged pushes".
#include "live.cuh"
#include "tc.cuh"
#include <cub/device/device_scan.cuh>
#include <algorithm>

namespace kws {

constexpr int kLc0Warps = 4;     // conv_0: one row per warp
constexpr int kLc1Jobs = 32;     // conv_1: rows per CTA (8 warps x 4 rows)
constexpr int kLc1Threads = 256;
constexpr int kLcRow1 = 512;     // conv_1 row: 4 x 8 x 16 bf16

__device__ __forceinline__ int64_t lc_floor_div(int64_t a, int64_t b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }
__device__ __forceinline__ int lc_mod(int64_t a, int m) { const int64_t r = a % m; return (int)(r < 0 ? r + m : r); }

__device__ __forceinline__ uint32_t lc_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void lc_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(src));
}
__device__ __forceinline__ uint32_t lc_pack(float a, float b) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t lc_pack_relu(float a, float b) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}

// Row jobs of a push, shared by both convolutions: jobs [0, S P) are stream rows (stream j / P, row
// (k0 - 1) m + H - 2 + j % P); jobs [S P, S P + 4 S K) are window rows (slot w / 4, row 0, 1, H-2, H-1 for w % 4).
struct LcPush {
  static constexpr bool kRagged = false;
  const int64_t* count;
  int S, n, window, shift, K, m, P;
  int64_t jobs;
  __device__ __forceinline__ int64_t first_window(int s) const {
    return lc_floor_div(count[s] - n - window, shift) + 1;
  }
};
struct LcJob {
  int s;
  bool stream;
  int64_t row;    // stream row (stream job) or window index k (window job)
  int64_t slot;   // window slot (window job)
  int e;          // 0..3: window row 0, 1, H-2, H-1
};
__device__ __forceinline__ LcJob lc_job(const LcPush& p, int64_t j, int H) {
  LcJob J;
  const int64_t sp = (int64_t)p.S * p.P;
  if (j < sp) {
    J.s = (int)(j / p.P);
    J.stream = true;
    J.row = (p.first_window(J.s) - 1) * p.m + H - 2 + (j - (int64_t)J.s * p.P);
    J.slot = 0; J.e = 0;
  } else {
    const int64_t w = j - sp;
    J.slot = w >> 2; J.e = (int)(w & 3);
    J.s = (int)(J.slot / p.K);
    J.stream = false;
    J.row = p.first_window(J.s) + (J.slot - (int64_t)J.s * p.K);
  }
  return J;
}
__device__ __forceinline__ int64_t lc_total(const LcPush& p) { return p.jobs; }

// Row jobs of a ragged push: jobs [0, R) are stream rows, rows (top(c), top(c')] of each stream in stream order
// (rows[s]: exclusive scan of the per-stream counts, rows[S] = R); jobs [R, R + 4 M) are window rows (window w / 4 of the
// push's compacted list, row 0, 1, H-2, H-1 for w % 4; wins: the front-end's plan, windows in the low 32 bits, wins[S]
// = M).  R and M live on the device and the launch covers the host's bounds: CTAs past R + 4 M exit.  conv_0 also writes
// each window's stream and index and M (each pointer may be null).
struct LcRagged {
  static constexpr bool kRagged = true;
  const int64_t* count;   // this push included
  const int* len;
  const int64_t* rows;
  const int64_t* wins;
  int S, window, shift, m;
  int64_t *win_stream, *win_index, *n_windows;
};
__device__ __forceinline__ int64_t lc_total(const LcRagged& p) {
  return __ldg(p.rows + p.S) + 4 * (__ldg(p.wins + p.S) & 0xffffffffll);
}
// stream of entry e of a compacted list (plan & mask: exclusive scan of the per-stream counts) and the entries before it
__device__ __forceinline__ int lc_stream_of(const int64_t* plan, int S, int64_t mask, int64_t e, int64_t* before) {
  int lo = 0, hi = S;   // (plan[lo] <= e < plan[hi])
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((__ldg(plan + mid) & mask) <= e) lo = mid;
    else hi = mid;
  }
  *before = __ldg(plan + lo) & mask;
  return lo;
}
__device__ __forceinline__ LcJob lc_job(const LcRagged& p, int64_t j, int H) {
  LcJob J;
  const int64_t R = __ldg(p.rows + p.S);
  int64_t before;
  if (j < R) {
    J.s = lc_stream_of(p.rows, p.S, ~0ll, j, &before);
    J.stream = true;
    const int64_t c_old = __ldg(p.count + J.s) - __ldg(p.len + J.s);
    J.row = lc_floor_div(c_old - p.window, p.shift) * p.m + H - 2 + (j - before);   // top(c) + 1 + ...
    J.slot = 0; J.e = 0;
  } else {
    const int64_t w = j - R;
    J.slot = w >> 2; J.e = (int)(w & 3);
    J.s = lc_stream_of(p.wins, p.S, 0xffffffffll, J.slot, &before);
    J.stream = false;
    const int64_t c_old = __ldg(p.count + J.s) - __ldg(p.len + J.s);
    const int64_t k0 = lc_floor_div(c_old - p.window, p.shift) + 1;
    J.row = (k0 > 0 ? k0 : 0) + (J.slot - before);
  }
  return J;
}

// window row of job J (window job) for kernel row kh, and whether it is one of the window's own rows
__device__ __forceinline__ int lc_win_row(const LcJob& J, int H) { return J.e < 2 ? J.e : H - 4 + J.e; }

// ---------------------------------------------------------------------------------------------
// conv_0 + max pool (1, 3) + bias + ReLU.  One warp computes one pooled row: M = 3 pool members x 16 pooled columns
// (column 3j + e is row j of m-tile e), N = 64, K = ks0 steps of two kernel rows x 8 taps (conv_0's packed weights).
// JOBS: LcPush (uniform pushes) or LcRagged.
template <typename JOBS>
struct Lc0Params {
  JOBS p;
  const float* frames; int fcap;      // live frame rings [S][fcap][F]
  const float* edges;                 // [S K][4][F]
  const __nv_bfloat16* w0;            // [ks0][2][64][8]
  const float* b0;
  __nv_bfloat16* ring0; int cap0;     // [S][cap0][WP][64]
  __nv_bfloat16* edge0;               // [S K][4][WP][64]
  int T, F, KH0, H0, WP, ks0;
};

template <typename JOBS>
__global__ void __launch_bounds__(32 * kLc0Warps)
live_cnn_conv0_kernel(const Lc0Params<JOBS> q) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t jobs = lc_total(q.p);
  if constexpr (JOBS::kRagged) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && q.p.n_windows) *q.p.n_windows = __ldg(q.p.wins + q.p.S) & 0xffffffffll;
    if ((int64_t)blockIdx.x * kLc0Warps >= jobs) return;
  }
  const int kh2 = 2 * q.ks0;
  unsigned char* s_w = smem;                                          // ks0 * 2048 B
  unsigned char* s_a = smem + q.ks0 * 2048 + warp * (3 * kh2 * 256);  // [3][kh2][16 columns][16 B]
  for (int i = threadIdx.x; i < q.ks0 * 128; i += blockDim.x)
    reinterpret_cast<uint4*>(s_w)[i] = reinterpret_cast<const uint4*>(q.w0)[i];
  const int64_t job = (int64_t)blockIdx.x * kLc0Warps + warp;
  const bool live = job < jobs;
  const LcJob J = lc_job(q.p, live ? job : jobs - 1, q.H0);
  if constexpr (JOBS::kRagged) {
    if (live && lane == 0 && !J.stream && J.e == 0) {
      if (q.p.win_stream) q.p.win_stream[J.slot] = J.s;
      if (q.p.win_index) q.p.win_index[J.slot] = J.row;
    }
  }
  const int r = J.stream ? 0 : lc_win_row(J, q.H0);
  const int64_t slot4 = J.slot * 4;
  const float* frames_s = q.frames + (int64_t)J.s * q.fcap * q.F;
  auto frame = [&](int kh) -> const float* {
    if (J.stream) return frames_s + (int64_t)lc_mod(J.row + kh, q.fcap) * q.F;
    const int t = r + kh;
    if (t < 2) return q.edges + (slot4 + t) * q.F;
    if (t >= q.T - 2) return q.edges + (slot4 + t - q.T + 4) * q.F;
    return frames_s + (int64_t)lc_mod(J.row * q.p.m + t, q.fcap) * q.F;
  };
  // A_e[kh][j] = bf16(x[kh][3j + e .. 3j + e + 7]) (zero past the features, the pooled width and KH0)
  for (int item = lane; item < kh2 * 16; item += 32) {
    const int kh = item >> 4, j = item & 15;
    float v[10];
    if (kh < q.KH0 && j < q.WP) {
      const float* x = frame(kh) + 3 * j;
#pragma unroll
      for (int i = 0; i < 10; ++i) v[i] = 3 * j + i < q.F ? __ldg(x + i) : 0.f;
    } else {
#pragma unroll
      for (int i = 0; i < 10; ++i) v[i] = 0.f;
    }
#pragma unroll
    for (int e = 0; e < 3; ++e)
      *reinterpret_cast<uint4*>(s_a + ((e * kh2 + kh) * 16 + j) * 16) =
          make_uint4(lc_pack(v[e], v[e + 1]), lc_pack(v[e + 2], v[e + 3]), lc_pack(v[e + 4], v[e + 5]),
                     lc_pack(v[e + 6], v[e + 7]));
  }
  __syncthreads();
  if (!live) return;
  float c[3][8][4];
#pragma unroll
  for (int e = 0; e < 3; ++e)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[e][nt][i] = 0.f;
  const int mi = lane >> 3, l8 = lane & 7;
  const uint32_t a_base = lc_smem(s_a) + (uint32_t)((((mi >> 1) * 16) + (mi & 1) * 8 + l8) * 16);
  const uint32_t b_base = lc_smem(s_w) + (uint32_t)((((mi & 1) * 64) + (mi >> 1) * 8 + l8) * 16);
  for (int ks = 0; ks < q.ks0; ++ks) {
    uint32_t b[8][2];
#pragma unroll
    for (int np = 0; np < 4; ++np)
      ldsm_x4(b_base + (uint32_t)((ks * 128 + np * 16) * 16), b[2 * np][0], b[2 * np][1], b[2 * np + 1][0],
              b[2 * np + 1][1]);
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      uint32_t a[4];
      ldsm_x4(a_base + (uint32_t)(((e * kh2 + 2 * ks) * 16) * 16), a[0], a[1], a[2], a[3]);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) lc_mma(c[e][nt], a, b[nt][0], b[nt][1]);
    }
  }
  __nv_bfloat16* out = J.stream ? q.ring0 + ((int64_t)J.s * q.cap0 + lc_mod(J.row, q.cap0)) * q.WP * 64
                                : q.edge0 + (slot4 + J.e) * q.WP * 64;
  const int gq = lane >> 2, tq = lane & 3;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int co = nt * 8 + 2 * tq;
    const float bx = __ldg(q.b0 + co), by = __ldg(q.b0 + co + 1);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = gq + 8 * h;
      if (j < q.WP) {
        const float vx = fmaxf(fmaxf(c[0][nt][2 * h], c[1][nt][2 * h]), c[2][nt][2 * h]) + bx;
        const float vy = fmaxf(fmaxf(c[0][nt][2 * h + 1], c[1][nt][2 * h + 1]), c[2][nt][2 * h + 1]) + by;
        *reinterpret_cast<uint32_t*>(out + j * 64 + co) = lc_pack_relu(vx, vy);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// conv_1 + bias + ReLU.  A CTA computes 32 rows (warp w: rows 4w .. 4w+3, two m16 tiles of two rows x 8 positions),
// N = 64, K = KH1 x KW1 x 64 in the batch kernel's order ((kh, kw) units outer, 16-channel chunks inner).  Per kernel row
// kh the CTA stages that input row of its 32 rows (WP x 128 B each, 16-byte chunks XOR-swizzled by position so that
// ldmatrix's eight rows hit distinct banks) and the KW1 weight units of kh.
template <typename JOBS>
struct Lc1Params {
  JOBS p;
  const __nv_bfloat16* ring0; int cap0;   // [S][cap0][WP][64]
  const __nv_bfloat16* edge0;             // [S K][4][WP][64]
  const __nv_bfloat16* w1;                // [KH1*KW1][4][2][64][8]
  const float* b1;
  __nv_bfloat16* ring1; int cap1;         // [S][cap1][512]
  __nv_bfloat16* edge1;                   // [S K][4][512]
  int H0, WP, KH1, KW1, H1;
};

template <typename JOBS>
__device__ __forceinline__ const __nv_bfloat16* lc1_in(const Lc1Params<JOBS>& q, const LcJob& J, int kh) {
  const __nv_bfloat16* ring = q.ring0 + (int64_t)J.s * q.cap0 * q.WP * 64;
  if (J.stream) return ring + (int64_t)lc_mod(J.row + kh, q.cap0) * q.WP * 64;
  const int t = lc_win_row(J, q.H1) + kh;
  if (t < 2) return q.edge0 + (J.slot * 4 + t) * q.WP * 64;
  if (t >= q.H0 - 2) return q.edge0 + (J.slot * 4 + t - q.H0 + 4) * q.WP * 64;
  return ring + (int64_t)lc_mod(J.row * q.p.m + t, q.cap0) * q.WP * 64;
}

template <typename JOBS>
__global__ void __launch_bounds__(kLc1Threads)
live_cnn_conv1_kernel(const Lc1Params<JOBS> q) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if constexpr (JOBS::kRagged) {
    if ((int64_t)blockIdx.x * kLc1Jobs >= lc_total(q.p)) return;
  }
  const int row_bytes = q.WP * 128;
  unsigned char* s_a = smem;                                   // [32][WP][128 B]
  unsigned char* s_w = smem + kLc1Jobs * row_bytes;            // [KW1][4][2][64][16 B]
  const __nv_bfloat16** s_ptr = reinterpret_cast<const __nv_bfloat16**>(s_w + q.KW1 * 8192);   // [32]
  const int64_t job0 = (int64_t)blockIdx.x * kLc1Jobs;
  float c[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[mt][nt][i] = 0.f;
  const int mi = lane >> 3, l8 = lane & 7;
  const uint32_t a_s = lc_smem(s_a), w_s = lc_smem(s_w);
  const uint32_t b_base = w_s + (uint32_t)((((mi & 1) * 64) + (mi >> 1) * 8 + l8) * 16);
  LcJob mine{};   // threads 0..31: the row this thread stages pointers for
  if (tid < kLc1Jobs) mine = lc_job(q.p, job0 + tid < lc_total(q.p) ? job0 + tid : lc_total(q.p) - 1, q.H1);
  for (int kh = 0; kh < q.KH1; ++kh) {
    __syncthreads();   // the previous kernel row's operands are consumed
    if (tid < kLc1Jobs) s_ptr[tid] = lc1_in(q, mine, kh);
    __syncthreads();
    const int chunks = kLc1Jobs * q.WP * 8;
    for (int i = tid; i < chunks; i += kLc1Threads) {
      const int jb = i / (q.WP * 8), rem = i - jb * q.WP * 8, p = rem >> 3, ch = rem & 7;
      cp_async16(a_s + (uint32_t)(jb * row_bytes + p * 128 + ((ch ^ (p & 7)) << 4)), s_ptr[jb] + p * 64 + ch * 8);
    }
    const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(q.w1) + (size_t)kh * q.KW1 * 8192;
    for (int i = tid; i < q.KW1 * 512; i += kLc1Threads) cp_async16(w_s + (uint32_t)(i * 16), wsrc + (size_t)i * 16);
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    for (int kw = 0; kw < q.KW1; ++kw) {
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        uint32_t b[8][2];
#pragma unroll
        for (int np = 0; np < 4; ++np)
          ldsm_x4(b_base + (uint32_t)(((kw * 4 + kc) * 128 + np * 16) * 16), b[2 * np][0], b[2 * np][1],
                  b[2 * np + 1][0], b[2 * np + 1][1]);
        const int p = l8 + kw, ch = 2 * kc + (mi >> 1);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const int jb = 4 * warp + 2 * mt + (mi & 1);
          uint32_t a[4];
          ldsm_x4(a_s + (uint32_t)(jb * row_bytes + p * 128 + ((ch ^ (p & 7)) << 4)), a[0], a[1], a[2], a[3]);
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) lc_mma(c[mt][nt], a, b[nt][0], b[nt][1]);
        }
      }
    }
  }
  const int gq = lane >> 2, tq = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t job = job0 + 4 * warp + 2 * mt + h;
      if (job >= lc_total(q.p)) continue;
      const LcJob J = lc_job(q.p, job, q.H1);
      __nv_bfloat16* out = J.stream ? q.ring1 + ((int64_t)J.s * q.cap1 + lc_mod(J.row, q.cap1)) * kLcRow1
                                    : q.edge1 + (J.slot * 4 + J.e) * kLcRow1;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int co = nt * 8 + 2 * tq;
        const float vx = c[mt][nt][2 * h] + __ldg(q.b1 + co), vy = c[mt][nt][2 * h + 1] + __ldg(q.b1 + co + 1);
        *reinterpret_cast<uint32_t*>(out + (co >> 4) * 128 + gq * 16 + (co & 15)) = lc_pack_relu(vx, vy);
      }
    }
}

// Ragged pushes: stream s's number of new stream rows of each convolution, m (floor((c' - W) / H) - floor((c - W) / H))
// (the row rule above), into counts[s]; counts[S] = 0, so that the exclusive scan of counts[0 .. S] ends in the total.
__global__ void live_cnn_ragged_rows_kernel(const int64_t* __restrict__ count, const int* __restrict__ len, int S,
                                            int window, int shift, int m, int64_t* __restrict__ counts) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) {
    const int64_t c = count[s];
    counts[s] = m * (lc_floor_div(c - window, shift) - lc_floor_div(c - len[s] - window, shift));
  } else if (s == S) {
    counts[S] = 0;
  }
}

// Warm-up slots (window index < 0) get all-zero logits.
__global__ void live_cnn_zero_warmup_kernel(float* __restrict__ logits, LcPush p, int n_labels) {
  const int64_t slot = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (slot >= (int64_t)p.S * p.K) return;
  const int s = (int)(slot / p.K);
  if (p.first_window(s) + (slot - (int64_t)s * p.K) < 0)
    for (int i = 0; i < n_labels; ++i) logits[slot * n_labels + i] = 0.f;
}

}  // namespace kws

using namespace kws;

// ---------------------------------------------------------------------------------------------
// host side

struct kws_live_cnn {
  kws_live_t* live = nullptr;
  TcCnn* plan = nullptr;        // this state's copy of the model's plan and packed weights
  TcCnnView v{};
  int S = 0, window = 0, shift = 0, max_push = 0, n_mels = 0, cap0 = 0, cap1 = 0;
  void* dev = nullptr;
  float* edges = nullptr;         // [S Kmax][4][n_mels]
  __nv_bfloat16 *ring0 = nullptr, *edge0 = nullptr, *ring1 = nullptr, *edge1 = nullptr;
  float* partial = nullptr;       // [8][S Kmax][32]
  size_t smem0 = 0, smem1 = 0;
};

namespace {
struct LcLayout {
  TcCnnView v;
  int n_mels, cap0, cap1;
  size_t o_ring0, o_edge0, o_ring1, o_edge1, o_partial, total;   // this state's own allocation
  size_t live_bytes;
};

int lc_layout(const char* who, const kws_model_t* m, const kws_frontend_t* fe, int S, int window, int shift,
              int max_push, LcLayout* L) {
  KWS_REQUIRE(m != nullptr, "%s: model is null", who);
  KWS_REQUIRE(fe != nullptr, "%s: frontend is null", who);
  bool weights_set = false;
  const TcCnn* tc = model_tc_cnn(m, &weights_set);
  if (tc == nullptr) {
    set_error("%s: the model is not a CNN (live states of ResNets recompute every window: see LiveStreams.push)", who);
    return KWS_ERR_UNSUPPORTED;
  }
  if (!tc_cnn_view(tc, &L->v)) {
    const char* why = "";
    tc_cnn_supported(tc, &why);
    set_error("%s: the CNN has no bf16 tensor-core path (%s)", who, why);
    return KWS_ERR_UNSUPPORTED;
  }
  const TcCnnGeom& g = L->v.g;
  KWS_REQUIRE(weights_set, "%s: the model's weights were never set", who);
  L->live_bytes = kws_live_state_bytes(fe, S, window, shift, max_push);
  if (L->live_bytes == 0) {   // kws_live_create's refusals, with its message
    kws_live_t* probe = nullptr;
    const int st = kws_live_create(fe, S, window, shift, max_push, &probe);
    if (probe) kws_live_destroy(probe);
    if (st != KWS_OK) return st;
  }
  if (window >= 1 && 1 + window / 160 != g.T) {
    set_error("%s: a window of %d samples has %d frames, the CNN was built for %d", who, window, 1 + window / 160, g.T);
    return KWS_ERR_UNSUPPORTED;
  }
  if (g.H1 < 4 || g.WP > 16 || g.KW1 > 9) {
    set_error("%s: the CNN's maps are outside what the live row kernels take (H1 >= 4, pooled width <= 16)", who);
    return KWS_ERR_UNSUPPORTED;
  }
  L->n_mels = kws_frontend_n_mels(fe);
  KWS_REQUIRE(L->n_mels == g.F, "%s: the front-end gives %d features per frame, the CNN takes %d", who, L->n_mels, g.F);
  const int P = max_push / 160;
  L->cap0 = P + g.H0;
  L->cap1 = P + g.H1;
  const int64_t slots = (int64_t)S * (max_push / shift);
  const size_t row0 = (size_t)g.WP * 64 * 2, row1 = (size_t)kLcRow1 * 2;
  size_t off = round_up<size_t>((size_t)slots * 4 * L->n_mels * sizeof(float), 256);   // edges
  L->o_ring0 = off; off += round_up<size_t>((size_t)S * L->cap0 * row0, 256);
  L->o_edge0 = off; off += round_up<size_t>((size_t)slots * 4 * row0, 256);
  L->o_ring1 = off; off += round_up<size_t>((size_t)S * L->cap1 * row1, 256);
  L->o_edge1 = off; off += round_up<size_t>((size_t)slots * 4 * row1, 256);
  L->o_partial = off; off += round_up<size_t>((size_t)kTcCnnLin0Split * slots * 32 * sizeof(float), 256);
  L->total = off;
  return KWS_OK;
}
}  // namespace

extern "C" size_t kws_live_cnn_state_bytes(const kws_model_t* m, const kws_frontend_t* fe, int n_streams, int window,
                                           int shift, int max_push) {
  LcLayout L;
  if (lc_layout("kws_live_cnn_state_bytes", m, fe, n_streams, window, shift, max_push, &L) != KWS_OK) return 0;
  return L.live_bytes + L.v.blob_bytes + L.total;
}

extern "C" void kws_live_cnn_destroy(kws_live_cnn_t* lc) {
  if (!lc) return;
  if (lc->live) kws_live_destroy(lc->live);
  if (lc->plan) tc_cnn_destroy(lc->plan);
  if (lc->dev) cudaFree(lc->dev);
  delete lc;
}

extern "C" int kws_live_cnn_create(const kws_model_t* m, const kws_frontend_t* fe, int n_streams, int window, int shift,
                                   int max_push, kws_live_cnn_t** out) {
  KWS_REQUIRE(out != nullptr, "kws_live_cnn_create: out is null");
  *out = nullptr;
  LcLayout L;
  KWS_TRY(lc_layout("kws_live_cnn_create", m, fe, n_streams, window, shift, max_push, &L));
  bool weights_set = false;
  kws_live_cnn* lc = new kws_live_cnn();
  lc->S = n_streams; lc->window = window; lc->shift = shift; lc->max_push = max_push;
  lc->n_mels = L.n_mels; lc->cap0 = L.cap0; lc->cap1 = L.cap1;
  int st = kws_live_create(fe, n_streams, window, shift, max_push, &lc->live);
  if (st == KWS_OK) st = tc_cnn_copy(model_tc_cnn(m, &weights_set), &lc->plan, nullptr);
  if (st == KWS_OK) {
    tc_cnn_view(lc->plan, &lc->v);
    cudaError_t e = cudaMalloc(&lc->dev, L.total);
    if (e == cudaSuccess) e = cudaMemset(lc->dev, 0, L.total);   // rows are never read stale by a valid window; zero
    if (e == cudaSuccess) e = cudaDeviceSynchronize();           // keeps them finite (and the weight copy is done)
    const TcCnnGeom& g = lc->v.g;
    lc->smem0 = (size_t)g.ks0 * 2048 + (size_t)kLc0Warps * 3 * 2 * g.ks0 * 256;
    lc->smem1 = (size_t)kLc1Jobs * g.WP * 128 + (size_t)g.KW1 * 8192 + kLc1Jobs * sizeof(void*);
    if (e == cudaSuccess) e = raise_dynamic_smem(live_cnn_conv0_kernel<LcPush>, lc->smem0);
    if (e == cudaSuccess) e = raise_dynamic_smem(live_cnn_conv1_kernel<LcPush>, lc->smem1);
    if (e == cudaSuccess) e = raise_dynamic_smem(live_cnn_conv0_kernel<LcRagged>, lc->smem0);
    if (e == cudaSuccess) e = raise_dynamic_smem(live_cnn_conv1_kernel<LcRagged>, lc->smem1);
    if (e != cudaSuccess) {
      set_error("kws_live_cnn_create: %zu bytes of device state: %s", L.total, cudaGetErrorString(e));
      st = KWS_ERR_CUDA;
    }
  }
  if (st != KWS_OK) {
    kws_live_cnn_destroy(lc);
    return st;
  }
  unsigned char* d = static_cast<unsigned char*>(lc->dev);
  lc->edges = reinterpret_cast<float*>(d);
  lc->ring0 = reinterpret_cast<__nv_bfloat16*>(d + L.o_ring0);
  lc->edge0 = reinterpret_cast<__nv_bfloat16*>(d + L.o_edge0);
  lc->ring1 = reinterpret_cast<__nv_bfloat16*>(d + L.o_ring1);
  lc->edge1 = reinterpret_cast<__nv_bfloat16*>(d + L.o_edge1);
  lc->partial = reinterpret_cast<float*>(d + L.o_partial);
  *out = lc;
  return KWS_OK;
}

extern "C" int kws_live_cnn_reset(kws_live_cnn_t* lc, const int64_t* stream_ids, int64_t count, void* stream) {
  KWS_REQUIRE(lc != nullptr, "kws_live_cnn_reset: live CNN state is null");
  return kws_live_reset(lc->live, stream_ids, count, stream);
}

template <typename SMP>
static int live_cnn_push_any(const char* who, kws_live_cnn_t* lc, const SMP* chunk, int n, float* logits,
                             void* stream) {
  KWS_REQUIRE(lc != nullptr, "%s: live CNN state is null", who);
  KWS_REQUIRE(logits != nullptr, "%s: null buffer", who);
  cudaStream_t st = as_stream(stream);
  KWS_TRY(live_append_rows(who, lc->live, chunk, n, st));
  const TcCnnGeom& g = lc->v.g;
  const int K = n / lc->shift;
  const int64_t slots = (int64_t)lc->S * K;
  LcPush p{lc->live->count, lc->S, n, lc->window, lc->shift, K, lc->shift / 160, n / 160, 0};
  p.jobs = (int64_t)lc->S * p.P + 4 * slots;
  KWS_TRY(live_edge_frames(lc->live, n, lc->edges, st));
  Lc0Params<LcPush> q0{p, lc->live->frames, lc->live->fcap, lc->edges, lc->v.w0, lc->v.b0, lc->ring0, lc->cap0, lc->edge0,
               g.T, g.F, g.KH0, g.H0, g.WP, g.ks0};
  live_cnn_conv0_kernel<<<(unsigned)ceil_div<int64_t>(p.jobs, kLc0Warps), 32 * kLc0Warps, lc->smem0, st>>>(q0);
  KWS_CHECK_LAUNCH();
  Lc1Params<LcPush> q1{p, lc->ring0, lc->cap0, lc->edge0, lc->v.w1, lc->v.b1, lc->ring1, lc->cap1, lc->edge1,
               g.H0, g.WP, g.KH1, g.KW1, g.H1};
  live_cnn_conv1_kernel<<<(unsigned)ceil_div<int64_t>(p.jobs, kLc1Jobs), kLc1Threads, lc->smem1, st>>>(q1);
  KWS_CHECK_LAUNCH();
  const LiveActRows rows{lc->ring1, lc->edge1, lc->live->count, n, lc->window, lc->shift, K, lc->cap1, g.H1};
  KWS_TRY(tc_cnn_live_linear(lc->plan, rows, slots, lc->partial, logits, st));
  live_cnn_zero_warmup_kernel<<<(unsigned)ceil_div<int64_t>(slots, 256), 256, 0, st>>>(logits, p, lc->v.n_labels);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

extern "C" int kws_live_cnn_push(kws_live_cnn_t* lc, const float* chunk, int n, float* logits, void* stream) {
  return live_cnn_push_any<float>("kws_live_cnn_push", lc, chunk, n, logits, stream);
}

extern "C" int kws_live_cnn_push_pcm16(kws_live_cnn_t* lc, const int16_t* chunk, int n, float* logits, void* stream) {
  return live_cnn_push_any<int16_t>("kws_live_cnn_push_pcm16", lc, chunk, n, logits, stream);
}

// ---- ragged pushes ----------------------------------------------------------------------------
// Workspace: the front-end's ragged workspace (offsets, lengths, its plan), then the per-stream stream-row counts
// i64[S+1], their exclusive scan i64[S+1] and CUB's scan scratch.
namespace {
struct LcRaggedLayout {
  size_t o_rows, o_temp, temp, total;
};

int lc_ragged_layout(const char* who, const kws_live_cnn* lc, LcRaggedLayout* R) {
  const size_t plan = round_up<size_t>((size_t)(lc->S + 1) * sizeof(int64_t), 256);
  R->o_rows = plan;
  R->o_temp = 2 * plan;
  R->temp = 0;
  const cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, R->temp, static_cast<int64_t*>(nullptr),
                                                      static_cast<int64_t*>(nullptr), lc->S + 1);
  if (e != cudaSuccess) {
    set_error("%s: scan size query failed: %s", who, cudaGetErrorString(e));
    return KWS_ERR_CUDA;
  }
  R->total = R->o_temp + R->temp;
  return KWS_OK;
}
}  // namespace

extern "C" size_t kws_live_cnn_ragged_workspace_bytes(const kws_live_cnn_t* lc) {
  const char* who = "kws_live_cnn_ragged_workspace_bytes";
  if (lc == nullptr) {
    set_error("%s: live CNN state is null", who);
    return 0;
  }
  LcRaggedLayout R;
  if (lc_ragged_layout(who, lc, &R) != KWS_OK) return 0;
  return live_ragged_workspace_bytes(who, lc->live, R.total);
}

template <typename SMP>
static int live_cnn_push_ragged_any(const char* who, kws_live_cnn_t* lc, const SMP* samples, const int32_t* lengths,
                                    float* logits, int64_t* win_stream, int64_t* win_index, int64_t capacity,
                                    int64_t* n_windows, void* workspace, size_t ws_bytes, void* stream) {
  KWS_REQUIRE(lc != nullptr, "%s: live CNN state is null", who);
  LcRaggedLayout X;
  KWS_TRY(lc_ragged_layout(who, lc, &X));
  cudaStream_t st = as_stream(stream);
  kws_live_t* L = lc->live;
  // the whole push is checked on the host first; then the samples, the front-end's plan and the new frame-table rows
  LiveRagged P;
  KWS_TRY(live_ragged_append_rows(who, L, samples, lengths, capacity, logits, "logits", workspace, ws_bytes, X.total, st,
                                  &P));
  unsigned char* x = static_cast<unsigned char*>(P.extra);
  int64_t* counts = reinterpret_cast<int64_t*>(x);
  int64_t* rows = reinterpret_cast<int64_t*>(x + X.o_rows);
  const int m = lc->shift / 160;
  // the stream-row plan: where each stream's new convolution rows start in the job list, and their total
  live_cnn_ragged_rows_kernel<<<(unsigned)ceil_div(lc->S + 1, 256), 256, 0, st>>>(L->count, P.len, lc->S, lc->window,
                                                                                  lc->shift, m, counts);
  KWS_CHECK_LAUNCH();
  size_t temp = X.temp;
  KWS_CUDA(cub::DeviceScan::ExclusiveSum(x + X.o_temp, temp, counts, rows, lc->S + 1, st));
  // edge frames of the completed windows; conv_0 and conv_1 rows (stream rows even when no window completes: warm-up);
  // the Linear layers.  Launches are sized by the host's bounds, m + 4 jobs and one window per ceil(n_s / shift).
  KWS_TRY(live_ragged_edge_frames(L, P, lc->edges, st));
  const TcCnnGeom& g = lc->v.g;
  const LcRagged p{L->count, P.len, rows, P.plan, lc->S, lc->window, lc->shift, m, win_stream, win_index, n_windows};
  const int64_t job_bound = (int64_t)(m + 4) * P.win_bound;
  Lc0Params<LcRagged> q0{p, L->frames, L->fcap, lc->edges, lc->v.w0, lc->v.b0, lc->ring0, lc->cap0, lc->edge0,
                         g.T, g.F, g.KH0, g.H0, g.WP, g.ks0};
  // (one CTA even when nothing is pushed: it writes *n_windows)
  live_cnn_conv0_kernel<<<(unsigned)std::max<int64_t>(ceil_div<int64_t>(job_bound, kLc0Warps), 1), 32 * kLc0Warps,
                          lc->smem0, st>>>(q0);
  KWS_CHECK_LAUNCH();
  if (P.win_bound == 0) return KWS_OK;
  Lc1Params<LcRagged> q1{p, lc->ring0, lc->cap0, lc->edge0, lc->v.w1, lc->v.b1, lc->ring1, lc->cap1, lc->edge1,
                         g.H0, g.WP, g.KH1, g.KW1, g.H1};
  live_cnn_conv1_kernel<<<(unsigned)ceil_div<int64_t>(job_bound, kLc1Jobs), kLc1Threads, lc->smem1, st>>>(q1);
  KWS_CHECK_LAUNCH();
  const RaggedActRows act{lc->ring1, lc->edge1, L->count, P.len, P.plan, lc->S, lc->window, lc->shift, lc->cap1, g.H1};
  return tc_cnn_live_linear(lc->plan, act, P.win_bound, lc->partial, logits, st);
}

extern "C" int kws_live_cnn_push_ragged(kws_live_cnn_t* lc, const float* samples, const int32_t* lengths, float* logits,
                                        int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                                        void* workspace, size_t ws_bytes, void* stream) {
  return live_cnn_push_ragged_any<float>("kws_live_cnn_push_ragged", lc, samples, lengths, logits, win_stream,
                                         win_index, capacity, n_windows, workspace, ws_bytes, stream);
}

extern "C" int kws_live_cnn_push_ragged_pcm16(kws_live_cnn_t* lc, const int16_t* samples, const int32_t* lengths,
                                              float* logits, int64_t* win_stream, int64_t* win_index, int64_t capacity,
                                              int64_t* n_windows, void* workspace, size_t ws_bytes, void* stream) {
  return live_cnn_push_ragged_any<int16_t>("kws_live_cnn_push_ragged_pcm16", lc, samples, lengths, logits, win_stream,
                                           win_index, capacity, n_windows, workspace, ws_bytes, stream);
}
