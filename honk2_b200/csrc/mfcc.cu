// Fused MFCC front-end for sm_100a: reflect-pad framing, periodic Hann window, 480-point real
// STFT, power, Slaney mel filterbank, ln, and the reference's degenerate "DCT" (x2), one kernel.
//
// Replaces AudioProcessor.compute_mfccs (/root/reference/utils/audio_processor.py:18-30) for a
// whole batch (the collate loop of data_loader/audio_data_loader.py:26-29).
//
// Algorithm (fp32 throughout): the 480-point real DFT of a windowed frame is computed as a
// 240-point complex FFT of z[m] = x[2m] + i x[2m+1], factored 240 = 16 x 15 (Cooley-Tukey):
// 15 lanes each run a radix-2^4 FFT in registers, twiddle by W240^(n2 k1), exchange through
// shared memory, 16 lanes each run a 15-point DFT (conjugate-pair form, constant twiddles),
// then the real-FFT split recovers bins 0..239, |X|^2, sparse triangular mel weights, 2*ln.
// A warp works on two frames at a time (one per half-warp); a CTA stages the 2880 samples its
// 16 frames cover once (coalesced loads, reflect indexing at the clip edges).
#include "common.cuh"
#include "live.cuh"
#include <cub/device/device_scan.cuh>
#include <cmath>
#include <vector>
#include <cstring>
#include <type_traits>

namespace kws {

constexpr int kNfft = 480;
constexpr int kHop = 160;
constexpr int kNz = 240;            // complex FFT length
constexpr int kScStride = kNz + 8;   // per-frame scratch pitch (float2): 496 words = 16 banks off, so the two half-warps (two
                                     // frames) of a warp hit disjoint bank halves in the 32-bit phases (power / mel)
constexpr int kTwA = 16 * 16;        // stage-A twiddles, [k1][lane] (lane-contiguous: no bank conflicts)
constexpr int kFramesPerCta = 16;
constexpr int kMfccThreads = 256;
constexpr int kStageSamples = (kFramesPerCta - 1) * kHop + kNfft;  // 2880
constexpr int kEdgeStageSamples = kFramesPerCta * kNfft;            // 7680: every frame slot stages its own 480 samples
constexpr int kMaxMels = 64;

struct FrontendTables {
  const float* window;    // [480]
  const float2* tw240;    // [16][16] stage-A twiddles W240^(l k1) = (cos, -sin)(2 pi l k1 / 240) at [k1 * 16 + l]
  const float2* tw480;    // [240] (sin, cos)(2 pi k / 480)
  const int* mel_lo;      // [n_mels] first bin
  const int* mel_cnt;     // [n_mels] number of bins
  const int* mel_off;     // [n_mels] offset into mel_w
  const float* mel_w;     // [nnz]
  int n_mels, nnz, nb16;  // nb16: number of 16-bin groups to evaluate (bins 0..16*nb16-1)
};

struct Frontend {
  int sr, n_mels, n_fft, hop;
  float f_min, f_max;
  void* dev_blob = nullptr;
  FrontendTables t{};
  size_t smem_bytes = 0;         // batch kernel
  size_t smem_bytes_edges = 0;   // window-edge kernel of the streaming front-end
};

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// radix-2 decimation-in-frequency FFT of 16 complex values held in registers; on return
// x[i] holds X[bitrev4(i)].
__device__ __forceinline__ void fft16_dif(float2 (&x)[16]) {
  constexpr float c16[8] = {1.f, 0.923879533f, 0.707106781f, 0.382683432f,
                            0.f, -0.382683432f, -0.707106781f, -0.923879533f};
  constexpr float s16[8] = {0.f, 0.382683432f, 0.707106781f, 0.923879533f,
                            1.f, 0.923879533f, 0.707106781f, 0.382683432f};
#pragma unroll
  for (int len = 16; len >= 2; len >>= 1) {
    const int half = len >> 1;
    const int step = 16 / len;
#pragma unroll
    for (int base = 0; base < 16; base += len) {
#pragma unroll
      for (int j = 0; j < half; ++j) {
        float2 u = x[base + j], v = x[base + j + half];
        x[base + j] = make_float2(u.x + v.x, u.y + v.y);
        float2 t = make_float2(u.x - v.x, u.y - v.y);
        const int tw = j * step;  // W16^tw = (c, -s)
        if (tw == 0) {
          x[base + j + half] = t;
        } else if (tw == 4) {
          x[base + j + half] = make_float2(t.y, -t.x);
        } else {
          x[base + j + half] = make_float2(t.x * c16[tw] + t.y * s16[tw], t.y * c16[tw] - t.x * s16[tw]);
        }
      }
    }
  }
}

__host__ __device__ constexpr int bitrev4(int i) {
  return ((i & 1) << 3) | ((i & 2) << 1) | ((i & 4) >> 1) | ((i & 8) >> 3);
}

// 15-point DFT, Z[k] = sum_n y[n] exp(-2 pi i n k / 15), conjugate-pair form.
__device__ __forceinline__ void dft15(const float2 (&y)[15], float2 (&z)[15]) {
  constexpr float c15[15] = {1.f, 0.913545458f, 0.669130606f, 0.309016994f, -0.104528463f,
                             -0.5f, -0.809016994f, -0.978147601f, -0.978147601f, -0.809016994f,
                             -0.5f, -0.104528463f, 0.309016994f, 0.669130606f, 0.913545458f};
  constexpr float s15[15] = {0.f, 0.406736643f, 0.743144825f, 0.951056516f, 0.994521895f,
                             0.866025404f, 0.587785252f, 0.207911691f, -0.207911691f, -0.587785252f,
                             -0.866025404f, -0.994521895f, -0.951056516f, -0.743144825f, -0.406736643f};
  float2 a[8], b[8];
#pragma unroll
  for (int j = 1; j <= 7; ++j) {
    a[j] = make_float2(y[j].x + y[15 - j].x, y[j].y + y[15 - j].y);
    b[j] = make_float2(y[j].x - y[15 - j].x, y[j].y - y[15 - j].y);
  }
  float2 s0 = y[0];
#pragma unroll
  for (int j = 1; j <= 7; ++j) { s0.x += a[j].x; s0.y += a[j].y; }
  z[0] = s0;
#pragma unroll
  for (int k = 1; k <= 7; ++k) {
    float2 A = y[0], Bv = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 1; j <= 7; ++j) {
      const int idx = (j * k) % 15;
      A.x = fmaf(c15[idx], a[j].x, A.x);
      A.y = fmaf(c15[idx], a[j].y, A.y);
      Bv.x = fmaf(s15[idx], b[j].x, Bv.x);
      Bv.y = fmaf(s15[idx], b[j].y, Bv.y);
    }
    // Z[k] = A - i B ; Z[15-k] = A + i B
    z[k] = make_float2(A.x + Bv.y, A.y - Bv.x);
    z[15 - k] = make_float2(A.x - Bv.y, A.y + Bv.x);
  }
}

// EDGES = false: a CTA computes 16 consecutive frames of one clip (SRC says where the clip's samples are).
// EDGES = true (streaming front-ends): a CTA computes the four frames of four windows that touch the reflect padding
// (t = 0, 1, T-2, T-1); every other frame of a window is shared with the stream-level frame table.
//
// SMP = float: waveforms as the reference's loader hands them over (librosa float32 in [-1, 1)).  SMP = int16_t: the 16-bit
// PCM samples as they sit in the wav files (dataset/gsc_dataset.py:169 loads them through librosa, which returns exactly
// s / 32768): converted while staging, bit-identical features, half the bytes from the host and from HBM.
__device__ __forceinline__ float smp_ld(const float* p) { return __ldg(p); }
__device__ __forceinline__ float smp_ld(const int16_t* p) { return (float)__ldg(p) * (1.f / 32768.f); }

// Sample sources of mfcc_kernel's two staging loops: where sample j of clip b comes from and where frame t of clip b
// goes.  clip(b) is what the loops index from; ptr(w, j) addresses sample j of that clip (EDGES: of window b + wi via
// edge_ptr).  kReflect: librosa's reflect padding at the clip edges applies in the tile loop, so it needs bounds checks.
// kRagged: the number of entries lives on the device (entries()), and CTAs past it exit.  kPacked: a CTA computes 16
// single frames from anywhere (frame_ptr / frame_out), each staged from its own 480 samples like the edge frames.
//
// DenseSource: clip b is wav + b * stride (stride = N for a dense [B, N] batch, = the shift for the overlapping windows
// of a stream); features are dense [B, T, n_mels].
template <typename SMP>
struct DenseSource {
  static constexpr bool kReflect = true, kRagged = false, kPacked = false;
  using Clip = const SMP*;
  const SMP* __restrict__ wav;
  int64_t stride;
  __device__ __forceinline__ Clip clip(int64_t b) const { return wav + b * stride; }
  __device__ __forceinline__ const SMP* ptr(Clip w, int j) const { return w + j; }
  __device__ __forceinline__ const SMP* edge_ptr(Clip w, int64_t, int wi, int j) const {
    return w + (int64_t)wi * stride + j;
  }
  __device__ __forceinline__ float* out_row(float* feat, int64_t b, int T, int t, int n_mels) const {
    return feat + (b * (int64_t)T + t) * n_mels;
  }
};

__host__ __device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) {   // b > 0
  return a >= 0 ? a / b : -((-a + b - 1) / b);
}
__device__ __forceinline__ int64_t pos_mod(int64_t a, int64_t m) { const int64_t r = a % m; return r < 0 ? r + m : r; }
// At sample count c of a live stream: the last complete frame-table row (row r covers samples [160 r - 240, +480)),
// and the number of complete windows (window k covers [k shift, k shift + window)).  A push from c to c' completes rows
// ragged_rows(c) + 1 .. ragged_rows(c') and windows ragged_wins(c) .. ragged_wins(c') - 1.
__device__ __forceinline__ int64_t ragged_rows(int64_t c) { return floor_div(c - kNfft / 2, kHop); }
__device__ __forceinline__ int64_t ragged_wins(int64_t c, int window, int shift) {
  const int64_t k = floor_div(c - window, shift) + 1;
  return k > 0 ? k : 0;
}

// RingSource (live streams): stream s's samples sit in a float ring of `cap` samples (a multiple of 16, so a 16-byte
// load at a multiple of 4 samples never straddles the wrap), sample p at ring[s][p mod cap], p counted from the
// stream's last reset.  count[s] includes the current push of n samples; wpos[s] is the ring position of the start of
// the push's first window (both written by live_append_kernel).  A span is a ring and the ring position of its sample
// 0; at() takes j in [-cap, cap).
//  EDGES = false: clip b is stream b's new frame-table rows r0 = c_old/160 - 1 ...: clip sample j is stream sample
//                 160 r0 + j, read as is (no padding); frame t goes to frame-ring row (r0 + t) mod fcap of stream b.
//  EDGES = true:  window slot b = (stream b / K, the push's window b % K of that stream).  A CTA's clip holds the spans
//                 of its four slots b .. b+3, found once per CTA; features are dense [S K, T, n_mels] like DenseSource's.
template <bool EDGES>
struct RingSource {
  static constexpr bool kReflect = false, kRagged = false, kPacked = false;
  struct Span { const float* ring; int start; };
  struct Slots { Span w[4]; };
  using Clip = std::conditional_t<EDGES, Slots, Span>;
  const float* __restrict__ ring;
  const int64_t* __restrict__ count;
  const int* __restrict__ wpos;
  int cap, n, fcap, shift, K, slots;
  __device__ __forceinline__ const float* addr(const Span& w, int j) const {
    int p = w.start + j;
    if (p < 0) p += cap;
    else if (p >= cap) p -= cap;
    return w.ring + p;
  }
  __device__ __forceinline__ Span slot_span(int slot) const {
    const int s = slot / K;
    int start = wpos[s] + (slot - s * K) * shift;   // (< 2 cap: wpos < cap, K shift = n <= cap)
    if (start >= cap) start -= cap;
    return {ring + (int64_t)s * cap, start};
  }
  __device__ __forceinline__ Clip clip(int64_t b) const {
    if constexpr (EDGES) {
      Slots c;
#pragma unroll
      for (int q = 0; q < 4; ++q) c.w[q] = slot_span(min((int)b + q, slots - 1));   // (slots past the end: unused)
      return c;
    } else {
      return {ring + b * cap, (int)pos_mod(count[b] - n - kHop, cap)};
    }
  }
  __device__ __forceinline__ const float* ptr(const Span& w, int j) const { return addr(w, j); }
  __device__ __forceinline__ const float* edge_ptr(const Slots& c, int64_t, int wi, int j) const {
    Span w = c.w[0];
#pragma unroll
    for (int q = 1; q < 4; ++q)
      if (wi == q) w = c.w[q];   // (a select: the spans stay in registers)
    return addr(w, j);
  }
  __device__ __forceinline__ float* out_row(float* feat, int64_t b, int T, int t, int n_mels) const {
    if constexpr (EDGES) {
      return feat + (b * (int64_t)T + t) * n_mels;
    } else {
      const int64_t r = (count[b] - n) / kHop - 1 + t;
      return feat + (b * (int64_t)fcap + pos_mod(r, fcap)) * n_mels;
    }
  }
};

// EdgeRingSource (kws_live_cnn): RingSource<true>'s window slots, but only the four edge frames of a slot are stored,
// dense [S K][4][n_mels] (frames t = 0, 1, T-2, T-1 in that order).
struct EdgeRingSource : RingSource<true> {
  __device__ __forceinline__ float* out_row(float* feat, int64_t b, int T, int t, int n_mels) const {
    return feat + (b * 4 + (t < 2 ? t : t - T + 4)) * n_mels;
  }
};

// RaggedSource (ragged pushes): entries of two compacted lists ordered by stream, each stream with its own count.
// plan[s] (s = 0 .. S) is the exclusive scan of the per-stream counts of the push, new frame-table rows in the high 32
// bits and completed windows in the low 32 bits (both totals < 2^31, checked on the host): plan[S] holds the totals.  An
// entry's stream is a binary search over plan, done once per entry by the first threads of the CTA into a shared table
// (clip() holds one barrier, so every thread calls it).  count[s] already includes the push's len[s] samples.
//  EDGES = false (kPacked): row entry e = (stream s, row r = floor((c_old - 240) / 160) + 1 + e - plan_rows[s]); frame t
//                 of the CTA is entry 16 b + t: ring samples 160 r - 240 + [0, 480) (a multiple of 16 samples from the
//                 ring start, so 16-byte loads), written to row r mod fcap of stream s's frame ring.
//  EDGES = true:  window entry b = (stream s, window k = max(0, floor((c_old - W) / H) + 1) + b - plan_wins[s]): the
//                 spans of RingSource<true>, features dense [M, T, n_mels].
template <bool EDGES>
struct RaggedSource {
  static constexpr bool kReflect = false, kRagged = true, kPacked = !EDGES;
  using Span = RingSource<true>::Span;
  using Slots = RingSource<true>::Slots;
  struct Row { Span in; float* out; };
  using Clip = std::conditional_t<EDGES, Slots, const Row*>;
  const float* __restrict__ ring;
  float* frames;
  const int64_t* __restrict__ count;
  const int* __restrict__ len;
  const int64_t* __restrict__ plan;
  int S, cap, fcap, n_mels, window, shift;
  __device__ __forceinline__ int64_t field(int64_t p) const { return EDGES ? (p & 0xffffffffll) : (p >> 32); }
  __device__ __forceinline__ int64_t entries() const { return field(__ldg(plan + S)); }
  // stream of entry e (< entries()) and the entries of the streams before it
  __device__ __forceinline__ int stream_of(int64_t e, int64_t* before) const {
    int lo = 0, hi = S;   // field(plan[lo]) <= e < field(plan[hi])
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (field(__ldg(plan + mid)) <= e) lo = mid;
      else hi = mid;
    }
    *before = field(__ldg(plan + lo));
    return lo;
  }
  __device__ __forceinline__ const float* addr(const Span& w, int j) const {
    int p = w.start + j;
    if (p < 0) p += cap;
    else if (p >= cap) p -= cap;
    return w.ring + p;
  }
  __device__ __forceinline__ Clip clip(int64_t b) const {
    const int64_t last = entries() - 1;
    constexpr int kEntries = EDGES ? 4 : kFramesPerCta;
    __shared__ std::conditional_t<EDGES, Span, Row> tab[kEntries];
    if (threadIdx.x < kEntries) {
      const int64_t e = min(b + (int64_t)threadIdx.x, last);   // (entries past the end: unused)
      int64_t before;
      const int s = stream_of(e, &before);
      const int64_t c_old = __ldg(count + s) - __ldg(len + s);
      if constexpr (EDGES) {
        const int64_t k = ragged_wins(c_old, window, shift) + (e - before);
        tab[threadIdx.x] = Span{ring + (int64_t)s * cap, (int)pos_mod(k * shift, cap)};
      } else {
        const int64_t r = ragged_rows(c_old) + 1 + (e - before);
        tab[threadIdx.x] = Row{Span{ring + (int64_t)s * cap, (int)pos_mod(r * kHop - kNfft / 2, cap)},
                               frames + ((int64_t)s * fcap + pos_mod(r, fcap)) * n_mels};
      }
    }
    __syncthreads();
    if constexpr (EDGES) {
      Slots c;
#pragma unroll
      for (int q = 0; q < 4; ++q) c.w[q] = tab[q];
      return c;
    } else {
      return tab;
    }
  }
  __device__ __forceinline__ const float* edge_ptr(const Slots& c, int64_t, int wi, int j) const {
    Span w = c.w[0];
#pragma unroll
    for (int q = 1; q < 4; ++q)
      if (wi == q) w = c.w[q];
    return addr(w, j);
  }
  __device__ __forceinline__ const float* frame_ptr(const Row* c, int slot, int j) const { return addr(c[slot].in, j); }
  __device__ __forceinline__ float* frame_out(const Row* c, int slot) const { return c[slot].out; }
  __device__ __forceinline__ float* out_row(float* feat, int64_t b, int T, int t, int n_mels) const {
    return feat + (b * (int64_t)T + t) * n_mels;
  }
};

// RaggedEdgeSource (ragged pushes of kws_live_cnn): RaggedSource<true>'s windows, but only the four edge frames of a
// window are stored, dense [M][4][n_mels] (frames t = 0, 1, T-2, T-1 in that order).
struct RaggedEdgeSource : RaggedSource<true> {
  __device__ __forceinline__ float* out_row(float* feat, int64_t b, int T, int t, int n_mels) const {
    return feat + (b * 4 + (t < 2 ? t : t - T + 4)) * n_mels;
  }
};

template <bool EDGES, typename SMP, typename SRC = DenseSource<SMP>>
__global__ void __launch_bounds__(kMfccThreads)
mfcc_kernel(FrontendTables tb, SRC src, int64_t B, int N, int T, int tiles_per_utt, float* __restrict__ feat) {
  constexpr bool kPacked = SRC::kPacked;   // (T = 16: frame t of the CTA is entry 16 b + t)
  constexpr int kStage = EDGES || kPacked ? kEdgeStageSamples : kStageSamples;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* scratch = reinterpret_cast<float2*>(smem_raw);                 // [16][248]
  float2* s_tw240 = scratch + kFramesPerCta * kScStride;                 // [16][16]
  float2* s_tw480 = s_tw240 + kTwA;                                      // [240]
  float* s_wave = reinterpret_cast<float*>(s_tw480 + kNz);               // [2880] ([16][480] for EDGES)
  float* s_win = s_wave + kStage;                                        // [480]
  int* s_lo = reinterpret_cast<int*>(s_win + kNfft);                     // [64]
  int* s_cnt = s_lo + kMaxMels;
  int* s_off = s_cnt + kMaxMels;
  float* s_w = reinterpret_cast<float*>(s_off + kMaxMels);               // [nnz]

  const int tid = threadIdx.x;
  const int64_t b = EDGES ? (int64_t)blockIdx.x * 4                                  // (EDGES: first of four windows)
                          : kPacked ? (int64_t)blockIdx.x * kFramesPerCta : blockIdx.x / tiles_per_utt;
  const int t0 = EDGES || kPacked ? 0 : (blockIdx.x % tiles_per_utt) * kFramesPerCta;
  if constexpr (SRC::kRagged) {
    B = src.entries();   // (the grid covers the host's bound)
    if (b >= B) return;
  }
  const typename SRC::Clip w = src.clip(b);

  if constexpr (kPacked) {
    // frame slot s: samples [0, 480) of entry b + s's span, 16 bytes at a time (span starts are multiples of 16 samples)
    for (int iv = tid; iv < kEdgeStageSamples / 4; iv += kMfccThreads) {
      const int slot = iv / (kNfft / 4), n = (iv - slot * (kNfft / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b + slot < B) v = __ldg(reinterpret_cast<const float4*>(src.frame_ptr(w, slot, n)));
      *reinterpret_cast<float4*>(s_wave + slot * kNfft + n) = v;
    }
  } else if constexpr (EDGES) {
    // frame slot s = 4 * (window - b) + e, e -> frame t = 0, 1, T-2, T-1: samples [160 t - 240, +480) of its window
    for (int i = tid; i < kEdgeStageSamples; i += kMfccThreads) {
      const int slot = i / kNfft, n = i - slot * kNfft;
      const int wi = slot >> 2, e = slot & 3;
      const int te = e < 2 ? e : T - 4 + e;
      int j = te * kHop - kNfft / 2 + n;
      if (j < 0) j = -j;
      if (j >= N) j = 2 * (N - 1) - j;
      j = max(0, min(j, N - 1));
      s_wave[i] = b + wi < B ? smp_ld(src.edge_ptr(w, b, wi, j)) : 0.f;
    }
  } else {
    // stage: samples [160*t0 - 240, +2880) with librosa 'reflect' padding at the clip edges; only the frames that exist
    // (the last tile of a clip usually holds fewer than 16).  Interior runs are copied 16 bytes at a time.
    const int j0 = t0 * kHop - kNfft / 2;
    const int n_fr = min(kFramesPerCta, T - t0);
    const int n_stage = (n_fr - 1) * kHop + kNfft;
    // (j0 is a multiple of 16 samples; a ring source is always aligned: see RingSource)
    bool vec = true;
    if constexpr (SRC::kReflect) vec = ((reinterpret_cast<uintptr_t>(w) & 15) == 0);
    constexpr int V = 16 / (int)sizeof(SMP);   // samples per 16-byte load (n_stage is a multiple of 8)
    if (vec) {
      for (int iv = tid; iv < n_stage / V; iv += kMfccThreads) {
        const int i = iv * V, j = j0 + i;
        float e[V];
        if (!SRC::kReflect || (j >= 0 && j + V - 1 < N)) {
          const uint4 raw = __ldg(reinterpret_cast<const uint4*>(src.ptr(w, j)));
          if constexpr (sizeof(SMP) == 4) {
            e[0] = __uint_as_float(raw.x); e[1] = __uint_as_float(raw.y); e[2] = __uint_as_float(raw.z); e[3] = __uint_as_float(raw.w);
          } else {
            const uint32_t r[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              e[2 * q] = (float)(int16_t)(r[q] & 0xFFFFu) * (1.f / 32768.f);
              e[2 * q + 1] = (float)(int16_t)(r[q] >> 16) * (1.f / 32768.f);
            }
          }
        } else {
#pragma unroll
          for (int q = 0; q < V; ++q) {
            int jj = j + q;
            if (jj < 0) jj = -jj;
            if (jj >= N) jj = 2 * (N - 1) - jj;
            jj = max(0, min(jj, N - 1));  // only reachable for samples of masked frames
            e[q] = smp_ld(src.ptr(w, jj));
          }
        }
#pragma unroll
        for (int q = 0; q < V; q += 4)
          *reinterpret_cast<float4*>(s_wave + i + q) = make_float4(e[q], e[q + 1], e[q + 2], e[q + 3]);
      }
    } else {
      for (int i = tid; i < n_stage; i += kMfccThreads) {
        int j = j0 + i;
        if (j < 0) j = -j;
        if (j >= N) j = 2 * (N - 1) - j;
        j = max(0, min(j, N - 1));
        s_wave[i] = smp_ld(src.ptr(w, j));
      }
    }
  }
  for (int i = tid; i < kNfft; i += kMfccThreads) s_win[i] = tb.window[i];
  for (int i = tid; i < kNz; i += kMfccThreads) s_tw480[i] = tb.tw480[i];
  for (int i = tid; i < kTwA; i += kMfccThreads) s_tw240[i] = tb.tw240[i];
  for (int i = tid; i < tb.n_mels; i += kMfccThreads) {
    s_lo[i] = tb.mel_lo[i]; s_cnt[i] = tb.mel_cnt[i]; s_off[i] = tb.mel_off[i];
  }
  for (int i = tid; i < tb.nnz; i += kMfccThreads) s_w[i] = tb.mel_w[i];
  __syncthreads();

  const int warp = tid >> 5, lane = tid & 31;
  const int half = lane >> 4, l = lane & 15;
  const int t_local = 2 * warp + half;
  const int t = EDGES ? ((t_local & 3) < 2 ? (t_local & 3) : T - 4 + (t_local & 3)) : t0 + t_local;
  const int64_t b_out = EDGES ? b + (t_local >> 2) : b;
  // (whole warps without a frame -- the tail of a clip's last tile -- are done: only __syncwarp from here on)
  if (!EDGES && t0 + 2 * warp >= T) return;
  float2* sc = scratch + t_local * kScStride;
  const float* fr = s_wave + (EDGES || kPacked ? kNfft : kHop) * t_local;

  // ---- stage A: 15 radix-16 FFTs over n1 (lane = n2), twiddle by W240^(n2 k1)
  if (l < 15) {
    float2 x[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
      const int m = 15 * n1 + l;
      float2 s = *reinterpret_cast<const float2*>(fr + 2 * m);
      float2 wv = *reinterpret_cast<const float2*>(s_win + 2 * m);
      x[n1] = make_float2(s.x * wv.x, s.y * wv.y);
    }
    fft16_dif(x);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int k1 = bitrev4(i);
      sc[k1 * 15 + l] = cmul(x[i], s_tw240[k1 * 16 + l]);
    }
  }
  __syncwarp();

  // ---- stage B: 16 DFT-15 over n2 (lane = k1): Z[k1 + 16 k2] stays in this lane's registers
  float2 z[15];
  {
    float2 y[15];
#pragma unroll
    for (int n2 = 0; n2 < 15; ++n2) y[n2] = sc[l * 15 + n2];
    dft15(y, z);
  }

  // ---- real-FFT split + power: X[k] = E + (-sin, -cos)(theta_k) * O for k = l + 16 j.  Z[k] is this lane's z[j];
  // its mirror Z[240 - k] = Z[(16 - l) + 16 (14 - j)] is lane 16 - l's z[14 - j] (one shuffle inside the half-warp),
  // or, for lane 0, its own z[(15 - j) mod 15]: no trip through shared memory.
  float p[15];
  const int mirror = (16 - l) & 15;
#pragma unroll
  for (int j = 0; j < 15; ++j) {
    p[j] = 0.f;
    if (j < tb.nb16) {
      const int k = l + 16 * j;
      const float2 zk = z[j];
      float2 zm;
      zm.x = __shfl_sync(0xffffffffu, z[14 - j].x, mirror, 16);
      zm.y = __shfl_sync(0xffffffffu, z[14 - j].y, mirror, 16);
      if (l == 0) zm = z[(15 - j) % 15];
      const float2 tw = s_tw480[k];  // (sin, cos)
      const float er = 0.5f * (zk.x + zm.x), ei = 0.5f * (zk.y - zm.y);
      const float orr = 0.5f * (zk.x - zm.x), oi = 0.5f * (zk.y + zm.y);
      const float xr = er - tw.x * orr + tw.y * oi;
      const float xi = ei - tw.x * oi - tw.y * orr;
      p[j] = xr * xr + xi * xi;
    }
  }
  __syncwarp();
  float* P = reinterpret_cast<float*>(sc);
#pragma unroll
  for (int j = 0; j < 15; ++j)
    if (j < tb.nb16) P[l + 16 * j] = p[j];
  __syncwarp();

  // ---- sparse mel filterbank, ln, x2 (reference "DCT" of a length-1 axis)
  if (kPacked ? b + t_local < B : t < T && b_out < B) {
    float* out;
    if constexpr (kPacked) out = src.frame_out(w, t_local);
    else out = src.out_row(feat, b_out, T, t, tb.n_mels);
    for (int m = l; m < tb.n_mels; m += 16) {
      const int lo = s_lo[m], cnt = s_cnt[m], off = s_off[m];
      float acc = 0.f;
      for (int i = 0; i < cnt; ++i) acc = fmaf(s_w[off + i], P[lo + i], acc);
      out[m] = acc > 0.f ? 2.f * logf(acc) : 2.f * acc;
    }
  }
}

// Streaming front-end: interior frames of window k (t = 2 .. T-3) are rows (k * m + t) of the stream-level frame
// table S (m = shift / hop).  Pure copy, 16 bytes per thread when the row length allows.
template <typename V>
__global__ void __launch_bounds__(256)
mfcc_stream_gather_kernel(const V* __restrict__ S, int64_t K, int T, int m, int row_v, V* __restrict__ feat) {
  const int64_t per_win = (int64_t)(T - 4) * row_v;
  const int64_t total = K * per_win;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = i / per_win;
    const int64_t r = i - k * per_win;   // (t - 2) * row_v + c
    feat[k * (int64_t)T * row_v + 2 * row_v + r] = __ldg(S + (k * m + 2) * (int64_t)row_v + r);
  }
}

// ---------------------------------------------------------------------------------------------
// Live streams (kws_live_*): per stream a sample ring, a frame ring and a sample counter, all on the device.

// Launch 1 of a push: stream s's n new samples (chunk row s) go to its sample ring, converted to float, its counter
// advances by n, and wpos[s] receives the ring position of the push's first window, k = floor((c_old - W) / H) + 1.
// One CTA per stream, so the counter is written only after every thread has read it.
__device__ __forceinline__ float live_sample(float v) { return v; }
__device__ __forceinline__ float live_sample(int16_t v) { return (float)v * (1.f / 32768.f); }

template <typename SMP>
__global__ void __launch_bounds__(128)
live_append_kernel(const SMP* __restrict__ chunk, int n, float* __restrict__ ring, int cap, int window, int shift,
                   int64_t* __restrict__ count, int* __restrict__ wpos) {
  const int64_t s = blockIdx.x;
  const int64_t c = count[s];
  const int start = (int)(c % cap);
  const SMP* in = chunk + s * n;
  float* out = ring + s * cap;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int p = start + i;
    if (p >= cap) p -= cap;   // (n <= cap)
    out[p] = live_sample(__ldg(in + i));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    count[s] = c + n;
    wpos[s] = (int)pos_mod((floor_div(c - window, shift) + 1) * shift, cap);
  }
}

__global__ void live_reset_kernel(const int64_t* __restrict__ ids, int64_t n_ids, int64_t S, int64_t* __restrict__ count) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_ids; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t id = ids[i];
    if (id >= 0 && id < S) count[id] = 0;
  }
}

// Last launch of a push: window slot `slot` = (stream s, window k).  Interior frames t = 2 .. T-3 are frame-ring rows
// (k m + t) mod fcap of stream s (m = shift / hop); a slot with k < 0 (the warm-up of a fresh stream) is all zeros.
// One CTA per slot; the edge frames of valid slots are the edge launch's.
template <typename V>
__global__ void __launch_bounds__(256)
live_gather_kernel(const V* __restrict__ frames, const int64_t* __restrict__ count, int n, int window, int shift, int K,
                   int T, int fcap, int row_v, V* __restrict__ feat) {
  const int64_t slot = blockIdx.x;
  const int64_t s = slot / K;
  const int64_t k = floor_div(count[s] - n - window, shift) + 1 + (slot - s * K);
  const int r0 = k >= 0 ? (int)pos_mod(k * (shift / kHop), fcap) : 0;
  const V* rows = frames + s * fcap * (int64_t)row_v;
  V* out = feat + slot * T * (int64_t)row_v;
  for (int i = threadIdx.x; i < T * row_v; i += blockDim.x) {
    const int t = i / row_v, c = i - t * row_v;
    V v{};
    if (k >= 0) {
      if (t < 2 || t >= T - 2) continue;
      int r = r0 + t;
      if (r >= fcap) r -= fcap;   // (T <= fcap)
      v = __ldg(rows + r * (int64_t)row_v + c);
    }
    out[i] = v;
  }
}

// Ragged pushes.  Launch 1: stream s's len[s] new samples (samples + off[s]) go to its ring, its counter advances, and
// counts[s] receives the push's plan for s: new frame-table rows (high word) and completed windows (low word), from the
// counts before and after.  counts[S] = 0, so that the exclusive scan of counts[0 .. S] ends in the totals.

template <typename SMP>
__global__ void __launch_bounds__(128)
live_ragged_append_kernel(const SMP* __restrict__ samples, const int64_t* __restrict__ off, const int* __restrict__ len,
                          float* __restrict__ ring, int cap, int window, int shift, int S, int64_t* __restrict__ count,
                          int64_t* __restrict__ counts) {
  const int64_t s = blockIdx.x;
  const int n = len[s];
  const int64_t c = count[s];
  const int start = (int)(c % cap);
  const SMP* in = samples + off[s];
  float* out = ring + s * cap;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int p = start + i;
    if (p >= cap) p -= cap;   // (n <= max_push < cap)
    out[p] = live_sample(__ldg(in + i));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    count[s] = c + n;
    const int64_t rows = ragged_rows(c + n) - ragged_rows(c);
    const int64_t wins = ragged_wins(c + n, window, shift) - ragged_wins(c, window, shift);
    counts[s] = rows << 32 | wins;
    if (s == 0) counts[S] = 0;
  }
}

// Last launch: window entry i (stream s, window k; see RaggedSource<true>): interior frames t = 2 .. T-3 are frame-ring
// rows (k m + t) mod fcap of stream s.  One CTA per entry of the host's bound; CTAs past the device's count exit.
template <typename V>
__global__ void __launch_bounds__(256)
live_ragged_gather_kernel(const V* __restrict__ frames, const int64_t* __restrict__ count, const int* __restrict__ len,
                          const int64_t* __restrict__ plan, int S, int window, int shift, int T, int fcap, int row_v,
                          V* __restrict__ feat, int64_t* __restrict__ win_stream, int64_t* __restrict__ win_index,
                          int64_t* __restrict__ n_windows) {
  const int64_t i = blockIdx.x;
  const int64_t M = __ldg(plan + S) & 0xffffffffll;
  if (i == 0 && threadIdx.x == 0 && n_windows) *n_windows = M;
  if (i >= M) return;
  int lo = 0, hi = S;   // (plan[lo] <= i < plan[hi] in the low words)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((__ldg(plan + mid) & 0xffffffffll) <= i) lo = mid;
    else hi = mid;
  }
  const int64_t s = lo;
  const int64_t k = ragged_wins(__ldg(count + s) - __ldg(len + s), window, shift) + i -
                    (__ldg(plan + s) & 0xffffffffll);
  if (threadIdx.x == 0) {
    if (win_stream) win_stream[i] = s;
    if (win_index) win_index[i] = k;
  }
  const int r0 = (int)pos_mod(k * (shift / kHop), fcap);
  const V* rows = frames + s * fcap * (int64_t)row_v;
  V* out = feat + i * T * (int64_t)row_v;
  for (int j = threadIdx.x; j < (T - 4) * row_v; j += blockDim.x) {
    const int t = 2 + j / row_v, c = j - (t - 2) * row_v;
    int r = r0 + t;
    if (r >= fcap) r -= fcap;   // (T <= fcap)
    out[t * row_v + c] = __ldg(rows + r * (int64_t)row_v + c);
  }
}

// ---------------------------------------------------------------------------------------------
// host side: table construction (double precision, float32 rounding where numpy rounds)

static double hz_to_mel_slaney(double f) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
static double mel_to_hz_slaney(double m) {
  const double f_sp = 200.0 / 3, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
  const double logstep = std::log(6.4) / 27.0;
  return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

}  // namespace kws

using namespace kws;

struct kws_frontend : kws::Frontend {};

extern "C" int kws_frontend_create(int sr, int n_mels, float f_min, float f_max, int n_fft, int hop,
                                   kws_frontend_t** out) {
  KWS_REQUIRE(out != nullptr, "kws_frontend_create: out is null");
  *out = nullptr;
  KWS_REQUIRE(n_fft == kNfft && hop == kHop,
              "kws_frontend_create: only n_fft=480 / hop=160 is built (got %d / %d)", n_fft, hop);
  KWS_REQUIRE(n_mels >= 1 && n_mels <= kMaxMels, "kws_frontend_create: n_mels must be in [1,%d]", kMaxMels);
  KWS_REQUIRE(sr > 0 && f_min >= 0 && f_max > f_min && f_max <= sr / 2.0f,
              "kws_frontend_create: need 0 <= f_min < f_max <= sr/2");
  int major = 0, minor = 0, sms = 0;
  KWS_TRY(kws_device_info(&major, &minor, &sms));

  const int n_bins = 1 + n_fft / 2;
  // librosa.filters.mel(htk=False, norm='slaney'), float32 storage like numpy.  The band edges follow np.linspace:
  // m_lo + i * step, the last one exactly m_hi.  (m_lo + (m_hi - m_lo) * i / (n_mels + 1) can round the last edge above
  // f_max, which gives the last filter a weight at bin f_max; at f_max = sr/2 that is the Nyquist bin.)
  std::vector<double> mel_f(n_mels + 2);
  const double m_lo = hz_to_mel_slaney(f_min), m_hi = hz_to_mel_slaney(f_max);
  const double step = (m_hi - m_lo) / (n_mels + 1);
  for (int i = 0; i < n_mels + 1; ++i) mel_f[i] = mel_to_hz_slaney(m_lo + i * step);
  mel_f[n_mels + 1] = mel_to_hz_slaney(m_hi);
  std::vector<int> lo(n_mels), cnt(n_mels), off(n_mels);
  std::vector<float> wts;
  int max_bin = 0;
  for (int i = 0; i < n_mels; ++i) {
    const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
    int first = -1, last = -1;
    std::vector<float> row(n_bins);
    for (int k = 0; k < n_bins; ++k) {
      const double f = (double)sr / 2 * k / (n_bins - 1);
      const double lower = (f - mel_f[i]) / (mel_f[i + 1] - mel_f[i]);
      const double upper = (mel_f[i + 2] - f) / (mel_f[i + 2] - mel_f[i + 1]);
      const float tri = (float)std::fmax(0.0, std::fmin(lower, upper));
      row[k] = (float)((double)tri * enorm);
      if (row[k] != 0.f) { if (first < 0) first = k; last = k; }
    }
    off[i] = (int)wts.size();
    if (first < 0) { lo[i] = 0; cnt[i] = 0; continue; }
    lo[i] = first; cnt[i] = last - first + 1;
    for (int k = first; k <= last; ++k) wts.push_back(row[k]);
    if (last > max_bin) max_bin = last;
  }
  KWS_REQUIRE(max_bin < kNz, "kws_frontend_create: filterbank touches the Nyquist bin (unsupported)");
  const int nb16 = max_bin / 16 + 1;

  const double PI = 3.14159265358979323846;
  std::vector<float> window(kNfft);
  for (int n = 0; n < kNfft; ++n) window[n] = (float)(0.5 - 0.5 * std::cos(2.0 * PI * n / kNfft));
  std::vector<float2> tw240(kTwA), tw480(kNz);
  for (int k1 = 0; k1 < 16; ++k1)
    for (int l = 0; l < 16; ++l) {
      const int j = (l * k1) % kNz;
      tw240[k1 * 16 + l] = make_float2((float)std::cos(2.0 * PI * j / kNz), (float)(-std::sin(2.0 * PI * j / kNz)));
    }
  for (int j = 0; j < kNz; ++j)
    tw480[j] = make_float2((float)std::sin(2.0 * PI * j / kNfft), (float)std::cos(2.0 * PI * j / kNfft));

  // one device blob
  const size_t nnz = wts.size();
  size_t o_win = 0, o_tw240 = o_win + sizeof(float) * kNfft, o_tw480 = o_tw240 + sizeof(float2) * kTwA,
         o_lo = o_tw480 + sizeof(float2) * kNz, o_cnt = o_lo + sizeof(int) * n_mels,
         o_off = o_cnt + sizeof(int) * n_mels, o_w = o_off + sizeof(int) * n_mels,
         total = o_w + sizeof(float) * (nnz + 1);
  std::vector<unsigned char> host(total);
  memcpy(host.data() + o_win, window.data(), sizeof(float) * kNfft);
  memcpy(host.data() + o_tw240, tw240.data(), sizeof(float2) * kTwA);
  memcpy(host.data() + o_tw480, tw480.data(), sizeof(float2) * kNz);
  memcpy(host.data() + o_lo, lo.data(), sizeof(int) * n_mels);
  memcpy(host.data() + o_cnt, cnt.data(), sizeof(int) * n_mels);
  memcpy(host.data() + o_off, off.data(), sizeof(int) * n_mels);
  if (nnz) memcpy(host.data() + o_w, wts.data(), sizeof(float) * nnz);

  kws_frontend* fe = new kws_frontend();
  fe->sr = sr; fe->n_mels = n_mels; fe->n_fft = n_fft; fe->hop = hop; fe->f_min = f_min; fe->f_max = f_max;
  cudaError_t e = cudaMalloc(&fe->dev_blob, total);
  if (e == cudaSuccess) e = cudaMemcpy(fe->dev_blob, host.data(), total, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error("kws_frontend_create: table upload failed: %s", cudaGetErrorString(e));
    if (fe->dev_blob) cudaFree(fe->dev_blob);
    delete fe;
    return KWS_ERR_CUDA;
  }
  unsigned char* d = static_cast<unsigned char*>(fe->dev_blob);
  fe->t.window = reinterpret_cast<const float*>(d + o_win);
  fe->t.tw240 = reinterpret_cast<const float2*>(d + o_tw240);
  fe->t.tw480 = reinterpret_cast<const float2*>(d + o_tw480);
  fe->t.mel_lo = reinterpret_cast<const int*>(d + o_lo);
  fe->t.mel_cnt = reinterpret_cast<const int*>(d + o_cnt);
  fe->t.mel_off = reinterpret_cast<const int*>(d + o_off);
  fe->t.mel_w = reinterpret_cast<const float*>(d + o_w);
  fe->t.n_mels = n_mels; fe->t.nnz = (int)nnz; fe->t.nb16 = nb16;
  fe->smem_bytes = sizeof(float2) * (kFramesPerCta * kScStride + kTwA + kNz) +
                   sizeof(float) * (kStageSamples + kNfft) + sizeof(int) * 3 * kMaxMels +
                   sizeof(float) * (nnz + 1);
  fe->smem_bytes_edges = fe->smem_bytes + sizeof(float) * (kEdgeStageSamples - kStageSamples);
  e = raise_dynamic_smem(mfcc_kernel<false, float>, fe->smem_bytes);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<false, int16_t>, fe->smem_bytes);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, float>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, int16_t>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<false, float, RingSource<false>>, fe->smem_bytes);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, float, RingSource<true>>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, float, EdgeRingSource>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<false, float, RaggedSource<false>>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, float, RaggedSource<true>>, fe->smem_bytes_edges);
  if (e == cudaSuccess) e = raise_dynamic_smem(mfcc_kernel<true, float, RaggedEdgeSource>, fe->smem_bytes_edges);
  if (e != cudaSuccess) {
    set_error("kws_frontend_create: raising the shared memory limit failed: %s", cudaGetErrorString(e));
    cudaFree(fe->dev_blob);
    delete fe;
    return KWS_ERR_CUDA;
  }
  *out = fe;
  return KWS_OK;
}

extern "C" void kws_frontend_destroy(kws_frontend_t* fe) {
  if (!fe) return;
  if (fe->dev_blob) cudaFree(fe->dev_blob);
  delete fe;
}

extern "C" int kws_frontend_n_frames(const kws_frontend_t* fe, int n_samples) {
  if (!fe || n_samples < 0) return 0;
  return 1 + n_samples / fe->hop;
}

extern "C" int kws_frontend_n_mels(const kws_frontend_t* fe) { return fe ? fe->n_mels : 0; }

template <typename SMP>
static int mfcc_forward_any(const char* who, const kws_frontend_t* fe, const SMP* wav, int64_t B, int n_samples, float* feat,
                            void* stream) {
  KWS_REQUIRE(fe != nullptr, "%s: frontend is null", who);
  KWS_REQUIRE(B >= 0, "%s: negative batch", who);
  // librosa's reflect padding of n_fft/2 needs more than n_fft/2 samples
  KWS_REQUIRE(n_samples > kNfft / 2, "%s: need more than %d samples per clip (got %d)", who, kNfft / 2, n_samples);
  if (B == 0) return KWS_OK;
  KWS_REQUIRE(wav != nullptr && feat != nullptr, "%s: null buffer", who);
  const int T = 1 + n_samples / kHop;
  const int tiles = ceil_div(T, kFramesPerCta);
  const int64_t blocks = B * tiles;
  KWS_REQUIRE(blocks < (int64_t)2147483647, "%s: batch too large for one launch", who);
  mfcc_kernel<false, SMP><<<(unsigned)blocks, kMfccThreads, fe->smem_bytes, as_stream(stream)>>>(
      fe->t, DenseSource<SMP>{wav, (int64_t)n_samples}, B, n_samples, T, tiles, feat);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

extern "C" int kws_mfcc_forward(const kws_frontend_t* fe, const float* wav, int64_t B, int n_samples,
                                float* feat, void* stream) {
  return mfcc_forward_any<float>("kws_mfcc_forward", fe, wav, B, n_samples, feat, stream);
}

extern "C" int kws_mfcc_forward_pcm16(const kws_frontend_t* fe, const int16_t* wav, int64_t B, int n_samples,
                                      float* feat, void* stream) {
  return mfcc_forward_any<int16_t>("kws_mfcc_forward_pcm16", fe, wav, B, n_samples, feat, stream);
}

extern "C" size_t kws_mfcc_stream_scratch_bytes(const kws_frontend_t* fe, int64_t n_windows, int window, int shift) {
  if (!fe || n_windows < 1 || window < 1 || shift < 1) return 0;
  const int T = 1 + window / kHop;
  if (shift % kHop != 0 || T < 5) return 0;   // no frame is shared: computed straight into the output
  const int64_t span = (n_windows - 1) * (int64_t)shift + window;
  return (size_t)(1 + span / kHop) * fe->n_mels * sizeof(float);
}

template <typename SMP>
static int mfcc_stream_forward_any(const kws_frontend_t* fe, const SMP* wav, int64_t n_windows, int window,
                                   int shift, float* feat, void* scratch, size_t scratch_bytes, void* stream) {
  KWS_REQUIRE(fe != nullptr, "kws_mfcc_stream_forward: frontend is null");
  KWS_REQUIRE(n_windows >= 0, "kws_mfcc_stream_forward: negative window count");
  KWS_REQUIRE(window > kNfft / 2, "kws_mfcc_stream_forward: need more than %d samples per window (got %d)",
              kNfft / 2, window);
  KWS_REQUIRE(shift >= 1, "kws_mfcc_stream_forward: shift must be positive (got %d)", shift);
  if (n_windows == 0) return KWS_OK;
  KWS_REQUIRE(wav != nullptr && feat != nullptr, "kws_mfcc_stream_forward: null buffer");
  cudaStream_t st = as_stream(stream);
  const int T = 1 + window / kHop;
  const int tiles = ceil_div(T, kFramesPerCta);
  const int64_t span = (n_windows - 1) * (int64_t)shift + window;   // samples the windows cover
  if (shift % kHop != 0 || T < 5) {
    // windows do not share frames (or have no interior frame): every window in full, read in place from the stream
    const int64_t blocks = n_windows * tiles;
    KWS_REQUIRE(blocks < (int64_t)2147483647, "kws_mfcc_stream_forward: too many windows for one launch");
    mfcc_kernel<false, SMP><<<(unsigned)blocks, kMfccThreads, fe->smem_bytes, st>>>(
        fe->t, DenseSource<SMP>{wav, (int64_t)shift}, n_windows, window, T, tiles, feat);
    KWS_CHECK_LAUNCH();
    return KWS_OK;
  }
  KWS_REQUIRE(span < (int64_t)2147483647, "kws_mfcc_stream_forward: the windows cover %lld samples; split the call",
              (long long)span);
  const size_t need = kws_mfcc_stream_scratch_bytes(fe, n_windows, window, shift);
  KWS_REQUIRE(scratch != nullptr && scratch_bytes >= need,
              "kws_mfcc_stream_forward: needs %zu bytes of scratch, got %zu", need, scratch_bytes);
  // 1) the frame table of the whole span as ONE clip: rows 2 .. J-3 do not touch its reflect padding
  float* S = static_cast<float*>(scratch);
  const int J = 1 + (int)(span / kHop);
  mfcc_kernel<false, SMP><<<(unsigned)ceil_div(J, kFramesPerCta), kMfccThreads, fe->smem_bytes, st>>>(
      fe->t, DenseSource<SMP>{wav, span}, (int64_t)1, (int)span, J, ceil_div(J, kFramesPerCta), S);
  KWS_CHECK_LAUNCH();
  // 2) the four frames per window that do (reflect padding at the WINDOW's edges, audio_processor.py:19-26 per window)
  mfcc_kernel<true, SMP><<<(unsigned)ceil_div<int64_t>(n_windows, 4), kMfccThreads, fe->smem_bytes_edges, st>>>(
      fe->t, DenseSource<SMP>{wav, (int64_t)shift}, n_windows, window, T, 1, feat);
  KWS_CHECK_LAUNCH();
  // 3) interior frames: copies of table rows
  const int m = shift / kHop;
  const bool vec = fe->n_mels % 4 == 0 && (reinterpret_cast<uintptr_t>(S) & 15) == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0;
  const int row_v = vec ? fe->n_mels / 4 : fe->n_mels;
  const int64_t total = n_windows * (int64_t)(T - 4) * row_v;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(total, 256), 148 * 16);
  if (vec)
    mfcc_stream_gather_kernel<float4><<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(S), n_windows, T, m, row_v,
                                                            reinterpret_cast<float4*>(feat));
  else
    mfcc_stream_gather_kernel<float><<<grid, 256, 0, st>>>(S, n_windows, T, m, row_v, feat);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

extern "C" int kws_mfcc_stream_forward(const kws_frontend_t* fe, const float* wav, int64_t n_windows, int window,
                                       int shift, float* feat, void* scratch, size_t scratch_bytes, void* stream) {
  return mfcc_stream_forward_any<float>(fe, wav, n_windows, window, shift, feat, scratch, scratch_bytes, stream);
}

extern "C" int kws_mfcc_stream_forward_pcm16(const kws_frontend_t* fe, const int16_t* wav, int64_t n_windows, int window,
                                             int shift, float* feat, void* scratch, size_t scratch_bytes, void* stream) {
  return mfcc_stream_forward_any<int16_t>(fe, wav, n_windows, window, shift, feat, scratch, scratch_bytes, stream);
}

// ---- live streams ---------------------------------------------------------------------------
// One device allocation per state: sample rings [S][cap] f32, frame rings [S][fcap][n_mels] f32, counters [S] i64,
// first-window ring positions [S] i32.  Ragged pushes add a pinned host staging buffer for their per-stream sample
// offsets and lengths and the event that marks its last copy done; both are created by the first ragged push.
// (struct kws_live: live.cuh)

namespace {
struct LiveLayout {
  int T, cap, fcap;
  size_t o_frames, o_count, o_wpos, total;
};

int live_layout(const char* who, const kws_frontend_t* fe, int S, int window, int shift, int max_push, LiveLayout* L) {
  KWS_REQUIRE(fe != nullptr, "%s: frontend is null", who);
  KWS_REQUIRE(S >= 1, "%s: need at least one stream (got %d)", who, S);
  KWS_REQUIRE(shift >= 1 && shift % kHop == 0, "%s: the shift must be a positive multiple of the %d-sample hop (got %d)",
              who, kHop, shift);
  KWS_REQUIRE(window >= 1 && 1 + window / kHop >= 5,
              "%s: a window of %d samples has %d frames; at least 5 are needed so that windows share frames", who,
              window, window >= 1 ? 1 + window / kHop : 0);
  KWS_REQUIRE(max_push >= 1 && max_push % shift == 0, "%s: max_push must be a positive multiple of the shift %d (got %d)",
              who, shift, max_push);
  const int64_t span = (int64_t)window + max_push;   // the oldest sample a push reads lies < window before it
  KWS_REQUIRE(span <= (int64_t)1 << 30, "%s: window + max_push = %lld samples is too large", who, (long long)span);
  L->T = 1 + window / kHop;
  L->cap = (int)round_up<int64_t>(span, 16);          // 16-byte staging loads never straddle the wrap
  L->fcap = (int)ceil_div<int64_t>(span, kHop);
  const size_t ring = round_up<size_t>((size_t)S * L->cap * sizeof(float), 256);
  const size_t frames = round_up<size_t>((size_t)S * L->fcap * fe->n_mels * sizeof(float), 256);
  L->o_frames = ring;
  L->o_count = ring + frames;
  L->o_wpos = L->o_count + (size_t)S * sizeof(int64_t);
  L->total = L->o_wpos + (size_t)S * sizeof(int);
  return KWS_OK;
}
}  // namespace

extern "C" size_t kws_live_state_bytes(const kws_frontend_t* fe, int n_streams, int window, int shift, int max_push) {
  LiveLayout L;
  return live_layout("kws_live_state_bytes", fe, n_streams, window, shift, max_push, &L) == KWS_OK ? L.total : 0;
}

extern "C" int kws_live_create(const kws_frontend_t* fe, int n_streams, int window, int shift, int max_push,
                               kws_live_t** out) {
  KWS_REQUIRE(out != nullptr, "kws_live_create: out is null");
  *out = nullptr;
  LiveLayout L;
  KWS_TRY(live_layout("kws_live_create", fe, n_streams, window, shift, max_push, &L));
  void* dev = nullptr;
  cudaError_t e = cudaMalloc(&dev, L.total);
  if (e == cudaSuccess) e = cudaMemset(dev, 0, L.total);   // counters start at 0; the rings' contents are never read stale
  if (e != cudaSuccess) {                                   // by a valid window, zeroing only keeps them finite
    set_error("kws_live_create: %zu bytes of device state: %s", L.total, cudaGetErrorString(e));
    if (dev) cudaFree(dev);
    return KWS_ERR_CUDA;
  }
  unsigned char* d = static_cast<unsigned char*>(dev);
  *out = new kws_live{fe, n_streams, window, shift, max_push, L.T, L.cap, L.fcap, dev, reinterpret_cast<float*>(d),
                      reinterpret_cast<float*>(d + L.o_frames), reinterpret_cast<int64_t*>(d + L.o_count),
                      reinterpret_cast<int*>(d + L.o_wpos)};
  return KWS_OK;
}

extern "C" void kws_live_destroy(kws_live_t* live) {
  if (!live) return;
  cudaFree(live->dev);
  if (live->ragged_copied) cudaEventDestroy(live->ragged_copied);
  if (live->ragged_host) cudaFreeHost(live->ragged_host);
  delete live;
}

extern "C" int kws_live_reset(kws_live_t* live, const int64_t* stream_ids, int64_t count, void* stream) {
  KWS_REQUIRE(live != nullptr, "kws_live_reset: live state is null");
  KWS_REQUIRE(count >= 0, "kws_live_reset: negative count");
  if (count == 0) return KWS_OK;
  KWS_REQUIRE(stream_ids != nullptr, "kws_live_reset: stream_ids is null");
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div<int64_t>(count, 256), 1024);
  live_reset_kernel<<<grid, 256, 0, as_stream(stream)>>>(stream_ids, count, live->S, live->count);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

namespace kws {
template <typename SMP>
int live_append_rows(const char* who, kws_live_t* L, const SMP* chunk, int n, cudaStream_t st) {
  KWS_REQUIRE(L != nullptr, "%s: live state is null", who);
  KWS_REQUIRE(n >= 1 && n <= L->max_push && n % L->shift == 0,
              "%s: a push of %d samples per stream: need a multiple of the shift %d in [%d, %d]", who, n, L->shift,
              L->shift, L->max_push);
  KWS_REQUIRE(chunk != nullptr, "%s: null buffer", who);
  const kws_frontend* fe = L->fe;
  const int K = n / L->shift;
  const int64_t slots = (int64_t)L->S * K;
  const int rows = n / kHop;
  const int tiles = ceil_div(rows, kFramesPerCta);
  KWS_REQUIRE(slots < (int64_t)2147483647 && (int64_t)L->S * tiles < (int64_t)2147483647,
              "%s: too many streams for one launch", who);
  // 1) the new samples into the sample rings; counters and first-window positions
  live_append_kernel<SMP><<<(unsigned)L->S, 128, 0, st>>>(chunk, n, L->ring, L->cap, L->window, L->shift, L->count,
                                                         L->wpos);
  KWS_CHECK_LAUNCH();
  // 2) the n / 160 frame-table rows per stream the push completes, r = c_old/160 - 1 .. c_new/160 - 2 (no padding: N
  //    is not read)
  mfcc_kernel<false, float, RingSource<false>><<<(unsigned)(L->S * tiles), kMfccThreads, fe->smem_bytes, st>>>(
      fe->t, RingSource<false>{L->ring, L->count, L->wpos, L->cap, n, L->fcap, L->shift, K, (int)slots}, (int64_t)L->S, 0,
      rows, tiles, L->frames);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}
template int live_append_rows<float>(const char*, kws_live_t*, const float*, int, cudaStream_t);
template int live_append_rows<int16_t>(const char*, kws_live_t*, const int16_t*, int, cudaStream_t);

int live_edge_frames(kws_live_t* L, int n, float* edges, cudaStream_t st) {
  const int K = n / L->shift;
  const int64_t slots = (int64_t)L->S * K;
  mfcc_kernel<true, float, EdgeRingSource><<<(unsigned)ceil_div<int64_t>(slots, 4), kMfccThreads,
                                             L->fe->smem_bytes_edges, st>>>(
      L->fe->t, EdgeRingSource{{L->ring, L->count, L->wpos, L->cap, n, L->fcap, L->shift, K, (int)slots}}, slots,
      L->window, L->T, 1, edges);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}
}  // namespace kws

template <typename SMP>
static int live_push_any(const char* who, kws_live_t* L, const SMP* chunk, int n, float* feat, void* stream) {
  KWS_REQUIRE(feat != nullptr || L == nullptr, "%s: null buffer", who);
  cudaStream_t st = as_stream(stream);
  KWS_TRY(live_append_rows(who, L, chunk, n, st));
  const kws_frontend* fe = L->fe;
  const int K = n / L->shift;
  const int64_t slots = (int64_t)L->S * K;
  // 3) the four reflect-padded edge frames of each of the S K new windows
  mfcc_kernel<true, float, RingSource<true>><<<(unsigned)ceil_div<int64_t>(slots, 4), kMfccThreads, fe->smem_bytes_edges,
                                               st>>>(
      fe->t, RingSource<true>{L->ring, L->count, L->wpos, L->cap, n, L->fcap, L->shift, K, (int)slots}, slots, L->window,
      L->T, 1, feat);
  KWS_CHECK_LAUNCH();
  // 4) interior frames from the frame rings; warm-up slots zeroed
  const bool vec = fe->n_mels % 4 == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0;
  const int row_v = vec ? fe->n_mels / 4 : fe->n_mels;
  if (vec)
    live_gather_kernel<float4><<<(unsigned)slots, 256, 0, st>>>(reinterpret_cast<const float4*>(L->frames), L->count, n,
                                                                L->window, L->shift, K, L->T, L->fcap, row_v,
                                                                reinterpret_cast<float4*>(feat));
  else
    live_gather_kernel<float><<<(unsigned)slots, 256, 0, st>>>(L->frames, L->count, n, L->window, L->shift, K, L->T,
                                                               L->fcap, row_v, feat);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

extern "C" int kws_live_push(kws_live_t* live, const float* chunk, int n, float* feat, void* stream) {
  return live_push_any<float>("kws_live_push", live, chunk, n, feat, stream);
}

extern "C" int kws_live_push_pcm16(kws_live_t* live, const int16_t* chunk, int n, float* feat, void* stream) {
  return live_push_any<int16_t>("kws_live_push_pcm16", live, chunk, n, feat, stream);
}

// ---- ragged pushes --------------------------------------------------------------------------
// Workspace: per-stream sample offsets i64[S] and lengths i32[S] (one copy from the pinned staging buffer), the plan
// counts i64[S+1], their exclusive scan i64[S+1], and CUB's scan scratch; then, 256-byte aligned, the caller's own part
// (kws_live_cnn's).
namespace {
struct RaggedLayout {
  size_t o_len, o_counts, o_plan, o_temp, temp, o_extra, total;
};

int ragged_layout(const char* who, const kws_live* L, size_t extra, RaggedLayout* R) {
  const size_t S = (size_t)L->S;
  R->o_len = S * sizeof(int64_t);
  R->o_counts = round_up<size_t>(R->o_len + S * sizeof(int32_t), 256);
  R->o_plan = R->o_counts + round_up<size_t>((S + 1) * sizeof(int64_t), 256);
  R->o_temp = R->o_plan + round_up<size_t>((S + 1) * sizeof(int64_t), 256);
  R->temp = 0;
  const cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, R->temp, static_cast<int64_t*>(nullptr),
                                                      static_cast<int64_t*>(nullptr), L->S + 1);
  if (e != cudaSuccess) {
    set_error("%s: scan size query failed: %s", who, cudaGetErrorString(e));
    return KWS_ERR_CUDA;
  }
  R->o_extra = round_up<size_t>(R->o_temp + R->temp, 256);
  R->total = extra ? R->o_extra + extra : R->o_temp + R->temp;
  return KWS_OK;
}
}  // namespace

extern "C" size_t kws_live_ragged_workspace_bytes(const kws_live_t* live) {
  return live ? live_ragged_workspace_bytes("kws_live_ragged_workspace_bytes", live, 0) : 0;
}

namespace kws {
size_t live_ragged_workspace_bytes(const char* who, const kws_live_t* L, size_t extra) {
  RaggedLayout R;
  return ragged_layout(who, L, extra, &R) == KWS_OK ? R.total : 0;
}

template <typename SMP>
int live_ragged_append_rows(const char* who, kws_live_t* L, const SMP* samples, const int32_t* lengths,
                            int64_t capacity, const void* out, const char* out_name, void* workspace, size_t ws_bytes,
                            size_t ws_extra, cudaStream_t st, LiveRagged* P) {
  KWS_REQUIRE(L != nullptr, "%s: live state is null", who);
  KWS_REQUIRE(lengths != nullptr, "%s: lengths is null", who);
  // the whole plan is checked on the host, before anything is staged or launched
  int64_t n_samples = 0, row_bound = 0, win_bound = 0;
  for (int s = 0; s < L->S; ++s) {
    const int n = lengths[s];
    KWS_REQUIRE(n >= 0 && n <= L->max_push, "%s: stream %d brings %d samples; a push takes 0 to max_push = %d", who, s,
                n, L->max_push);
    n_samples += n;
    row_bound += ceil_div(n, kHop);
    win_bound += ceil_div(n, L->shift);
  }
  KWS_REQUIRE(row_bound < INT32_MAX && win_bound < INT32_MAX, "%s: too many new rows or windows for one launch", who);
  KWS_REQUIRE(capacity >= win_bound,
              "%s: the push can complete up to %lld windows (sum of ceil(length / shift)); capacity is %lld", who,
              (long long)win_bound, (long long)capacity);
  KWS_REQUIRE(n_samples == 0 || samples != nullptr, "%s: samples is null", who);
  KWS_REQUIRE(win_bound == 0 || out != nullptr, "%s: %s is null", who, out_name);
  RaggedLayout R;
  KWS_TRY(ragged_layout(who, L, ws_extra, &R));
  KWS_REQUIRE(workspace != nullptr && ws_bytes >= R.total, "%s: needs %zu bytes of workspace, got %zu", who, R.total,
              workspace ? ws_bytes : (size_t)0);
  const size_t stage_bytes = R.o_len + (size_t)L->S * sizeof(int32_t);
  if (!L->ragged_host) {
    KWS_CUDA(cudaMallocHost(&L->ragged_host, stage_bytes));
    KWS_CUDA(cudaEventCreateWithFlags(&L->ragged_copied, cudaEventDisableTiming));
  } else {
    KWS_CUDA(cudaEventSynchronize(L->ragged_copied));   // the previous ragged push's copy out of the staging buffer
  }
  int64_t* off_h = static_cast<int64_t*>(L->ragged_host);
  int32_t* len_h = reinterpret_cast<int32_t*>(off_h + L->S);
  for (int64_t s = 0, o = 0; s < L->S; o += lengths[s], ++s) {
    off_h[s] = o;
    len_h[s] = lengths[s];
  }
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  const int64_t* off = reinterpret_cast<const int64_t*>(ws);
  const int* len = reinterpret_cast<const int*>(ws + R.o_len);
  int64_t* counts = reinterpret_cast<int64_t*>(ws + R.o_counts);
  int64_t* plan = reinterpret_cast<int64_t*>(ws + R.o_plan);
  *P = LiveRagged{len, plan, row_bound, win_bound, ws_extra ? ws + R.o_extra : nullptr};
  KWS_CUDA(cudaMemcpyAsync(ws, L->ragged_host, stage_bytes, cudaMemcpyHostToDevice, st));
  KWS_CUDA(cudaEventRecord(L->ragged_copied, st));
  const kws_frontend* fe = L->fe;
  // 1) the new samples into the sample rings; counters; per-stream counts of new rows and windows
  live_ragged_append_kernel<SMP><<<(unsigned)L->S, 128, 0, st>>>(samples, off, len, L->ring, L->cap, L->window,
                                                                 L->shift, L->S, L->count, counts);
  KWS_CHECK_LAUNCH();
  // the plan: where each stream's rows and windows start in the compacted lists, and the totals
  size_t temp = R.temp;
  KWS_CUDA(cub::DeviceScan::ExclusiveSum(ws + R.o_temp, temp, counts, plan, L->S + 1, st));
  // 2) the new frame-table rows, 16 entries of the compacted list per CTA, from any streams
  const RaggedSource<false> rows{L->ring, L->frames, L->count, len, plan, L->S, L->cap, L->fcap, fe->n_mels, L->window,
                                 L->shift};
  if (row_bound > 0) {
    mfcc_kernel<false, float, RaggedSource<false>><<<(unsigned)ceil_div<int64_t>(row_bound, kFramesPerCta),
                                                     kMfccThreads, fe->smem_bytes_edges, st>>>(
        fe->t, rows, row_bound, 0, kFramesPerCta, 1, nullptr);
    KWS_CHECK_LAUNCH();
  }
  return KWS_OK;
}
template int live_ragged_append_rows<float>(const char*, kws_live_t*, const float*, const int32_t*, int64_t,
                                            const void*, const char*, void*, size_t, size_t, cudaStream_t, LiveRagged*);
template int live_ragged_append_rows<int16_t>(const char*, kws_live_t*, const int16_t*, const int32_t*, int64_t,
                                              const void*, const char*, void*, size_t, size_t, cudaStream_t,
                                              LiveRagged*);

int live_ragged_edge_frames(kws_live_t* L, const LiveRagged& P, float* edges, cudaStream_t st) {
  if (P.win_bound == 0) return KWS_OK;
  const RaggedEdgeSource src{{L->ring, L->frames, L->count, P.len, P.plan, L->S, L->cap, L->fcap, L->fe->n_mels,
                              L->window, L->shift}};
  mfcc_kernel<true, float, RaggedEdgeSource><<<(unsigned)ceil_div<int64_t>(P.win_bound, 4), kMfccThreads,
                                               L->fe->smem_bytes_edges, st>>>(L->fe->t, src, P.win_bound, L->window,
                                                                              L->T, 1, edges);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}
}  // namespace kws

template <typename SMP>
static int live_push_ragged_any(const char* who, kws_live_t* L, const SMP* samples, const int32_t* lengths, float* feat,
                                int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                                void* workspace, size_t ws_bytes, void* stream) {
  cudaStream_t st = as_stream(stream);
  LiveRagged P;
  KWS_TRY(live_ragged_append_rows(who, L, samples, lengths, capacity, feat, "feat", workspace, ws_bytes, 0, st, &P));
  const kws_frontend* fe = L->fe;
  const int64_t win_bound = P.win_bound;
  const int* len = P.len;
  const int64_t* plan = P.plan;
  // 3) the four reflect-padded edge frames of each completed window, four windows per CTA
  if (win_bound > 0) {
    const RaggedSource<true> edges{L->ring, L->frames, L->count, len, plan, L->S, L->cap, L->fcap, fe->n_mels,
                                   L->window, L->shift};
    mfcc_kernel<true, float, RaggedSource<true>><<<(unsigned)ceil_div<int64_t>(win_bound, 4), kMfccThreads,
                                                   fe->smem_bytes_edges, st>>>(fe->t, edges, win_bound, L->window,
                                                                               L->T, 1, feat);
    KWS_CHECK_LAUNCH();
  }
  // 4) interior frames from the frame rings, the window ids, and the count (one CTA even when no window completes)
  const bool vec = fe->n_mels % 4 == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0;
  const int row_v = vec ? fe->n_mels / 4 : fe->n_mels;
  const unsigned grid = (unsigned)std::max<int64_t>(win_bound, 1);
  if (vec)
    live_ragged_gather_kernel<float4><<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(L->frames), L->count, len,
                                                            plan, L->S, L->window, L->shift, L->T, L->fcap, row_v,
                                                            reinterpret_cast<float4*>(feat), win_stream, win_index,
                                                            n_windows);
  else
    live_ragged_gather_kernel<float><<<grid, 256, 0, st>>>(L->frames, L->count, len, plan, L->S, L->window, L->shift,
                                                           L->T, L->fcap, row_v, feat, win_stream, win_index, n_windows);
  KWS_CHECK_LAUNCH();
  return KWS_OK;
}

extern "C" int kws_live_push_ragged(kws_live_t* live, const float* samples, const int32_t* lengths, float* feat,
                                    int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                                    void* workspace, size_t ws_bytes, void* stream) {
  return live_push_ragged_any<float>("kws_live_push_ragged", live, samples, lengths, feat, win_stream, win_index,
                                     capacity, n_windows, workspace, ws_bytes, stream);
}

extern "C" int kws_live_push_ragged_pcm16(kws_live_t* live, const int16_t* samples, const int32_t* lengths, float* feat,
                                          int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                                          void* workspace, size_t ws_bytes, void* stream) {
  return live_push_ragged_any<int16_t>("kws_live_push_ragged_pcm16", live, samples, lengths, feat, win_stream,
                                       win_index, capacity, n_windows, workspace, ws_bytes, stream);
}
