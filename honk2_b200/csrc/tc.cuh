// Interface of the bf16 tensor-core (tcgen05 / TMEM / TMA) ResNet path, conv_tc.cu.
#pragma once
#include "common.cuh"

namespace kws {

struct TcResNet;  // opaque plan: packed bf16 weights, tensor maps, geometry

int tc_resnet_create(const kws_resnet_config& cfg, TcResNet** out);
void tc_resnet_destroy(TcResNet* p);
// w: torch-layout fp32 device tensors; bn_scale/bn_shift: per-layer [C] device vectors that
// the caller already derived from running_mean / running_var.
int tc_resnet_set_weights(TcResNet* p, const kws_resnet_weights& w, float* const* bn_scale,
                          float* const* bn_shift, cudaStream_t st);
// split: the "bf16x3" precision (operands as bf16 pairs hi + lo, three MMAs per product) instead of plain bf16
size_t tc_resnet_workspace_bytes(const TcResNet* p, int64_t B, int T, int F, int chunk, bool split);
int tc_resnet_forward(TcResNet* p, const float* feat, int64_t B, int T, int F, float* logits, void* ws,
                      size_t ws_bytes, int chunk, bool split, LaunchProfiler* prof, cudaStream_t st);

// Which kernel a bf16 / split-bf16 forward of a [B][T][F] batch runs: "resnet_tc_sweep_kernel" if the column-sweep
// plan can stage the map, else "resnet_tc_fused_kernel" if the position-major plan can, else "unsupported".
const char* tc_resnet_kernel_path(const TcResNet* p, int T, int F, bool split);


// ---- bf16 tensor-core path of model.CNN (cnn_tc.cu): the cnn-trad-fpool3 shape family --------------------------
struct TcCnn;   // opaque plan: packed bf16 weights and the shared-memory geometry

struct TcCnnGeom {
  int T, F, KH0, KW0, H0, WP, KH1, KW1, H1;
  int n0;        // pooled rows = H0 * WP
  int tiles0;    // conv_0 M-tiles per pool member
  int ks0;       // conv_0 K steps (two kernel rows each)
  int tiles1;    // conv_1 M-tiles (16 output rows each)
  int units1;    // KH1 * KW1 weight units
  int a_rows;    // rows of an A_e array (T*WP + WP zero rows)
  int off_w0, off_a, a_bytes, off_pool, plane_bytes, off_ring, n_ring;
  int smem_bytes;
};

// Where the first Linear (cnn_lin0_kernel) finds row r's conv_1 output.  Element k of a row is channel group
// cg = k / (H1*128), conv_1 row oh, position ow, channel c (k = cg*H1*128 + oh*128 + ow*16 + c); a kernel step of 32
// elements lies inside one (cg, oh).  row(r, K, tq) returns a cursor whose at(o) is the 16-byte group o + tq (o = k / 8).
// DenseActRows: the batch path's [B][K] activations, written by cnn_tc_fused_kernel.
struct DenseActRows {
  const __nv_bfloat16* act;
  struct Cursor {
    const uint4* p;
    __device__ __forceinline__ const uint4* at(int o) const { return p + o; }
  };
  __device__ __forceinline__ Cursor row(int64_t r, int K, int tq) const {
    return {reinterpret_cast<const uint4*>(act + r * K) + tq};
  }
};

// LiveActRows (kws_live_cnn): row r is window slot r = (stream s, window k) of a push.  Its conv_1 rows 0, 1, H1-2,
// H1-1 are the push's window-specific rows edge[r][4][1 KB]; row oh of the others is stream s's conv_1 ring row
// (k m + oh) mod cap, ring[s][cap][1 KB] (m = shift / 160).  A row is [cg][8 positions][16 channels] bf16.
struct LiveActRows {
  const __nv_bfloat16* ring;
  const __nv_bfloat16* edge;
  const int64_t* count;   // samples per stream, this push included
  int n, window, shift, K, cap, H1;
  struct Cursor {
    const __nv_bfloat16* ring;   // stream s's ring
    const __nv_bfloat16* edge;   // the slot's four window-specific rows
    int64_t k0;                  // k * m (the stream row of window row 0)
    int cap, H1, tq;
    __device__ __forceinline__ const uint4* at(int o) const {
      const int e = 8 * (o + tq);
      const int cg = e / (H1 * 128);
      const int rem = e - cg * H1 * 128;
      const int oh = rem >> 7, within = (rem & 127) + cg * 128;
      const __nv_bfloat16* p;
      if (oh < 2) p = edge + oh * 512 + within;
      else if (oh >= H1 - 2) p = edge + (oh - H1 + 4) * 512 + within;
      else {
        int64_t q = (k0 + oh) % cap;
        if (q < 0) q += cap;
        p = ring + q * 512 + within;
      }
      return reinterpret_cast<const uint4*>(p);
    }
  };
  __device__ __forceinline__ Cursor row(int64_t r, int, int tq) const {
    const int64_t s = r / K;
    const int64_t c_old = count[s] - n;
    const int64_t d = c_old - window;   // k = floor(d / shift) + 1 + (r - s K)
    const int64_t k = (d >= 0 ? d / shift : -((-d + shift - 1) / shift)) + 1 + (r - s * K);
    return {ring + s * (int64_t)cap * 512, edge + r * 2048, k * (shift / 160), cap, H1, tq};
  }
};

// RaggedActRows (ragged pushes of kws_live_cnn): row r is window r of the push's compacted list, the (stream s, window
// k) of live_ragged_append_rows' plan (low 32 bits of plan[s]: the windows of the streams before s; plan[S]: M), with
// its window-specific rows at edge[r] and the others in stream s's ring as for LiveActRows.  Rows past the device's M
// (the launch covers the host's bound) read window min(r, M - 1), or window 0 of the last stream when M = 0: valid
// memory, results nobody reads.
struct RaggedActRows {
  const __nv_bfloat16* ring;
  const __nv_bfloat16* edge;
  const int64_t* count;   // samples per stream, this push included
  const int* len;         // samples per stream of this push
  const int64_t* plan;
  int S, window, shift, cap, H1;
  using Cursor = LiveActRows::Cursor;
  __device__ __forceinline__ Cursor row(int64_t r, int, int tq) const {
    const int64_t M = __ldg(plan + S) & 0xffffffffll;
    r = r < M ? r : (M > 0 ? M - 1 : 0);
    int lo = 0, hi = S;   // (plan[lo] <= r < plan[hi] in the low words)
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if ((__ldg(plan + mid) & 0xffffffffll) <= r) lo = mid;
      else hi = mid;
    }
    const int64_t d = __ldg(count + lo) - __ldg(len + lo) - window;   // first window = max(0, floor(d / shift) + 1)
    int64_t k = (d >= 0 ? d / shift : -((-d + shift - 1) / shift)) + 1;
    k = (k > 0 ? k : 0) + r - (__ldg(plan + lo) & 0xffffffffll);
    return {ring + lo * (int64_t)cap * 512, edge + r * 2048, k * (shift / 160), cap, H1, tq};
  }
};

// What a live CNN state needs of a plan: geometry, packed conv weights (tc_cnn_set_weights' layouts), sizes.
struct TcCnnView {
  TcCnnGeom g;
  const __nv_bfloat16 *w0, *w1;   // [ks0][2][64][8], [KH1*KW1][4][2][64][8]
  const float *b0, *b1;
  size_t blob_bytes;              // device bytes of the plan's packed tensors
  int n_labels;
};
bool tc_cnn_view(const TcCnn* p, TcCnnView* v);   // false: no tensor-core path
// A new plan of src's configuration holding a copy of src's packed weights (copied on st).
int tc_cnn_copy(const TcCnn* src, TcCnn** out, cudaStream_t st);
// The first Linear over rows addressed by `rows` (the batch path's split-K slices), then the remaining layers, for B
// windows.  partial: kTcCnnLin0Split * B * 32 floats; logits [B][n_labels].
int tc_cnn_live_linear(const TcCnn* p, const LiveActRows& rows, int64_t B, float* partial, float* logits,
                       cudaStream_t st);
int tc_cnn_live_linear(const TcCnn* p, const RaggedActRows& rows, int64_t B, float* partial, float* logits,
                       cudaStream_t st);
// The tensor-core plan of a CNN model handle (model.cu): nullptr for a ResNet; *weights_set: kws_cnn_set_weights ran.
const TcCnn* model_tc_cnn(const kws_model_t* m, bool* weights_set);
constexpr int kTcCnnLin0Split = 8;

// Always yields a plan; tc_cnn_supported tells whether this configuration has a tensor-core path (and why not).
int tc_cnn_create(const kws_cnn_config& cfg, TcCnn** out);
void tc_cnn_destroy(TcCnn* p);
bool tc_cnn_supported(const TcCnn* p, const char** why);
int tc_cnn_set_weights(TcCnn* p, const kws_cnn_weights& w, cudaStream_t st);
size_t tc_cnn_workspace_bytes(const TcCnn* p, int64_t B, int T, int F, int chunk);   // 0: unsupported
int tc_cnn_forward(TcCnn* p, const float* feat, int64_t B, int T, int F, float* logits, void* ws, size_t ws_bytes,
                   int chunk, LaunchProfiler* prof, cudaStream_t st);

}  // namespace kws
