// Internal interface of the live front-end (mfcc.cu) for the states built on it (live_cnn.cu).
#pragma once
#include "common.cuh"

struct kws_frontend;

// One device allocation per state: sample rings [S][cap] f32, frame rings [S][fcap][n_mels] f32, counters [S] i64,
// first-window ring positions [S] i32.  Ragged pushes add a pinned host staging buffer for their per-stream sample
// offsets and lengths and the event that marks its last copy done; both are created by the first ragged push.
struct kws_live {
  const kws_frontend* fe;
  int S, window, shift, max_push, T, cap, fcap;
  void* dev;
  float* ring;
  float* frames;
  int64_t* count;
  int* wpos;
  void* ragged_host = nullptr;
  cudaEvent_t ragged_copied = nullptr;
};

namespace kws {

// Launches 1 and 2 of kws_live_push: the push's n samples per stream into the sample rings (counters advance), then the
// n / 160 frame-table rows per stream it completes.  Checks n against the state (KWS_ERR_INVALID, nothing launched).
template <typename SMP>
int live_append_rows(const char* who, kws_live_t* L, const SMP* chunk, int n, cudaStream_t st);
// Launch 3 for a state that keeps no features: the four reflect-padded edge frames (t = 0, 1, T-2, T-1) of each of the
// push's S K window slots into edges [S K][4][n_mels].
int live_edge_frames(kws_live_t* L, int n, float* edges, cudaStream_t st);

}  // namespace kws
