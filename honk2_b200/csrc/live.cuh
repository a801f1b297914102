// Internal interface of the live front-end (mfcc.cu) for the states built on it (live_cnn.cu): the stages of the
// uniform push and of the ragged push that do not depend on what the state keeps.
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

// A ragged push's plan on the device.  len[s]: samples stream s brings; plan[s] (s = 0 .. S): exclusive scan of the
// per-stream counts of new frame-table rows (high 32 bits) and completed windows (low 32 bits), plan[S] the totals.  The
// bounds are the host's: row_bound = sum ceil(n_s / 160), win_bound = sum ceil(n_s / shift).  extra: the caller's part
// of the workspace (null when it asked for none).
struct LiveRagged {
  const int* len;
  const int64_t* plan;
  int64_t row_bound, win_bound;
  void* extra;
};
// Workspace of a ragged push whose caller needs `extra` bytes of its own (0 if the scan size query fails).
size_t live_ragged_workspace_bytes(const char* who, const kws_live_t* L, size_t extra);
// Launches 1 and 2 of kws_live_push_ragged and the plan's scan: the samples into the sample rings (counters advance),
// then the new frame-table rows.  First checks the whole push on the host (KWS_ERR_INVALID, nothing staged or
// launched): lengths in [0, max_push], capacity >= win_bound, samples given when any are pushed, `out` (the caller's
// output, named out_name in the message) given when a window can complete, and a workspace of
// live_ragged_workspace_bytes(L, ws_extra) bytes.
template <typename SMP>
int live_ragged_append_rows(const char* who, kws_live_t* L, const SMP* samples, const int32_t* lengths,
                            int64_t capacity, const void* out, const char* out_name, void* workspace, size_t ws_bytes,
                            size_t ws_extra, cudaStream_t st, LiveRagged* P);
// Launch 3 for a state that keeps no features: the four edge frames of each completed window into edges [M][4][n_mels]
// (frames t = 0, 1, T-2, T-1), window i of the compacted list at row i.
int live_ragged_edge_frames(kws_live_t* L, const LiveRagged& P, float* edges, cudaStream_t st);

}  // namespace kws
