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

// Always yields a plan; tc_cnn_supported tells whether this configuration has a tensor-core path (and why not).
int tc_cnn_create(const kws_cnn_config& cfg, TcCnn** out);
void tc_cnn_destroy(TcCnn* p);
bool tc_cnn_supported(const TcCnn* p, const char** why);
int tc_cnn_set_weights(TcCnn* p, const kws_cnn_weights& w, cudaStream_t st);
size_t tc_cnn_workspace_bytes(const TcCnn* p, int64_t B, int T, int F, int chunk);   // 0: unsupported
int tc_cnn_forward(TcCnn* p, const float* feat, int64_t B, int T, int F, float* logits, void* ws, size_t ws_bytes,
                   int chunk, LaunchProfiler* prof, cudaStream_t st);

}  // namespace kws
