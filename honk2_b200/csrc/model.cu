// Model handles of the honk2_b200 C ABI: construction from the reference's config fields,
// weight repacking (the library owns device copies of everything), and the layer-by-layer
// forward orchestration for model.ResNet (/root/reference/model/resnet.py:11-60) and model.CNN
// (/root/reference/model/cnn.py:12-107).  The batch is processed in sub-batches ("chunks") so
// that the ping-pong activation buffers stay L2 resident.
#include "kernels.cuh"
#include "tc.cuh"
#include <vector>
#include <algorithm>

namespace kws {

constexpr float kBnEps = 1e-5f;  // nn.BatchNorm2d default (resnet.py:27)

enum { KIND_RESNET = 0, KIND_CNN = 1 };

struct Model {
  int kind = KIND_RESNET;
  kws_resnet_config rc{};
  kws_cnn_config cc{};
  bool weights_set = false;
  int64_t last_launches = 0;
  int chunk[3] = {0, 0, 0};   // per precision
  bool f32_resident = true;   // fp32 C -> C layers on the resident-weight persistent kernel (HONK2_F32_RESIDENT=0: the tile-per-CTA kernel)
  LaunchProfiler prof;

  // ---- ResNet fp32 packed weights
  float* blob = nullptr;  // one allocation
  size_t blob_bytes = 0;
  float* r_conv0 = nullptr;               // [C][9]
  std::vector<float*> r_conv;             // [n][C][9][CG*QP]
  std::vector<float*> r_bn_scale, r_bn_shift;  // [n][C]
  float* r_out_w = nullptr;               // [L][C]
  float* r_out_b = nullptr;               // [L]
  TcResNet* tc = nullptr;                 // bf16 tensor-core plan (conv_tc.cu)
  TcCnn* tcc = nullptr;                   // bf16 tensor-core plan of the CNN family (cnn_tc.cu)

  // ---- CNN packed weights
  float *c_conv0_w = nullptr, *c_conv0_b = nullptr, *c_conv1_w = nullptr, *c_conv1_b = nullptr;
  float *c_lin_w[4] = {nullptr, nullptr, nullptr, nullptr}, *c_lin_b[4] = {nullptr, nullptr, nullptr, nullptr};
  int c_lin_in[4] = {0, 0, 0, 0}, c_lin_out[4] = {0, 0, 0, 0};  // lin_0, dnn_0, dnn_1, lin_1 (out 0 = absent)
  int c_h0 = 0, c_w0 = 0, c_hp0 = 0, c_wp0 = 0, c_h1 = 0, c_w1 = 0, c_hp1 = 0, c_wp1 = 0, c_flat = 0;
};

// ---------------------------------------------------------------------------------------------
// packing kernels (run once per load_state_dict)

// torch [Cout][Cin][3][3] -> [Cin][9][CG*QP], zero padded (QP = Q rounded up to a multiple of 4)
__global__ void pack_conv3x3_f32_kernel(const float* __restrict__ w, float* __restrict__ out, int C, int Q,
                                        int CG) {
  const int QP = (Q + 3) & ~3;
  const int total = C * 9 * CG * QP;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int q = i % QP;
    int t = i / QP;
    const int cg = t % CG; t /= CG;
    const int tap = t % 9;
    const int ci = t / 9;
    const int co = cg * Q + q;
    out[i] = (q < Q && co < C) ? w[((int64_t)co * C + ci) * 9 + tap] : 0.f;
  }
}

__global__ void pack_bn_kernel(const float* __restrict__ mean, const float* __restrict__ var,
                               float* __restrict__ scale, float* __restrict__ shift, int C, float eps) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    const float s = 1.0f / sqrtf(var[c] + eps);
    scale[c] = s;
    shift[c] = -mean[c] * s;
  }
}

// torch [Cout][Cin][KH][KW] -> [Cin][KH][KW][CoutPad], zero padded
__global__ void pack_conv_gen_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin,
                                     int KHW, int CoutPad) {
  const int64_t total = (int64_t)Cin * KHW * CoutPad;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % CoutPad);
    const int64_t t = i / CoutPad;
    const int k = (int)(t % KHW);
    const int ci = (int)(t / KHW);
    out[i] = co < Cout ? w[((int64_t)co * Cin + ci) * KHW + k] : 0.f;
  }
}

struct BlobPlan {
  size_t off = 0;
  size_t take(size_t floats) {
    const size_t o = off;
    off += round_up<size_t>(floats * sizeof(float), 256);
    return o;
  }
};

}  // namespace kws

using namespace kws;

struct kws_model : kws::Model {};

const TcCnn* kws::model_tc_cnn(const kws_model_t* m, bool* weights_set) {
  *weights_set = m && m->weights_set;
  return m && m->kind == KIND_CNN ? m->tcc : nullptr;
}

// =============================================================================================
// ResNet

extern "C" int kws_resnet_create(const kws_resnet_config* cfg, kws_model_t** out) {
  KWS_REQUIRE(out != nullptr && cfg != nullptr, "kws_resnet_create: null argument");
  *out = nullptr;
  KWS_REQUIRE(cfg->n_layers >= 0 && cfg->n_layers <= 256, "kws_resnet_create: n_layers=%d", cfg->n_layers);
  KWS_REQUIRE(cfg->n_maps >= 1 && cfg->n_maps <= 72, "kws_resnet_create: n_feature_maps=%d not in [1,72]",
              cfg->n_maps);
  KWS_REQUIRE(cfg->n_labels >= 1 && cfg->n_labels <= 1024, "kws_resnet_create: n_labels=%d", cfg->n_labels);
  KWS_REQUIRE((cfg->pool_h == 0 && cfg->pool_w == 0) || (cfg->pool_h >= 1 && cfg->pool_w >= 1),
              "kws_resnet_create: pool must be 0,0 (absent) or positive");
  KWS_REQUIRE(!cfg->use_dilation || cfg->n_layers <= 60, "kws_resnet_create: dilation overflows at %d layers",
              cfg->n_layers);
  KWS_TRY(kws_device_info(nullptr, nullptr, nullptr));
  kws_model* m = new kws_model();
  m->kind = KIND_RESNET;
  m->rc = *cfg;
  { const char* e = getenv("HONK2_F32_RESIDENT"); m->f32_resident = !(e && e[0] == '0'); }
  const int C = cfg->n_maps, n = cfg->n_layers, L = cfg->n_labels;
  const int Q = conv3x3_f32_q(C), CG = ceil_div(C, Q);
  BlobPlan bp;
  const size_t o_conv0 = bp.take((size_t)C * 9);
  std::vector<size_t> o_conv(n), o_sc(n), o_sh(n);
  for (int i = 0; i < n; ++i) {
    o_conv[i] = bp.take((size_t)C * 9 * CG * ((Q + 3) & ~3));
    o_sc[i] = bp.take(C);
    o_sh[i] = bp.take(C);
  }
  const size_t o_ow = bp.take((size_t)L * C), o_ob = bp.take(L);
  m->blob_bytes = bp.off;
  cudaError_t e = cudaMalloc(&m->blob, m->blob_bytes);
  if (e != cudaSuccess) {
    set_error("kws_resnet_create: cudaMalloc(%zu) failed: %s", m->blob_bytes, cudaGetErrorString(e));
    delete m;
    return KWS_ERR_CUDA;
  }
  char* base = reinterpret_cast<char*>(m->blob);
  m->r_conv0 = reinterpret_cast<float*>(base + o_conv0);
  m->r_conv.resize(n); m->r_bn_scale.resize(n); m->r_bn_shift.resize(n);
  for (int i = 0; i < n; ++i) {
    m->r_conv[i] = reinterpret_cast<float*>(base + o_conv[i]);
    m->r_bn_scale[i] = reinterpret_cast<float*>(base + o_sc[i]);
    m->r_bn_shift[i] = reinterpret_cast<float*>(base + o_sh[i]);
  }
  m->r_out_w = reinterpret_cast<float*>(base + o_ow);
  m->r_out_b = reinterpret_cast<float*>(base + o_ob);
  int st = tc_resnet_create(*cfg, &m->tc);
  if (st != KWS_OK) {
    cudaFree(m->blob);
    delete m;
    return st;
  }
  *out = m;
  return KWS_OK;
}

extern "C" int kws_resnet_set_weights(kws_model_t* m, const kws_resnet_weights* w, void* stream) {
  KWS_REQUIRE(m != nullptr && w != nullptr, "kws_resnet_set_weights: null argument");
  KWS_REQUIRE(m->kind == KIND_RESNET, "kws_resnet_set_weights: handle is not a ResNet");
  const int C = m->rc.n_maps, n = m->rc.n_layers, L = m->rc.n_labels;
  KWS_REQUIRE(w->conv0_w && w->out_w && w->out_b, "kws_resnet_set_weights: null tensor");
  KWS_REQUIRE(n == 0 || (w->conv_w && w->bn_mean && w->bn_var), "kws_resnet_set_weights: null layer table");
  cudaStream_t st = as_stream(stream);
  const int Q = conv3x3_f32_q(C), CG = ceil_div(C, Q);
  KWS_CUDA(cudaMemcpyAsync(m->r_conv0, w->conv0_w, sizeof(float) * C * 9, cudaMemcpyDeviceToDevice, st));
  for (int i = 0; i < n; ++i) {
    KWS_REQUIRE(w->conv_w[i] && w->bn_mean[i] && w->bn_var[i], "kws_resnet_set_weights: layer %d has a null tensor",
                i + 1);
    pack_conv3x3_f32_kernel<<<ceil_div(C * 9 * CG * ((Q + 3) & ~3), 256), 256, 0, st>>>(w->conv_w[i], m->r_conv[i], C, Q, CG);
    KWS_CUDA(cudaGetLastError());
    pack_bn_kernel<<<ceil_div(C, 128), 128, 0, st>>>(w->bn_mean[i], w->bn_var[i], m->r_bn_scale[i],
                                                    m->r_bn_shift[i], C, kBnEps);
    KWS_CUDA(cudaGetLastError());
  }
  KWS_CUDA(cudaMemcpyAsync(m->r_out_w, w->out_w, sizeof(float) * L * C, cudaMemcpyDeviceToDevice, st));
  KWS_CUDA(cudaMemcpyAsync(m->r_out_b, w->out_b, sizeof(float) * L, cudaMemcpyDeviceToDevice, st));
  KWS_TRY(tc_resnet_set_weights(m->tc, *w, m->r_bn_scale.data(), m->r_bn_shift.data(), st));
  m->weights_set = true;
  return KWS_OK;
}

namespace kws {

static int64_t default_chunk(const Model* m, int precision, int64_t per_utt_bytes) {
  if (m->chunk[precision] > 0) return m->chunk[precision];
  // The fp32 CUDA-core path is FMA-bound (a layer moves ~2.2 MB per utterance through DRAM at < 10 % of the HBM
  // bandwidth), so its sub-batch only has to be large enough that the persistent convolution kernel's last wave is a
  // small fraction of a launch: ~2 GB of activations.
  int64_t c = (2048ll << 20) / (3 * std::max<int64_t>(per_utt_bytes, 1));
  if (c < 8) c = 8;
  if (c > 4096) c = 4096;
  return c;
}

static size_t resnet_ws_f32(const Model* m, int64_t B, int T, int F, int64_t* chunk_out) {
  int H, W;
  resnet_map(m->rc, T, F, &H, &W);
  const int64_t per = (int64_t)m->rc.n_maps * H * W * sizeof(float);
  int64_t chunk = default_chunk(m, KWS_FP32, per);
  if (chunk > B) chunk = B;
  if (chunk < 1) chunk = 1;
  if (chunk_out) *chunk_out = chunk;
  return 3 * round_up<size_t>((size_t)chunk * per, 256);
}

static int resnet_forward_f32(Model* m, const float* feat, int64_t B, int T, int F, float* logits, void* ws,
                              size_t ws_bytes, cudaStream_t st) {
  const kws_resnet_config& c = m->rc;
  int H, W;
  resnet_map(c, T, F, &H, &W);
  KWS_REQUIRE(H >= 1 && W >= 1, "ResNet: input %dx%d is smaller than the pooling window", T, F);
  int64_t chunk = 0;
  const size_t need = resnet_ws_f32(m, B, T, F, &chunk);
  if (ws_bytes < need || ws == nullptr) {
    set_error("ResNet fp32 forward needs %zu bytes of workspace, got %zu", need, ws_bytes);
    return KWS_ERR_WORKSPACE;
  }
  const int C = c.n_maps;
  const size_t buf = round_up<size_t>((size_t)chunk * C * H * W * sizeof(float), 256);
  float* P = reinterpret_cast<float*>(static_cast<char*>(ws));            // skip tensor / conv_0 output
  float* A0 = reinterpret_cast<float*>(static_cast<char*>(ws) + buf);
  float* A1 = reinterpret_cast<float*>(static_cast<char*>(ws) + 2 * buf);
  const auto [ph, pw] = resnet_pool(c);
  // equal sub-batches (2048 utterances = 3 x 683, not 985 + 985 + 78): the persistent kernels' last wave stays full
  if (B > chunk) chunk = ceil_div<int64_t>(B, ceil_div<int64_t>(B, chunk));
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int64_t nb = min(chunk, B - b0);
    m->prof.tick(1, st);
    KWS_TRY(launch_conv0_f32(feat + b0 * (int64_t)T * F, m->r_conv0, P, nb, T, F, C, ph, pw, st));
    const float* x = P;
    float* pp[2] = {A0, A1};
    int flip = 0;
    for (int i = 1; i <= c.n_layers; ++i) {
      Conv3x3F32 a;
      a.x = x;
      a.wt = m->r_conv[i - 1];
      a.prev_in = (i % 2 == 0) ? P : nullptr;   // resnet.py:51-53
      a.prev_out = (i % 2 == 0) ? P : nullptr;
      a.y = pp[flip];
      a.bn_scale = m->r_bn_scale[i - 1];
      a.bn_shift = m->r_bn_shift[i - 1];
      a.B = nb; a.C = C; a.H = H; a.W = W; a.d = resnet_dilation(c, i);
      a.resident = m->f32_resident ? 1 : 0;
      m->prof.tick(0, st);
      KWS_TRY(launch_conv3x3_f32(a, st));
      x = pp[flip];
      flip ^= 1;
    }
    m->prof.tick(1, st);
    KWS_TRY(launch_tail_f32(x, m->r_out_w, m->r_out_b, logits + b0 * c.n_labels, nb, C, H * W, c.n_labels, st));
  }
  return KWS_OK;
}

}  // namespace kws

// =============================================================================================
// CNN

extern "C" int kws_cnn_create(const kws_cnn_config* cfg, kws_model_t** out) {
  KWS_REQUIRE(out != nullptr && cfg != nullptr, "kws_cnn_create: null argument");
  *out = nullptr;
  const kws_cnn_config& c = *cfg;
  KWS_REQUIRE(c.time >= 1 && c.freq >= 1, "kws_cnn_create: time/frequency must be positive");
  KWS_REQUIRE(c.conv0_out >= 1 && c.conv0_kh >= 1 && c.conv0_kw >= 1 && c.conv0_sh >= 1 && c.conv0_sw >= 1,
              "kws_cnn_create: bad conv_0");
  KWS_REQUIRE(c.pool0_kh >= 1 && c.pool0_kw >= 1, "kws_cnn_create: bad pool_0");
  KWS_REQUIRE(c.n_labels >= 1, "kws_cnn_create: n_labels");
  KWS_TRY(kws_device_info(nullptr, nullptr, nullptr));
  kws_model* m = new kws_model();
  m->kind = KIND_CNN;
  m->cc = c;
  { const char* e = getenv("HONK2_F32_RESIDENT"); m->f32_resident = !(e && e[0] == '0'); }
  // utils/torch_utils.py:29-65 (floor mode, no padding, dilation 1)
  m->c_h0 = (c.time - c.conv0_kh) / c.conv0_sh + 1;
  m->c_w0 = (c.freq - c.conv0_kw) / c.conv0_sw + 1;
  bool ok = c.time >= c.conv0_kh && c.freq >= c.conv0_kw && m->c_h0 >= c.pool0_kh && m->c_w0 >= c.pool0_kw;
  m->c_hp0 = ok ? m->c_h0 / c.pool0_kh : 0;
  m->c_wp0 = ok ? m->c_w0 / c.pool0_kw : 0;
  int Cl = c.conv0_out, Hl = m->c_hp0, Wl = m->c_wp0;
  if (ok && c.conv1_out > 0) {
    ok = c.conv1_kh >= 1 && c.conv1_kw >= 1 && c.conv1_sh >= 1 && c.conv1_sw >= 1 && c.pool1_kh >= 1 &&
         c.pool1_kw >= 1 && Hl >= c.conv1_kh && Wl >= c.conv1_kw;
    if (ok) {
      m->c_h1 = (Hl - c.conv1_kh) / c.conv1_sh + 1;
      m->c_w1 = (Wl - c.conv1_kw) / c.conv1_sw + 1;
      ok = m->c_h1 >= c.pool1_kh && m->c_w1 >= c.pool1_kw;
      m->c_hp1 = ok ? m->c_h1 / c.pool1_kh : 0;
      m->c_wp1 = ok ? m->c_w1 / c.pool1_kw : 0;
      Cl = c.conv1_out; Hl = m->c_hp1; Wl = m->c_wp1;
    }
  }
  if (!ok || Hl < 1 || Wl < 1) {
    set_error("kws_cnn_create: the conv/pool stack does not fit a %dx%d input", c.time, c.freq);
    delete m;
    return KWS_ERR_INVALID;
  }
  m->c_flat = Cl * Hl * Wl;
  const int outs[4] = {c.lin0_out, c.dnn0_out, c.dnn1_out, c.n_labels};
  int in = m->c_flat;
  BlobPlan bp;
  const int pad0 = round_up(c.conv0_out, 8);
  const size_t o_c0w = bp.take((size_t)c.conv0_kh * c.conv0_kw * pad0), o_c0b = bp.take(c.conv0_out);
  size_t o_c1w = 0, o_c1b = 0;
  if (c.conv1_out > 0) {
    o_c1w = bp.take((size_t)c.conv0_out * c.conv1_kh * c.conv1_kw * round_up(c.conv1_out, 8));
    o_c1b = bp.take(c.conv1_out);
  }
  size_t o_lw[4] = {0, 0, 0, 0}, o_lb[4] = {0, 0, 0, 0};
  for (int i = 0; i < 4; ++i) {
    if (outs[i] <= 0) continue;
    m->c_lin_in[i] = in;
    m->c_lin_out[i] = outs[i];
    o_lw[i] = bp.take((size_t)outs[i] * in);
    o_lb[i] = bp.take(outs[i]);
    in = outs[i];
  }
  m->blob_bytes = bp.off;
  cudaError_t e = cudaMalloc(&m->blob, m->blob_bytes);
  if (e != cudaSuccess) {
    set_error("kws_cnn_create: cudaMalloc(%zu) failed: %s", m->blob_bytes, cudaGetErrorString(e));
    delete m;
    return KWS_ERR_CUDA;
  }
  char* base = reinterpret_cast<char*>(m->blob);
  m->c_conv0_w = reinterpret_cast<float*>(base + o_c0w);
  m->c_conv0_b = reinterpret_cast<float*>(base + o_c0b);
  if (c.conv1_out > 0) {
    m->c_conv1_w = reinterpret_cast<float*>(base + o_c1w);
    m->c_conv1_b = reinterpret_cast<float*>(base + o_c1b);
  }
  for (int i = 0; i < 4; ++i)
    if (m->c_lin_out[i] > 0) {
      m->c_lin_w[i] = reinterpret_cast<float*>(base + o_lw[i]);
      m->c_lin_b[i] = reinterpret_cast<float*>(base + o_lb[i]);
    }
  {
    const int st = tc_cnn_create(c, &m->tcc);
    if (st != KWS_OK) {
      cudaFree(m->blob);
      delete m;
      return st;
    }
  }
  *out = m;
  return KWS_OK;
}

extern "C" int kws_cnn_set_weights(kws_model_t* m, const kws_cnn_weights* w, void* stream) {
  KWS_REQUIRE(m != nullptr && w != nullptr, "kws_cnn_set_weights: null argument");
  KWS_REQUIRE(m->kind == KIND_CNN, "kws_cnn_set_weights: handle is not a CNN");
  const kws_cnn_config& c = m->cc;
  cudaStream_t st = as_stream(stream);
  KWS_REQUIRE(w->conv0_w && w->conv0_b && w->lin1_w && w->lin1_b, "kws_cnn_set_weights: null tensor");
  {
    const int khw = c.conv0_kh * c.conv0_kw, pad = round_up(c.conv0_out, 8);
    pack_conv_gen_kernel<<<ceil_div(khw * pad, 256), 256, 0, st>>>(w->conv0_w, m->c_conv0_w, c.conv0_out, 1, khw, pad);
    KWS_CUDA(cudaGetLastError());
    KWS_CUDA(cudaMemcpyAsync(m->c_conv0_b, w->conv0_b, sizeof(float) * c.conv0_out, cudaMemcpyDeviceToDevice, st));
  }
  if (c.conv1_out > 0) {
    KWS_REQUIRE(w->conv1_w && w->conv1_b, "kws_cnn_set_weights: conv_1 tensors are null");
    const int khw = c.conv1_kh * c.conv1_kw, pad = round_up(c.conv1_out, 8);
    const int64_t total = (int64_t)c.conv0_out * khw * pad;
    pack_conv_gen_kernel<<<(unsigned)std::min<int64_t>(ceil_div<int64_t>(total, 256), 4096), 256, 0, st>>>(
        w->conv1_w, m->c_conv1_w, c.conv1_out, c.conv0_out, khw, pad);
    KWS_CUDA(cudaGetLastError());
    KWS_CUDA(cudaMemcpyAsync(m->c_conv1_b, w->conv1_b, sizeof(float) * c.conv1_out, cudaMemcpyDeviceToDevice, st));
  }
  const float* lw[4] = {w->lin0_w, w->dnn0_w, w->dnn1_w, w->lin1_w};
  const float* lb[4] = {w->lin0_b, w->dnn0_b, w->dnn1_b, w->lin1_b};
  for (int i = 0; i < 4; ++i) {
    if (m->c_lin_out[i] <= 0) continue;
    KWS_REQUIRE(lw[i] && lb[i], "kws_cnn_set_weights: linear layer %d tensors are null", i);
    KWS_CUDA(cudaMemcpyAsync(m->c_lin_w[i], lw[i], sizeof(float) * (size_t)m->c_lin_out[i] * m->c_lin_in[i],
                             cudaMemcpyDeviceToDevice, st));
    KWS_CUDA(cudaMemcpyAsync(m->c_lin_b[i], lb[i], sizeof(float) * m->c_lin_out[i], cudaMemcpyDeviceToDevice, st));
  }
  KWS_TRY(tc_cnn_set_weights(m->tcc, *w, st));
  m->weights_set = true;
  return KWS_OK;
}

namespace kws {

static int64_t cnn_max_act(const Model* m) {
  const kws_cnn_config& c = m->cc;
  int64_t mx = (int64_t)c.conv0_out * m->c_h0 * m->c_w0;
  if (c.conv1_out > 0) mx = std::max<int64_t>(mx, (int64_t)c.conv1_out * m->c_h1 * m->c_w1);
  for (int i = 0; i < 4; ++i) mx = std::max<int64_t>(mx, m->c_lin_out[i]);
  return mx;
}

static size_t cnn_ws_f32(const Model* m, int64_t B, int64_t* chunk_out) {
  const int64_t per = cnn_max_act(m) * (int64_t)sizeof(float);
  int64_t chunk = m->chunk[KWS_FP32] > 0 ? m->chunk[KWS_FP32] : 1024;   // (~1.4 GB of scratch for cnn-trad-fpool3)
  if (chunk > B) chunk = B;
  if (chunk < 1) chunk = 1;
  if (chunk_out) *chunk_out = chunk;
  return 2 * round_up<size_t>((size_t)chunk * per, 256);
}

static int cnn_forward_f32(Model* m, const float* feat, int64_t B, int T, int F, float* logits, void* ws,
                           size_t ws_bytes, cudaStream_t st) {
  const kws_cnn_config& c = m->cc;
  KWS_REQUIRE(T == c.time && F == c.freq, "CNN: input is %dx%d but the model was built for %dx%d (cnn.py:16-17)", T, F,
              c.time, c.freq);
  int64_t chunk = 0;
  const size_t need = cnn_ws_f32(m, B, &chunk);
  if (ws_bytes < need || ws == nullptr) {
    set_error("CNN fp32 forward needs %zu bytes of workspace, got %zu", need, ws_bytes);
    return KWS_ERR_WORKSPACE;
  }
  float* buf[2] = {reinterpret_cast<float*>(ws), reinterpret_cast<float*>(static_cast<char*>(ws) + need / 2)};
  for (int64_t b0 = 0; b0 < B; b0 += chunk) {
    const int64_t nb = min(chunk, B - b0);
    int cur = 0;
    ConvGenF32 a;
    a.row_kernel = m->f32_resident ? 1 : 0;
    a.x = feat + b0 * (int64_t)T * F; a.wt = m->c_conv0_w; a.bias = m->c_conv0_b; a.y = buf[cur];
    a.B = nb; a.Cin = 1; a.H = T; a.W = F; a.Cout = c.conv0_out;
    a.KH = c.conv0_kh; a.KW = c.conv0_kw; a.SH = c.conv0_sh; a.SW = c.conv0_sw;
    m->prof.tick(1, st);
    KWS_TRY(launch_conv_gen_f32(a, st));
    if (c.pool0_kh != 1 || c.pool0_kw != 1) {
      m->prof.tick(1, st);
      KWS_TRY(launch_maxpool_f32(buf[cur], buf[cur ^ 1], nb * c.conv0_out, m->c_h0, m->c_w0, c.pool0_kh, c.pool0_kw, st));
      cur ^= 1;
    }
    if (c.conv1_out > 0) {
      a.x = buf[cur]; a.wt = m->c_conv1_w; a.bias = m->c_conv1_b; a.y = buf[cur ^ 1];
      a.Cin = c.conv0_out; a.H = m->c_hp0; a.W = m->c_wp0; a.Cout = c.conv1_out;
      a.KH = c.conv1_kh; a.KW = c.conv1_kw; a.SH = c.conv1_sh; a.SW = c.conv1_sw;
      m->prof.tick(0, st);
      KWS_TRY(launch_conv_gen_f32(a, st));
      cur ^= 1;
      if (c.pool1_kh != 1 || c.pool1_kw != 1) {
        m->prof.tick(1, st);
        KWS_TRY(launch_maxpool_f32(buf[cur], buf[cur ^ 1], nb * c.conv1_out, m->c_h1, m->c_w1, c.pool1_kh, c.pool1_kw, st));
        cur ^= 1;
      }
    }
    for (int i = 0; i < 4; ++i) {
      if (m->c_lin_out[i] <= 0) continue;
      float* dst = (i == 3) ? logits + b0 * c.n_labels : buf[cur ^ 1];
      // the rest of the output buffer holds the split-K partial sums of a long reduction (the first Linear: K = 37376)
      const size_t out_floats = (size_t)nb * m->c_lin_out[i];
      float* scratch = (i == 3) ? nullptr : buf[cur ^ 1] + round_up<size_t>(out_floats, 64);
      const size_t scratch_floats = (i == 3) ? 0 : need / 2 / sizeof(float) - round_up<size_t>(out_floats, 64);
      m->prof.tick(1, st);
      KWS_TRY(launch_linear_f32(buf[cur], m->c_lin_w[i], m->c_lin_b[i], dst, nb, m->c_lin_out[i], m->c_lin_in[i], scratch,
                                scratch_floats, st));
      cur ^= 1;
    }
  }
  return KWS_OK;
}

}  // namespace kws

// =============================================================================================
// common entry points

extern "C" void kws_model_destroy(kws_model_t* m) {
  if (!m) return;
  if (m->tc) tc_resnet_destroy(m->tc);
  if (m->tcc) tc_cnn_destroy(m->tcc);
  if (m->blob) cudaFree(m->blob);
  delete m;
}

extern "C" int kws_model_n_labels(const kws_model_t* m) {
  if (!m) return 0;
  return m->kind == KIND_RESNET ? m->rc.n_labels : m->cc.n_labels;
}

extern "C" size_t kws_model_workspace_bytes(const kws_model_t* m, int64_t B, int T, int F, int precision) {
  if (!m || B < 0 || T < 1 || F < 1) return 0;
  if (B == 0) return 256;
  if (m->kind == KIND_RESNET) {
    if (precision == KWS_FP32) return resnet_ws_f32(m, B, T, F, nullptr);
    if (precision == KWS_BF16 || precision == KWS_BF16X3)
      return tc_resnet_workspace_bytes(m->tc, B, T, F, m->chunk[precision], precision == KWS_BF16X3);
    return 0;
  }
  if (precision == KWS_FP32) return cnn_ws_f32(m, B, nullptr);
  if (precision == KWS_BF16) return tc_cnn_workspace_bytes(m->tcc, B, T, F, m->chunk[KWS_BF16]);
  return 0;
}

extern "C" int kws_model_forward(kws_model_t* m, const float* feat, int64_t B, int T, int F, float* logits,
                                 int precision, void* workspace, size_t workspace_bytes, void* stream) {
  KWS_REQUIRE(m != nullptr, "kws_model_forward: model is null");
  KWS_REQUIRE(m->weights_set, "kws_model_forward: weights were never set");
  KWS_REQUIRE(B >= 0 && T >= 1 && F >= 1, "kws_model_forward: bad shape B=%lld T=%d F=%d", (long long)B, T, F);
  KWS_REQUIRE(precision == KWS_FP32 || precision == KWS_BF16 || precision == KWS_BF16X3,
              "kws_model_forward: unknown precision %d", precision);
  if (B == 0) return KWS_OK;
  KWS_REQUIRE(feat != nullptr && logits != nullptr, "kws_model_forward: null buffer");
  g_launches = 0;
  int st;
  if (m->kind == KIND_RESNET) {
    if (precision == KWS_FP32)
      st = resnet_forward_f32(m, feat, B, T, F, logits, workspace, workspace_bytes, as_stream(stream));
    else
      st = tc_resnet_forward(m->tc, feat, B, T, F, logits, workspace, workspace_bytes, m->chunk[precision],
                             precision == KWS_BF16X3, &m->prof, as_stream(stream));
  } else {
    const char* why = "";
    if (precision == KWS_BF16 && tc_cnn_supported(m->tcc, &why)) {
      st = tc_cnn_forward(m->tcc, feat, B, T, F, logits, workspace, workspace_bytes, m->chunk[KWS_BF16], &m->prof,
                          as_stream(stream));
    } else if (precision != KWS_FP32) {
      set_error("kws_model_forward: this CNN configuration has no tensor-core path in precision %d (%s)", precision,
                precision == KWS_BF16 ? why : "only bf16 is built for the CNN family");
      return KWS_ERR_UNSUPPORTED;
    } else {
      st = cnn_forward_f32(m, feat, B, T, F, logits, workspace, workspace_bytes, as_stream(stream));
    }
  }
  m->prof.finish(as_stream(stream));
  m->last_launches = g_launches;
  return st;
}

extern "C" size_t kws_model_wave_workspace_bytes(const kws_model_t* m, const kws_frontend_t* fe, int64_t B,
                                                 int n_samples, int precision) {
  if (!m || !fe || B < 0) return 0;
  const int T = kws_frontend_n_frames(fe, n_samples);
  const int F = kws_frontend_n_mels(fe);
  if (T < 1 || F < 1) return 0;
  const size_t model_ws = kws_model_workspace_bytes(m, B, T, F, precision);
  if (model_ws == 0) return 0;
  return model_ws + round_up<size_t>((size_t)B * T * F * sizeof(float), 256);
}

template <typename SMP>
static int model_forward_wave_any(const char* who, kws_model_t* m, const kws_frontend_t* fe, const SMP* wav, int64_t B,
                                  int n_samples, float* logits, int precision, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  KWS_REQUIRE(m != nullptr && fe != nullptr, "%s: null handle", who);
  KWS_REQUIRE(B >= 0, "%s: negative batch", who);
  if (B == 0) return KWS_OK;
  const int T = kws_frontend_n_frames(fe, n_samples);
  const int F = kws_frontend_n_mels(fe);
  const size_t need = kws_model_wave_workspace_bytes(m, fe, B, n_samples, precision);
  if (need == 0 || workspace == nullptr || workspace_bytes < need) {
    set_error("%s needs %zu bytes of workspace, got %zu", who, need, workspace_bytes);
    return KWS_ERR_WORKSPACE;
  }
  // the model's scratch comes FIRST: its address (which the whole-network kernels' cached tensor maps are keyed on)
  // then does not move when the batch size, and with it the size of the feature buffer, changes
  const size_t feat_bytes = round_up<size_t>((size_t)B * T * F * sizeof(float), 256);
  const size_t model_bytes = need - feat_bytes;
  float* feat = reinterpret_cast<float*>(static_cast<char*>(workspace) + model_bytes);
  if constexpr (sizeof(SMP) == 4) KWS_TRY(kws_mfcc_forward(fe, wav, B, n_samples, feat, stream));
  else KWS_TRY(kws_mfcc_forward_pcm16(fe, wav, B, n_samples, feat, stream));
  int st = kws_model_forward(m, feat, B, T, F, logits, precision, workspace, model_bytes, stream);
  m->last_launches += 1;
  return st;
}

extern "C" int kws_model_forward_wave(kws_model_t* m, const kws_frontend_t* fe, const float* wav, int64_t B,
                                      int n_samples, float* logits, int precision, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  return model_forward_wave_any<float>("kws_model_forward_wave", m, fe, wav, B, n_samples, logits, precision, workspace,
                                       workspace_bytes, stream);
}

extern "C" int kws_model_forward_wave_pcm16(kws_model_t* m, const kws_frontend_t* fe, const int16_t* wav, int64_t B,
                                            int n_samples, float* logits, int precision, void* workspace,
                                            size_t workspace_bytes, void* stream) {
  return model_forward_wave_any<int16_t>("kws_model_forward_wave_pcm16", m, fe, wav, B, n_samples, logits, precision,
                                         workspace, workspace_bytes, stream);
}

extern "C" int64_t kws_model_last_launches(const kws_model_t* m) { return m ? m->last_launches : 0; }

extern "C" const char* kws_model_kernel_path(const kws_model_t* m, int T, int F, int precision) {
  if (m == nullptr) return "unsupported";
  if (precision != KWS_BF16 && precision != KWS_BF16X3) return "fp32 CUDA-core kernels";
  if (m->kind == KIND_CNN)
    return precision == KWS_BF16 && tc_cnn_supported(m->tcc, nullptr) ? "cnn_tc_fused_kernel" : "unsupported";
  return m->tc != nullptr ? tc_resnet_kernel_path(m->tc, T, F, precision == KWS_BF16X3) : "unsupported";
}

extern "C" int kws_model_set_profile(kws_model_t* m, int enabled) {
  KWS_REQUIRE(m != nullptr, "kws_model_set_profile: model is null");
  m->prof.enabled = enabled != 0;
  m->prof.reset();
  return KWS_OK;
}

extern "C" int kws_model_profile_read(kws_model_t* m, double* conv_ms, int64_t* conv_launches, double* other_ms,
                                      int64_t* other_launches) {
  KWS_REQUIRE(m != nullptr, "kws_model_profile_read: model is null");
  if (conv_ms) *conv_ms = m->prof.ms[0];
  if (conv_launches) *conv_launches = m->prof.n[0];
  if (other_ms) *other_ms = m->prof.ms[1];
  if (other_launches) *other_launches = m->prof.n[1];
  m->prof.reset();
  return KWS_OK;
}

extern "C" int kws_model_set_chunk(kws_model_t* m, int precision, int chunk) {
  KWS_REQUIRE(m != nullptr, "kws_model_set_chunk: model is null");
  KWS_REQUIRE(precision == KWS_FP32 || precision == KWS_BF16 || precision == KWS_BF16X3,
              "kws_model_set_chunk: unknown precision");
  KWS_REQUIRE(chunk >= 0 && chunk <= 65535, "kws_model_set_chunk: chunk must be in [0, 65535]");
  m->chunk[precision] = chunk;
  return KWS_OK;
}
