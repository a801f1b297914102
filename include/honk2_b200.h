/* honk2_b200 -- C ABI of the B200-native keyword-spotting inference path.
 *
 * This is the drop-in boundary for honk2's batched inference hot path (SURVEY.md section 8b).
 * The reference is pure Python and has no FFI of its own; each entry point below names the
 * reference interface it replaces.  All pointers are DEVICE pointers unless said otherwise,
 * all tensors are dense row-major, `stream` is a cudaStream_t passed as void*.
 * Every function returns 0 (KWS_OK) or a KWS_ERR_* code; the message for the calling thread's
 * last failure is kws_last_error().  No exceptions cross this boundary and no hot call
 * allocates: scratch memory is supplied by the caller (kws_model_workspace_bytes).
 * Handles are not thread-safe; calls on different handles are.  There is NO CPU fallback:
 * creating a handle on a device that is not compute capability 10.x fails.
 */
#ifndef HONK2_B200_H
#define HONK2_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KWS_ABI_VERSION 2

enum {
  KWS_OK = 0,
  KWS_ERR_INVALID = 1,      /* bad argument / unsupported shape */
  KWS_ERR_CUDA = 2,         /* a CUDA runtime / driver call failed */
  KWS_ERR_UNSUPPORTED = 3,  /* not an sm_100 device, or feature not built */
  KWS_ERR_WORKSPACE = 4     /* workspace too small */
};

enum {
  KWS_FP32 = 0,  /* CUDA-core FFMA path, fp32 storage and accumulate (parity mode) */
  KWS_BF16 = 1,  /* tcgen05 tensor-core path: bf16 operands, fp32 TMEM accumulate */
  KWS_BF16X3 = 2 /* tcgen05 tensor-core path with split-bf16 operands: every activation and weight is a bf16 pair
                    hi + lo (16 mantissa bits), every product three MMAs (hi*hi + hi*lo + lo*hi), fp32 accumulate:
                    meets the fp32 tolerance (1e-3 of the logit scale, identical argmax) at tensor-core speed */
};

typedef struct kws_frontend kws_frontend_t;
typedef struct kws_model kws_model_t;

int kws_abi_version(void);
const char* kws_last_error(void);
/* Fills compute capability and SM count of the current device; KWS_ERR_UNSUPPORTED unless 10.x */
int kws_device_info(int* cc_major, int* cc_minor, int* n_sms);

/* ---- front-end: replaces AudioProcessor (utils/audio_processor.py:8-30) -------------------
 * kws_frontend_create   <- AudioProcessor.__init__ (:8-16); n_fft must be 480 and hop 160
 *                          (the only geometry honk2 constructs, audio_data_loader.py:14).
 * kws_frontend_n_frames <- T = 1 + n_samples / hop (librosa center=True framing).
 * kws_mfcc_forward      <- compute_mfccs (:18-30) for a whole batch, i.e. the per-sample loop
 *                          of AudioDataLoader.collate_fn (data_loader/audio_data_loader.py:26-29):
 *                          wav [B, n_samples] f32 -> feat [B, T, n_mels] f32 = 2*ln(mel power),
 *                          exact zeros stay 0.
 */
int kws_frontend_create(int sr, int n_mels, float f_min, float f_max, int n_fft, int hop,
                        kws_frontend_t** out);
void kws_frontend_destroy(kws_frontend_t* fe);
int kws_frontend_n_frames(const kws_frontend_t* fe, int n_samples);
int kws_frontend_n_mels(const kws_frontend_t* fe);
int kws_mfcc_forward(const kws_frontend_t* fe, const float* wav, int64_t B, int n_samples,
                     float* feat, void* stream);
/* The same front-end on the 16-bit PCM samples of the wav files the reference's datasets read
 * (dataset/gsc_dataset.py:169, dataset/hey_snips_dataset.py:74 -> librosa.core.load, which returns float32(s / 32768) for a 16-bit file): wav
 * [B, n_samples] int16.  The conversion happens while the samples are staged, so feat is bit-identical to
 * kws_mfcc_forward on the converted floats; host->device and HBM traffic of the waveforms halve. */
int kws_mfcc_forward_pcm16(const kws_frontend_t* fe, const int16_t* wav, int64_t B, int n_samples,
                           float* feat, void* stream);
/* Streaming-window front-end (SURVEY 8f-1): replaces StreamingDataset.__getitem__'s window slicing
 * (dataset/dataset_utils.py:28-31,72 -- window k = stream[k*shift : k*shift + window]) followed by the per-window
 * compute_mfccs of collate_fn (audio_data_loader.py:26-29).  wav points at the first sample of the first window and
 * must hold (n_windows-1)*shift + window samples; feat [n_windows, T, n_mels] is bit-identical to kws_mfcc_forward on
 * the materialised windows.  When shift is a multiple of the hop (gsc_dev_config.json:62-63: 1000 ms / 10 ms), every
 * frame that does not touch a window's reflect padding (t = 2 .. T-3) is computed ONCE per stream position and copied;
 * only 4 frames per window are computed per window.  scratch: kws_mfcc_stream_scratch_bytes (0 = none needed). */
size_t kws_mfcc_stream_scratch_bytes(const kws_frontend_t* fe, int64_t n_windows, int window, int shift);
int kws_mfcc_stream_forward(const kws_frontend_t* fe, const float* wav, int64_t n_windows, int window, int shift,
                            float* feat, void* scratch, size_t scratch_bytes, void* stream);
/* The same on an int16 PCM stream (see kws_mfcc_forward_pcm16); same scratch size, bit-identical features. */
int kws_mfcc_stream_forward_pcm16(const kws_frontend_t* fe, const int16_t* wav, int64_t n_windows, int window, int shift,
                                  float* feat, void* scratch, size_t scratch_bytes, void* stream);

/* Live streams: the streaming-window front-end above for S streams whose audio arrives a few milliseconds at a time.
 * There is no reference interface: this replaces the caller's own per-stream ring buffer around compute_mfccs.
 * A state holds, per stream, a device-resident sample ring, a ring of frame-table rows and a sample counter c_s
 * (samples pushed since the stream's last reset).  Window k of stream s is samples [k*shift, k*shift + window) of it,
 * the windows of StreamingDataset.__getitem__ (dataset/dataset_utils.py:72).
 *   kws_live_state_bytes  device bytes kws_live_create allocates (0 on invalid arguments).
 *   kws_live_create       refuses (KWS_ERR_INVALID) a shift that is not a multiple of the 160-sample hop, windows of
 *                         fewer than 5 frames, a max_push that is not a multiple of the shift, and n_streams < 1.  The
 *                         front-end must outlive the state.
 *   kws_live_push         chunk [S, n] f32 holds n new samples of every stream, n a multiple of the shift in
 *                         [shift, max_push].  It completes K = n / shift window indices per stream: slot j of stream s
 *                         is window k = floor((c_s - window) / shift) + 1 + j, c_s counted before the push; the last
 *                         slot is the newest complete window.  feat [S, K, T, n_mels] receives their features,
 *                         bit-identical to kws_mfcc_forward on the materialised windows; slots with k < 0 (the warm-up
 *                         of a fresh stream) are all zeros.  Only the n / 160 new frame-table rows per stream and the
 *                         four reflect-padded edge frames per window are computed.
 *                         Precondition: every c_s is a multiple of 160 (the hop), which holds unless a ragged push
 *                         left it otherwise.  The counters live on the device, so the library cannot check it; a
 *                         caller that mixes the two pushes checks its own copy (LiveStreams.push raises ValueError).
 *   kws_live_push_pcm16   the same on int16 PCM (see kws_mfcc_forward_pcm16): bit-identical to a float push of s/32768.
 *   kws_live_reset        stream_ids: DEVICE int64[count]; those streams restart at sample 0 (ids outside [0, S) are
 *                         ignored).  Other streams are unaffected.
 * Push and reset allocate nothing and do not synchronise the host; counters live on the device, so a caller that
 * needs the validity of each slot keeps its own copy of c_s (honk2_b200.LiveStreams does).
 *
 * Ragged pushes: stream s brings its own number n_s of new samples, any n_s in [0, max_push] (not necessarily a multiple
 * of the shift or of 160), and only the windows the push completes come back, compacted.  With c_s' = c_s + n_s, the
 * push completes windows k with max(0, floor((c_s - window)/shift) + 1) <= k <= floor((c_s' - window)/shift).
 *   kws_live_ragged_workspace_bytes  device scratch a ragged push needs (0 on a null state).
 *   kws_live_push_ragged  samples: all streams' new samples back to back in stream order, sum(n_s) floats.
 *                         lengths: HOST int32[S], read during the call.  Row i of feat [M, T, n_mels] holds window
 *                         win_index[i] of stream win_stream[i], rows ordered by stream, then by window; M goes to
 *                         *n_windows.  The features are bit-identical to kws_mfcc_forward on the materialised windows,
 *                         and across any sequence of pushes each stream emits windows 0, 1, 2, ... exactly once.  feat,
 *                         win_stream and win_index hold `capacity` rows; win_stream, win_index and n_windows may be null
 *                         (a caller that keeps its own copy of c_s can compute them: LiveStreams does).
 *                         Returns KWS_ERR_INVALID, launching nothing, unless every n_s is in [0, max_push], capacity >=
 *                         sum(ceil(n_s / shift)) (which bounds M) and the workspace is large enough.
 *   kws_live_push_ragged_pcm16  the same on int16 PCM: bit-identical to a float ragged push of s/32768.
 * A ragged push copies the per-stream offsets and lengths to the device through a pinned host buffer of the state,
 * allocated by the state's first ragged push; before refilling it, a push waits for the previous ragged push's copy
 * (not for its kernels).  Nothing else allocates and the host does not wait for the device: the device derives each
 * stream's new rows and windows from its counter and scans them (the totals are never read back).  The two pushes
 * and reset may be mixed on one state, with the precondition of kws_live_push. */
typedef struct kws_live kws_live_t;
size_t kws_live_state_bytes(const kws_frontend_t* fe, int n_streams, int window, int shift, int max_push);
int kws_live_create(const kws_frontend_t* fe, int n_streams, int window, int shift, int max_push, kws_live_t** out);
void kws_live_destroy(kws_live_t* live);
int kws_live_reset(kws_live_t* live, const int64_t* stream_ids, int64_t count, void* stream);
int kws_live_push(kws_live_t* live, const float* chunk, int n, float* feat, void* stream);
int kws_live_push_pcm16(kws_live_t* live, const int16_t* chunk, int n, float* feat, void* stream);
size_t kws_live_ragged_workspace_bytes(const kws_live_t* live);
int kws_live_push_ragged(kws_live_t* live, const float* samples, const int32_t* lengths, float* feat,
                         int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                         void* workspace, size_t ws_bytes, void* stream);
int kws_live_push_ragged_pcm16(kws_live_t* live, const int16_t* samples, const int32_t* lengths, float* feat,
                               int64_t* win_stream, int64_t* win_index, int64_t capacity, int64_t* n_windows,
                               void* workspace, size_t ws_bytes, void* stream);

/* ---- models: replace model.ResNet / model.CNN ---------------------------------------------
 * kws_resnet_create <- ResNet.__init__ (model/resnet.py:11-36); pool_h = pool_w = 0 when the
 *                      config has no "pool" key.
 * kws_cnn_create    <- CNN.__init__ (model/cnn.py:12-77); *_out == 0 means "layer absent".
 * *_set_weights     <- nn.Module.load_state_dict (utils/workspace.py:61): fp32 device tensors
 *                      in PyTorch layout (state_dict keys in the comments); the library repacks
 *                      them (transposes, BN folding, bf16 copies) into its own buffers.
 * kws_model_forward <- ResNet.forward (resnet.py:38-60) / CNN.forward (cnn.py:79-107) in eval
 *                      mode: feat [B, T, F] f32 -> logits [B, n_labels] f32 (raw, no softmax).
 * kws_model_forward_wave <- collate_fn + forward fused: wav [B, n_samples] -> logits.
 */
typedef struct {
  int n_layers;      /* config["n_layers"] */
  int n_maps;        /* config["n_feature_maps"] */
  int use_dilation;  /* config["use_dilation"]: dilation = padding = 2**((i-1)/3) */
  int pool_h, pool_w;/* config["pool"], 0,0 if absent (AvgPool2d, stride = kernel, floor) */
  int n_labels;      /* config["n_labels"] */
} kws_resnet_config;

typedef struct {
  const float* conv0_w;        /* layers.conv_0.weight            [C,1,3,3]  */
  const float* const* conv_w;  /* layers.conv_{i}.weight, i=1..n  [C,C,3,3] (HOST array of device ptrs) */
  const float* const* bn_mean; /* layers.bn_{i}.running_mean      [C] */
  const float* const* bn_var;  /* layers.bn_{i}.running_var       [C] */
  const float* out_w;          /* layers.output.weight            [n_labels,C] */
  const float* out_b;          /* layers.output.bias              [n_labels] */
} kws_resnet_weights;

typedef struct {
  int time, freq;                                   /* config["time"], config["frequency"] */
  int conv0_out, conv0_kh, conv0_kw, conv0_sh, conv0_sw;
  int pool0_kh, pool0_kw;                           /* MaxPool2d, stride = kernel, floor */
  int conv1_out, conv1_kh, conv1_kw, conv1_sh, conv1_sw;   /* conv1_out == 0: absent */
  int pool1_kh, pool1_kw;
  int lin0_out, dnn0_out, dnn1_out;                 /* 0: absent */
  int n_labels;
} kws_cnn_config;

typedef struct {
  const float *conv0_w, *conv0_b;   /* layers.conv_0.{weight,bias} [C0,1,kh,kw], [C0] */
  const float *conv1_w, *conv1_b;   /* layers.conv_1.*             [C1,C0,kh,kw], [C1] */
  const float *lin0_w, *lin0_b;     /* layers.lin_0.*  [out,in] */
  const float *dnn0_w, *dnn0_b;     /* layers.dnn_0.* */
  const float *dnn1_w, *dnn1_b;     /* layers.dnn_1.* */
  const float *lin1_w, *lin1_b;     /* layers.lin_1.*  [n_labels,in] */
} kws_cnn_weights;

int kws_resnet_create(const kws_resnet_config* cfg, kws_model_t** out);
int kws_resnet_set_weights(kws_model_t* m, const kws_resnet_weights* w, void* stream);
int kws_cnn_create(const kws_cnn_config* cfg, kws_model_t** out);
int kws_cnn_set_weights(kws_model_t* m, const kws_cnn_weights* w, void* stream);
void kws_model_destroy(kws_model_t* m);

int kws_model_n_labels(const kws_model_t* m);
/* Bytes of scratch kws_model_forward needs for this call shape (0 on invalid arguments). */
size_t kws_model_workspace_bytes(const kws_model_t* m, int64_t B, int T, int F, int precision);
int kws_model_forward(kws_model_t* m, const float* feat, int64_t B, int T, int F, float* logits,
                      int precision, void* workspace, size_t workspace_bytes, void* stream);
/* Scratch for the fused waveform -> logits call (adds the feature staging buffer). */
size_t kws_model_wave_workspace_bytes(const kws_model_t* m, const kws_frontend_t* fe, int64_t B,
                                      int n_samples, int precision);
int kws_model_forward_wave(kws_model_t* m, const kws_frontend_t* fe, const float* wav, int64_t B,
                           int n_samples, float* logits, int precision, void* workspace,
                           size_t workspace_bytes, void* stream);
/* kws_model_forward_wave on int16 PCM waveforms (see kws_mfcc_forward_pcm16); same workspace. */
int kws_model_forward_wave_pcm16(kws_model_t* m, const kws_frontend_t* fe, const int16_t* wav, int64_t B,
                                 int n_samples, float* logits, int precision, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* Number of kernel launches the last forward on this handle issued (bench "gpu_launches"). */
int64_t kws_model_last_launches(const kws_model_t* m);
/* Name of the kernel family a forward of a [B][T][F] batch runs in the given precision (bench / profile labels):
 * "resnet_tc_sweep_kernel", "resnet_tc_fused_kernel", "fp32 CUDA-core kernels" or "unsupported".  Static string,
 * never freed. */
const char* kws_model_kernel_path(const kws_model_t* m, int T, int F, int precision);
/* Per-launch timing for the bench roofline: while enabled, kws_model_forward brackets every
 * launch with CUDA events and synchronises the stream before returning.
 * kws_model_profile_read returns (and clears) the accumulated milliseconds / launch counts of
 * the dominant kernel's launches and of all other launches.  The dominant kernel is the C->C
 * convolution on the fp32 paths, the whole-network kernel on the ResNet tensor-core paths and the
 * fused conv_0 + conv_1 kernel on the CNN tensor-core path. */
int kws_model_set_profile(kws_model_t* m, int enabled);
int kws_model_profile_read(kws_model_t* m, double* conv_ms, int64_t* conv_launches, double* other_ms,
                           int64_t* other_launches);
/* Tuning knob: utterances per sub-batch (0 = default) of the fp32 paths, of the bf16 CNN path and of the
 * packed-strip mode of the ResNet column-sweep kernel.  The other ResNet tensor-core paths run the whole
 * batch in one launch and ignore it. */
int kws_model_set_chunk(kws_model_t* m, int precision, int chunk);

/* ---- metrics: replaces Acc.accumulate (metric/acc.py:14-24) -------------------------------
 * counts[0] += #(argmax(logits[b,:]) == target[b]), counts[1] += B  (device int64[2];
 * ties resolve to the lowest index like torch.argmax).  pred (nullable) receives argmax. */
int kws_acc_accumulate(const float* logits, const int64_t* target, int64_t B, int n_labels,
                       int64_t* counts, int64_t* pred, void* stream);

/* One pass over a batch of logits for the whole evaluate() bookkeeping (run/test.py:28-33), nothing leaves the device:
 *   counts        (nullable) int64[2]:            += [correct, total]                 (metric/acc.py:14-24)
 *   class_counts  (nullable) int64[2 * n_labels]: [2 t] += 1, [2 t + 1] += correct    (metric/per_class_acc.py:14-45)
 *   loss_sum      (nullable) double[1]:           += sum_b (logsumexp(row_b) - row_b[target_b]), i.e. the SUM form of
 *                                                 nn.CrossEntropyLoss (loss_function.py:7-9); divide by B for its mean
 *   pred          (nullable) int64[B]:            argmax (first maximum, NaN wins, like torch.argmax)
 * Targets outside [0, n_labels) count as misses in `counts` and are skipped by the other two. */
int kws_eval_accumulate(const float* logits, const int64_t* target, int64_t B, int n_labels,
                        int64_t* counts, int64_t* class_counts, double* loss_sum, int64_t* pred, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HONK2_B200_H */
