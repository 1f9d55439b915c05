/*
 * wetts_b200 -- C ABI of the B200-native VITS inference engine.
 *
 * This is the drop-in boundary (SURVEY.md §8b level B2).  It replaces what the
 * reference reaches through ONNXRuntime / PyTorch for the acoustic model:
 *   - runtime/core/model/vits_model.h:30-66   VitsModel::{ForwardEncoder,ForwardDecoder,Forward}
 *   - runtime/core/model/onnx_model.cc:89-94  OnnxModel::Run (session boundary)
 *   - wetts/vits/model/models.py:228-280      SynthesizerTrn.infer  (and the sub-module
 *     forwards it calls: encoders.py:47, duration_predictors.py:206/297, flows.py:442,
 *     decoders.py:63)
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; wetts_last_error()
 *     returns a thread-local message for the last failing call on this thread;
 *   - all tensor pointers are DEVICE pointers into caller-owned allocations
 *     (fp32 unless stated; ids / lengths / speaker ids are int64 as in the ONNX
 *     contract, wetts/vits/export_onnx.py:160-189), except wetts_vits_set_tensor
 *     which accepts host or device memory;
 *   - tensors use the reference layout [B, C, T] (channels-first, time contiguous);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it
 *     unless documented otherwise;
 *   - no hidden allocation after wetts_vits_finalize(): scratch comes from a
 *     caller-provided workspace sized by the matching *_workspace_bytes() query;
 *   - a finalized handle holds no per-call state: concurrent calls on different
 *     streams (and host threads) with different workspaces are legal; every
 *     scratch value of a call, including the device scalar behind the one host
 *     sync of the path, lives in that call's workspace.  Options must not be
 *     changed while calls on the same handle are in flight;
 *   - output audio stays float in [-1, 1]; x32767 / int16 belongs to the caller
 *     (vits_model.cc:84-86, wetts/cli/model.py:60).
 * There is no CPU fallback anywhere behind this interface.
 */
#ifndef WETTS_B200_H_
#define WETTS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WETTS_MAX_UPSAMPLES 6
#define WETTS_MAX_RESBLOCK_KERNELS 4
#define WETTS_MAX_DILATIONS 4

typedef struct wetts_vits_s* wetts_vits_t;

/* Mirrors the constructor arguments of SynthesizerTrn (models.py:19-51) that
 * shape the inference path. */
typedef struct wetts_vits_config {
  int32_t n_vocab;
  int32_t n_speakers;          /* 0: no speaker embedding (g == NULL everywhere) */
  int32_t inter_channels;      /* 192 */
  int32_t hidden_channels;     /* 192 */
  int32_t filter_channels;     /* 768 */
  int32_t n_heads;             /* 2 */
  int32_t n_layers;            /* 6 */
  int32_t kernel_size;         /* FFN kernel, 3 */
  int32_t gin_channels;        /* 256 */
  int32_t use_sdp;             /* 1: StochasticDurationPredictor, 0: DurationPredictor */
  int32_t resblock_type;       /* 1 or 2 */
  int32_t n_resblock_kernels;
  int32_t resblock_kernel_sizes[WETTS_MAX_RESBLOCK_KERNELS];
  int32_t resblock_n_dilations[WETTS_MAX_RESBLOCK_KERNELS];
  int32_t resblock_dilations[WETTS_MAX_RESBLOCK_KERNELS][WETTS_MAX_DILATIONS];
  int32_t n_upsamples;
  int32_t upsample_rates[WETTS_MAX_UPSAMPLES];
  int32_t upsample_kernel_sizes[WETTS_MAX_UPSAMPLES];
  int32_t upsample_initial_channel;
  /* SURVEY.md 8f rank 4 (the vits2_vocos_v1 recipe); all zero = the v1/v2/v3 recipes */
  int32_t vocoder_type;        /* 0: HiFi-GAN Generator (decoders.py:15), 1: VocosGenerator (decoders.py:250) */
  int32_t vocos_channels;      /* 512 */
  int32_t vocos_h_channels;    /* 1536 */
  int32_t vocos_out_channels;  /* 1026 = n_fft + 2 */
  int32_t vocos_num_layers;    /* 8 */
  int32_t vocos_n_fft;         /* 1024 (= win_length; center = True) */
  int32_t vocos_hop_length;    /* 256 */
  int32_t flow_type;           /* 0: ResidualCouplingLayer (flows.py:459), 1: VITS2 'pre_conv' transformer flow (flows.py:89) */
} wetts_vits_config;

const char* wetts_last_error(void);
const char* wetts_version(void);

/* Process-wide options.  "tensor_cores": 1 (default) routes eligible convolutions through the
 * tcgen05 3xTF32 implicit-GEMM kernel (fp32-accurate), 0 forces the fp32 SIMT kernels.
 * "fused_resblock": 1 (default) runs each eligible HiFi-GAN stage (ResBlock2, 32 or 64 channels)
 * as ONE fused MRF kernel (both convs of every resblock + the mean on chip), 0 keeps one launch
 * per convolution.  Only effective with tensor_cores = 1.
 * "mrf_item_rows": output samples per work item of the fused 32-channel ResBlock2 stage kernel:
 * 0 (default) = chosen per launch (384 when the launch has >= 4 items per CTA slot, else 128),
 * 128 / 256 / 384 = forced; every size computes bit-identical results.  Read-only
 * "mrf_item_rows_last": the size the last such launch used. */
int wetts_set_option(const char* name, int value);
int wetts_get_option(const char* name, int* value);

/* ---- lifetime ---------------------------------------------------------- */
int wetts_vits_create(const wetts_vits_config* cfg, int device, wetts_vits_t* out);
/* Register one checkpoint tensor under its reference state-dict key
 * (e.g. "dec.ups.0.weight_v"; key patterns: SURVEY.md App. B).  fp32, contiguous,
 * host or device memory; the engine keeps its own device copy.  Accepts both
 * weight-normed pairs (`weight_g`/`weight_v`, what inference.py loads) and folded
 * `weight` (what export_onnx.py:79-81 produces).  `enc_q.*` keys (the posterior encoder) are
 * kept for voice conversion; infer never reads them. */
int wetts_vits_set_tensor(wetts_vits_t h, const char* name, const void* data, const int64_t* dims, int ndim);
/* Fold weight-norm (per out-channel for Conv1d, per IN-channel for ConvTranspose1d,
 * decoders.py:41-48) and re-lay weights for the kernels.  Fails listing the first
 * missing key.  The posterior encoder (enc_q.*) is packed only when every one of its
 * keys is present; a checkpoint without it, or with an incomplete one, finalizes all
 * the same and the voice-conversion calls below then fail naming the first missing
 * key.  Synchronous. */
int wetts_vits_finalize(wetts_vits_t h);
void wetts_vits_destroy(wetts_vits_t h);
/* Per-handle options; they take precedence over the process-wide ones above.  "tensor_cores" and
 * "fused_resblock" as above (value -1: follow the process-wide option again); "length_aware": 1 lets the
 * generator skip tiles that lie wholly beyond an utterance's own length plus the receptive field when
 * y_lengths is given (valid samples unchanged, the padded tail is left unspecified; default 0 = compute the
 * full padded tail exactly as the reference does). */
int wetts_vits_set_option(wetts_vits_t h, const char* name, int value);
int wetts_vits_get_option(wetts_vits_t h, const char* name, int* value);
/* product of upsample_rates (256 for every reference config; vits_model.h:27) */
int wetts_vits_upsample_factor(wetts_vits_t h);

/* ---- block-level entry points (sub-module forwards, SURVEY §8b B0) ------ */

/* g = emb_g(sid)  (models.py:238-241).  sid int64[B] -> g f32[B, gin]. */
int wetts_speaker_embedding(wetts_vits_t h, const int64_t* sid, int B, float* g, void* stream);

/* TextEncoder.forward (encoders.py:47-57): ids int64[B,Tx], lengths int64[B]
 * -> h, m, logs f32[B,192,Tx] (h is the pre-projection hidden state). */
size_t wetts_text_encoder_workspace_bytes(wetts_vits_t h, int B, int Tx);
int wetts_text_encoder_forward(wetts_vits_t h, const int64_t* ids, const int64_t* lengths, int B, int Tx,
                               float* h_out, float* m_out, float* logs_out,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Duration predictor -> logw f32[B,1,Tx].  use_sdp=0: DurationPredictor.forward
 * (duration_predictors.py:297-311), noise_w ignored.  use_sdp=1:
 * StochasticDurationPredictor.forward(reverse=True) (:213-219,254-263) with
 * noise_w f32[B,2,Tx] explicit N(0,1) draws (required) scaled by noise_scale_w.
 * g f32[B,gin] or NULL. */
size_t wetts_duration_workspace_bytes(wetts_vits_t h, int B, int Tx);
int wetts_duration_forward(wetts_vits_t h, const float* h_in, const int64_t* lengths, const float* g,
                           const float* noise_w, float noise_scale_w, int B, int Tx, float* logw,
                           void* workspace, size_t workspace_bytes, void* stream);

/* w_ceil = ceil(exp(logw)*mask*length_scale), y_lengths = max(sum, 1), inclusive
 * cumsum (models.py:254-256, commons.py:120-125).  If `durations` (f32[B,Tx]) is
 * non-NULL it replaces ceil(...) (teacher forcing for staged parity).
 * Outputs: w_ceil f32[B,Tx], cum int32[B,Tx], y_lengths int64[B]. */
int wetts_length_regulate(wetts_vits_t h, const float* logw, const int64_t* x_lengths, const float* durations,
                          float length_scale, int B, int Tx, float* w_ceil, int32_t* cum, int64_t* y_lengths,
                          void* stream);

/* Expand the prior along the monotonic path and sample (models.py:257-267):
 * m_p/logs_p[b,:,y] = m/logs[b,:,t(y)], z_p = m_p + noise_z*exp(logs_p)*noise_scale.
 * noise_z f32 with batch stride noise_bs (>= 192*Ty) and row stride noise_rs (>= Ty).
 * attn (f32[B,1,Ty,Tx] one-hot, may be NULL), m_p_out/logs_p_out may be NULL. */
int wetts_expand_prior(wetts_vits_t h, const float* m, const float* logs, const int32_t* cum,
                       const int64_t* x_lengths, const int64_t* y_lengths, const float* noise_z,
                       int64_t noise_bs, int64_t noise_rs, float noise_scale, int B, int Tx, int Ty,
                       float* m_p_out, float* logs_p_out, float* z_p_out, float* attn, float* y_mask, void* stream);

/* ResidualCouplingTransformersBlock.forward(reverse=True) (flows.py:442-449).
 * z f32[B,192,Ty] is transformed IN PLACE (z_p -> z).  y_lengths int64[B]. */
size_t wetts_flow_workspace_bytes(wetts_vits_t h, int B, int Ty);
int wetts_flow_reverse(wetts_vits_t h, float* z, const int64_t* y_lengths, const float* g, int B, int Ty,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ResidualCouplingTransformersBlock.forward(reverse=False): the four coupling layers in
 * forward order, x1 = m + x1 * mask (flows.py:494-513).  z f32[B,192,Ty] IN PLACE (z -> z_p);
 * workspace sized by wetts_flow_workspace_bytes. */
int wetts_flow_forward(wetts_vits_t h, float* z, const int64_t* y_lengths, const float* g, int B, int Ty,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Generator.forward (decoders.py:63-82): z f32[B,192,T] (+ g f32[B,gin] or NULL)
 * -> audio f32[B,1,T*U].  If y_lengths != NULL the input is multiplied by the frame
 * mask first, as infer() does (models.py:271). */
size_t wetts_generator_workspace_bytes(wetts_vits_t h, int B, int T);
int wetts_generator_forward(wetts_vits_t h, const float* z, const int64_t* y_lengths, const float* g, int B, int T,
                            float* audio, void* workspace, size_t workspace_bytes, void* stream);
/* Same on a strided view of z: element (b, c, t) at z[b*z_batch_stride + c*z_channel_stride + t], t < T.  This is
 * how infer(max_len=...) vocodes (z * y_mask)[:, :, :max_len] without a copy (models.py:270-271). */
int wetts_generator_forward_view(wetts_vits_t h, const float* z, int64_t z_batch_stride, int64_t z_channel_stride,
                                 const int64_t* y_lengths, const float* g, int B, int T, float* audio,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ---- whole path, split at the one unavoidable host sync (Ty = max y_lengths) */

/* Stage 1: ids -> durations.  Runs speaker embedding, text encoder, duration
 * predictor and length regulation.  Keeps h/m/logs/cum in the workspace for
 * stage 2 (same workspace must be passed).  Outputs y_lengths int64[B] (device);
 * *max_frames_host receives max_b y_lengths (this call synchronises `stream`).
 * scales = {noise_scale, length_scale, noise_scale_w} (export contract row 0,
 * models.py:333-344).  noise_w: see wetts_duration_forward.  durations: optional
 * teacher forcing f32[B,Tx]. */
size_t wetts_vits_infer_workspace_bytes(wetts_vits_t h, int B, int Tx, int max_frames);
int wetts_vits_infer_durations(wetts_vits_t h, const int64_t* ids, const int64_t* x_lengths, const int64_t* sid,
                               const float* scales3, const float* noise_w, const float* durations, int B, int Tx,
                               int64_t* y_lengths, float* logw_out, float* w_ceil_out, int* max_frames_host,
                               void* workspace, size_t workspace_bytes, void* stream);
/* Stage 2: expand prior, sample, invert the flow, vocode.  Ty must be >= the
 * value stage 1 returned (normally equal).  gen_frames: number of leading frames
 * the vocoder runs on -- infer()'s `max_len` (models.py:270-271); <= 0 or > Ty means Ty.
 * Outputs (any may be NULL except audio): audio f32[B,1,gen_frames*U],
 * attn f32[B,1,Ty,Tx], y_mask f32[B,1,Ty], z, z_p, m_p, logs_p f32[B,192,Ty]. */
int wetts_vits_infer_synthesize(wetts_vits_t h, const int64_t* x_lengths, const int64_t* y_lengths,
                                const float* scales3, const float* noise_z, int64_t noise_bs, int64_t noise_rs,
                                int B, int Tx, int Ty, int gen_frames, float* audio, float* attn, float* y_mask, float* z,
                                float* z_p, float* m_p, float* logs_p, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ---- voice conversion (SynthesizerTrn.voice_conversion, models.py:369-376) ----------------
 * Need a checkpoint with the complete posterior encoder (enc_q.*). */

/* PosteriorEncoder.forward (encoders.py:91-99): y f32[B,S,T] features (S = the in-channels of
 * enc_q.pre: filter_length/2+1 linear bins, or n_mel_channels for a VITS2 mel posterior),
 * y_lengths int64[B], g f32[B,gin] or NULL, noise f32[B,192,T] explicit N(0,1) draws (required,
 * what the reference draws with randn_like) -> z f32[B,192,T]; m, logs f32[B,192,T] may be NULL. */
size_t wetts_posterior_workspace_bytes(wetts_vits_t h, int B, int T);
int wetts_posterior_encoder_forward(wetts_vits_t h, const float* y, const int64_t* y_lengths, const float* g,
                                    const float* noise, int B, int T, float* z, float* m, float* logs,
                                    void* workspace, size_t workspace_bytes, void* stream);

/* Linear spectrogram, spectrogram_torch(center=False) (mel_processing.py:42-93) applied to each
 * utterance on its own: reflection padding by p = (n_fft - hop)/2 at the utterance's own length,
 * periodic Hann window, onesided real DFT, sqrt(re^2 + im^2 + 1e-6).  n_fft = win = 2 (S - 1)
 * (S - 1 a power of two), hop = wetts_vits_upsample_factor.  audio f32[B,L], audio_lengths
 * int64[B] (each in [p+1, L]) -> spec f32[B,S,F] with F = 1 + (L + 2p - n_fft)/hop, frames at or
 * beyond an utterance's own count F_b = 1 + (L_b + 2p - n_fft)/hop exactly 0; spec_lengths
 * int64[B] = F_b (may be NULL).  Checks the lengths on the host: synchronises `stream`.
 * The workspace query returns 0 when L is too short or the model has no spectrogram. */
size_t wetts_spectrogram_workspace_bytes(wetts_vits_t h, int B, int64_t L);
int wetts_spectrogram(wetts_vits_t h, const float* audio, const int64_t* audio_lengths, int B, int64_t L, float* spec,
                      int64_t* spec_lengths, void* workspace, size_t workspace_bytes, void* stream);

/* The whole conversion: posterior encoder and forward flow with g = emb_g(sid_src), inverse flow
 * and generator with g = emb_g(sid_tgt) on z_hat * y_mask over all T frames.  y / y_lengths /
 * noise as for wetts_posterior_encoder_forward; sid_src, sid_tgt int64[B].  Outputs (any may be
 * NULL except audio): audio f32[B,1,T*U], y_mask f32[B,1,T], z, z_p, z_hat f32[B,192,T].
 * Fails for a single-speaker model (n_speakers == 0).  Honours "length_aware". */
size_t wetts_vits_voice_conversion_workspace_bytes(wetts_vits_t h, int B, int T);
int wetts_vits_voice_conversion(wetts_vits_t h, const float* y, const int64_t* y_lengths, const int64_t* sid_src,
                                const int64_t* sid_tgt, const float* noise, int B, int T, float* audio, float* y_mask,
                                float* z, float* z_p, float* z_hat, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ---- L2 session contract (export_onnx.py:93-148; VitsModel::ForwardDecoder) --
 * decoder(z f32[B,L,192] time-major, sid int64[B]) -> audio f32[B,1,L*U] */
size_t wetts_vits_decoder_workspace_bytes(wetts_vits_t h, int B, int L);
int wetts_vits_forward_decoder(wetts_vits_t h, const float* z_blc, const int64_t* sid, int B, int L, float* audio,
                               void* workspace, size_t workspace_bytes, void* stream);

/* ---- output stage of the callers (SURVEY.md 8f rank 3) ---------------------------------
 * audio f32[B,L] in [-1,1] -> int16[B,L] on the device.  mode 0: x32767 (cli/model.py:60, vits_model.cc:84-86);
 * mode 1: per utterance 32767 / max(0.01, max|a|) * 0.6 (inference.py:101-105), the peak searched over the first
 * lengths[b] samples when `lengths` (int64[B]) is given; mode 2: one such gain for the whole batch
 * (runtime/gpu_triton model.py:150-151).  Values are clipped to +-32767 and truncated toward zero like
 * numpy's astype(int16).  peak_scratch: device float[B] (modes 1, 2; may be NULL for mode 0). */
int wetts_audio_to_int16(const float* audio, const int64_t* lengths, int B, int64_t L, int mode, float* peak_scratch,
                         int16_t* out, void* stream);

/* Watchdog.  The tensor-pipe kernels synchronise through mbarriers; a wait that does not complete within 2^24 polls
 * (a pipeline bug, never normal operation) records the reason in a host-visible word and traps, so a defect shows up
 * as a failed launch within a fraction of a second instead of a hung GPU.  As after any device-side trap the CUDA
 * context is lost; every later call on it fails.  This call (optionally after synchronising `stream`) returns non-zero
 * with "pipeline watchdog fired" in wetts_last_error() when that was the cause, so a serving process can tell a
 * kernel defect from other launch failures before it restarts. */
int wetts_vits_check_fault(wetts_vits_t h, void* stream, int synchronize);

/* Counters for benchmarks: number of kernels this library has launched on behalf
 * of the handle since creation (monotonic). */
uint64_t wetts_vits_launch_count(wetts_vits_t h);

#ifdef __cplusplus
}
#endif
#endif /* WETTS_B200_H_ */
