// Internal kernel interface of libwetts_b200 (sm_100a).  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv_args.h"
#include "fused_mrf16_args.h"
#include "fused_rb_args.h"

namespace wetts {

// ---------------------------------------------------------------- conv1d (argument structs: conv_args.h)
void launch_conv1d(const ConvArgs& a, cudaStream_t s);
// out[b][co] = bias[co] + sum_ci w[ci][co] g[b][ci]   (w: SIMT layout of a 1x1 conv, [Cin][1][CoutPad])
void launch_cond_vector(const float* g, const float* w, const float* bias, float* out, int B, int Cin, int Cout,
                        int CoutPad, cudaStream_t s);
void launch_conv1d_simt(const ConvArgs& a, cudaStream_t s);

// Probes (once) the shared-window offset at which dynamic shared memory starts for kernels without static
// shared memory.  tcgen05 descriptors built from this kernel parameter are uniform by construction.
int dyn_smem_offset(uint32_t* off, cudaStream_t s);
bool tc_conv_plan(int Cin, int Cout, int K, int dil, TcPlan* plan);
size_t tc_conv_smem_bytes(int K, int dil, int N, int KC, int MB, int n_abuf, int n_bbuf);
void launch_pack_conv_tc(const float* src, float* dst, const int* co_map, const int* ci_map, int Cout, int Cin, int K,
                         int src_cin, const TcPlan& pl, cudaStream_t s);
void launch_conv1d_tc(const ConvArgs& a, cudaStream_t s);
// f16-split twin (tc16_conv_kernel.cu); plan->packed_floats counts HALFS for this format
bool tc16_conv_plan(int Cin, int Cout, int K, int dil, TcPlan* plan);
size_t tc16_conv_smem_bytes(int K, int dil, int N, int KC, int MB, int n_abuf, int n_bbuf);
void launch_pack_conv_tc16(const float* src, void* dst, const int* co_map, const int* ci_map, int Cout, int Cin, int K,
                           int src_cin, const TcPlan& pl, cudaStream_t s);
void launch_conv1d_tc16(const ConvArgs& a, cudaStream_t s);
// pipelined variant (tc16p_conv.cu): same weights and plan, dedicated staging / epilogue warps; false = not taken
bool launch_conv1d_tc16p(const ConvArgs& a, cudaStream_t s);
bool tc16p_enabled();
void set_tc16p_enabled(bool on);
int tc16p_install_fault_word(unsigned int* word);
// row-block-resident variant (tc16r_conv.cu) for layers planned with the two-CTA tiling and several N tiles; false = not taken
bool launch_conv1d_tc16r(const ConvArgs& a, cudaStream_t s);
bool tc16r_enabled();
int tc16r_install_fault_word(unsigned int* word);
void set_tensor_cores_enabled(bool on);
bool tensor_cores_enabled();

// fused ResBlock2/MRF stage (fused_rb.cu): one launch per generator stage with C in {32, 64}
bool fused_rb_supported(int C, int nrb, const int* k, const int* d1, const int* d2);
size_t fused_rb_conv_floats(int C, int K);
void launch_fused_rb_pack(const float* w_folded /*[C][C][K]*/, float* dst, int C, int K, cudaStream_t s);
int launch_fused_rb(int C, FusedRbArgs a, cudaStream_t s);   // fills Rp / nq; returns 0 on success
void set_fused_resblock_enabled(bool on);
bool fused_resblock_enabled();

// f16-split fused MRF stage (fused_mrf16.cu): ResBlock1 and ResBlock2 stages with C in {32, 64}
bool fused_mrf16_supported(int C, int type, int nrb, const int* k, const int (*dil)[kMrfMaxConv], int nconv);
void launch_fused_mrf16_pack(const float* w_folded /*[C][C][K]*/, void* dst, int C, int K, cudaStream_t s);
int launch_fused_mrf16(int C, FusedMrfArgs a, cudaStream_t s);
// length-aware work-item list of a stage (samples per frame `rate`, `margin` frames beyond each utterance's length)
size_t mrf_item_map_bytes(int B, int T);
int set_mrf16_item_rows(int rows);   // option "mrf_item_rows": 0 = policy, 128 / 256 / 384 forced (C = 32 ResBlock2 stage)
int mrf16_item_rows_option();
int mrf16_last_item_rows();
int fused_mrf16_item_rows(int C, int type, int B, int T);   // output samples per work item of the stage kernel launch_fused_mrf16 will pick
void launch_mrf_item_map(const long long* lengths, int B, int T, int rate, int margin, int item_rows, void* scratch,
                         const int2_t** item_map, const int** n_items_dev, cudaStream_t s);

struct ConvTArgs {
  const float* in = nullptr;  // [B][Cin][T]
  const float* w = nullptr;   // packed [Cin][ntaps][CoutPad][u]
  const float* bias = nullptr;
  float* out = nullptr;       // [B][Cout][T*u]
  int B = 0, Cin = 0, Cout = 0, CoutPad = 0, T = 0, u = 1, ntaps = 2, pad = 0;
  float pre_slope = 0.1f;     // leaky_relu on the input (decoders.py:69)
};
void launch_conv_transpose1d(const ConvTArgs& a, cudaStream_t s);

// conv_post: lrelu(slope) -> Conv1d(C->1, k, no bias) -> tanh   (decoders.py:78-80)
void launch_conv_post_tanh(const float* in, const float* w /*[C][K]*/, float* out, int B, int C, int T, int K,
                           float slope, cudaStream_t s, const long long* la_len = nullptr, int la_rate = 1, int la_margin = 0);

// ---------------------------------------------------------------- weight preparation
void launch_weight_norm_fold(const float* v, const float* g, float* out, int rows, int cols, cudaStream_t s);
// dst[ci][k][p] = src[co_map[p]][ci_map[ci]][k]   (co_map[p] < 0 -> 0)
void launch_pack_conv(const float* src, float* dst, const int* co_map, const int* ci_map, int Cin, int K, int CoutPad,
                      int src_cin, cudaStream_t s);
// dst[ci][tap][co][r] = src[ci][co][r + tap*u]  (src [Cin][Cout][k]); co >= Cout -> 0
void launch_pack_convT(const float* src, float* dst, int Cin, int Cout, int CoutPad, int k, int u, cudaStream_t s);
void launch_gather_vec(const float* src, float* dst, const int* map, int n, cudaStream_t s);
void launch_convT_as_conv(const float* src, const float* bias, float* dst, float* bias_out, int Cin, int Cout, int k, int u,
                          cudaStream_t s);

// ---------------------------------------------------------------- elementwise / norm
void launch_embed(const long long* ids, const long long* lengths, const float* table, float* out, int B, int Tx, int H,
                  int n_vocab, float scale, cudaStream_t s);
void launch_speaker_embed(const long long* sid, const float* table, float* g, int B, int gin, int n_speakers,
                          cudaStream_t s);

struct LnArgs {
  const float* a = nullptr;      // [B][C][T]
  const float* b = nullptr;      // optional addend (same shape)
  const float* gamma = nullptr;
  const float* beta = nullptr;
  const float* res = nullptr;    // optional: out = res + y
  float* out = nullptr;
  const long long* lengths = nullptr;
  // optional depthwise front-end: a' = dwbias[c] + sum_k dww[c][k] * a[c][t+(k-1)*dil] * mask(t+(k-1)*dil)
  const float* dww = nullptr;    // [C][3]
  const float* dwb = nullptr;
  int dil = 1;
  int act = 0;                   // 0 none, 1 gelu(erf)
  int out_mask = 0;
  int B = 0, C = 0, T = 0;
  float eps = 1e-5f;
};
void launch_layernorm(const LnArgs& a, cudaStream_t s);

// relative-position multi-head attention core (attentions.py:232-282)
// qkv [B][3C][T] (q rows 0..C-1, k rows C..2C-1, v rows 2C..3C-1), out [B][C][T]
void launch_rel_attention(const float* qkv, const float* emb_k, const float* emb_v, const long long* lengths, float* out,
                          int B, int C, int T, int n_heads, int window, cudaStream_t s);
// the same contraction on the tensor pipe (attn_tc.cu; 64 <= T <= 128, head dimension 96, window 4)
bool rel_attention_tc_supported(int C, int T, int n_heads, int window);
int launch_rel_attention_tc(const float* qkv, const float* emb_k, const float* emb_v, const long long* lengths, float* out,
                            int B, int C, int T, int n_heads, int window, cudaStream_t s);
int attn_tc_install_fault_word(unsigned int* word);

// ---------------------------------------------------------------- stochastic duration predictor
// h[b][c][t] = w[c]*z[b][src_ch][t] + bias[c] + cond[b][c][t]    (ConvFlow.pre + DDSConv `x + g`)
void launch_convflow_pre(const float* z, int src_ch, const float* w, const float* bias, const float* cond, float* out,
                         int B, int C, int T, cudaStream_t s);
// zout[b][0][t] = zin[b][1][t]*m ; zout[b][1][t] = RQS^-1(zin[b][0][t]; u[b][0:29][t])*m   (Flip + ConvFlow reverse)
void launch_spline_flip(const float* zin, const float* u /*[B][32pad?]*/, int u_cs_rows, float* zout,
                        const long long* lengths, int B, int T, float inv_sqrt_h, cudaStream_t s);
void launch_scale(const float* in, float* out, float scale, long long n, cudaStream_t s);
// logw[b][t] = (z[b][1][t] - m0) * exp(-logs0) * mask   (final Flip + ElementwiseAffine reverse, channel 0)
void launch_sdp_final(const float* z, const float* m, const float* logs, const long long* lengths, float* logw, int B,
                      int T, cudaStream_t s);

// ---------------------------------------------------------------- length regulation
void launch_length_regulate(const float* logw, const long long* x_lengths, const float* durations, float length_scale,
                            int B, int Tx, float* w_ceil, int* cum, long long* y_lengths, cudaStream_t s);
void launch_expand_prior(const float* m, const float* logs, const int* cum, const long long* x_lengths,
                         const long long* y_lengths, const float* noise, long long noise_bs, long long noise_rs,
                         float noise_scale, int B, int C, int Tx, int Ty, float* m_p, float* logs_p, float* z_p,
                         float* attn, float* y_mask, cudaStream_t s);
void launch_max_i64(const long long* v, int n, long long* out, cudaStream_t s);
// [B][L][C] -> [B][C][L]
void launch_transpose_blc(const float* in, float* out, int B, int L, int C, cudaStream_t s);
// callers' output stage: mode 0 x32767, 1 per-utterance peak * 0.6, 2 batch-global peak * 0.6; clip, truncate to int16
void launch_audio_to_int16(const float* audio, const long long* lengths, int B, long long L, int mode, float* peak,
                           short* out, cudaStream_t s);

// soft watchdog of the mbarrier pipelines (tc_prims.cuh): every translation unit with waits installs the host-visible
// fault word on the current device
int tc_conv_install_fault_word(unsigned int* word);
int tc16_conv_install_fault_word(unsigned int* word);
int fused_rb_install_fault_word(unsigned int* word);
int fused_mrf16_install_fault_word(unsigned int* word);

// ---------------------------------------------------------------- Vocos / VITS2 helpers (SURVEY.md 8f rank 4)
void launch_reflect_pad_left(const float* in, long long in_bs, int in_cs, const long long* lengths, float* out, int B, int C,
                             int T, cudaStream_t s);
void launch_gather_channels(const float* in, long long in_bs, int c0, int cstep, const long long* lengths, float* out,
                            float* out_masked, int B, int C, int T, cudaStream_t s);
void launch_vocos_spec(float* x, int B, int K, int F, cudaStream_t s);
void launch_idft_weight(float* w /*[N][N+2][1]*/, int N, cudaStream_t s);
void launch_istft_overlap_add(const float* frames /*[B][N][F]*/, float* out /*[B][hop*(F-1)]*/, int B, int N, int hop, int F,
                              cudaStream_t s);
void launch_scale_rows(const float* w, const float* bias, const float* sc, float* w_out, float* b_out, int rows, int cols,
                       cudaStream_t s);

// ---------------------------------------------------------------- posterior encoder / linear spectrogram (voice conversion)
// stats [B][2C][T] -> z = (m + noise * exp(logs)) * mask; m, logs [B][C][T] and y_mask [B][1][T] optional
void launch_posterior_sample(const float* stats, const float* noise, const long long* lengths, float* z, float* m, float* logs,
                             float* y_mask, int B, int C, int T, cudaStream_t s);
// audio [B][L] -> frames [B][N][F] of each utterance reflect-padded by `pad` at its own length (0 beyond its F_b frames)
void launch_spec_frames(const float* audio, long long L, const long long* lengths, float* frames, int B, int N, int hop, int pad,
                        int F, cudaStream_t s);
void launch_dft_weight(float* w /*[N+2][N][1]*/, int N, cudaStream_t s);
// dft [B][2K][F] -> spec [B][K][F] magnitudes (+1e-6 inside the root), 0 beyond F_b; spec_lengths int64[B] (optional)
void launch_spec_magnitude(const float* dft, const long long* lengths, float* spec, long long* spec_lengths, int B, int K, int F,
                           int N, int hop, int pad, cudaStream_t s);

unsigned long long kernel_launch_counter();
void count_launch();

// Per-DEVICE cache of cudaFuncAttributeMaxDynamicSharedMemorySize (the attribute is per device and per function;
// a process may drive several GPUs and several host threads).  One static instance per launch site / kernel
// instantiation.  ensure() is thread-safe (double-checked under a mutex) and returns the CUDA error, if any.
struct DynSmemAttr {
  static constexpr int kMaxDev = 64;
  size_t have[kMaxDev] = {};
  cudaError_t ensure(const void* func, size_t bytes);
};
// SM count of the current device (cached per device)
int current_device_sm_count();
// last launcher-side error (cudaFuncSetAttribute failures etc.); cleared when read
cudaError_t take_launcher_error();
void note_launcher_error(cudaError_t e);

}  // namespace wetts
