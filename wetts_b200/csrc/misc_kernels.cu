// Non-convolution kernels of the VITS hot path: embedding, channel LayerNorm (+ fused
// depthwise front-end / GELU / residual), relative-position attention, the
// rational-quadratic spline inverse, length regulation, prior expansion + sampling,
// and the weight-preparation kernels (weight-norm folding, re-layout).
#include <math_constants.h>

#include "kernels.cuh"

namespace wetts {
namespace {

// ------------------------------------------------------------------ weight preparation
__global__ void weight_norm_fold_kernel(const float* __restrict__ v, const float* __restrict__ g, float* __restrict__ out,
                                        int rows, int cols) {
  // one block per row (dim 0): out = v * g / ||v||   (torch weight_norm, dim=0)
  const int r = blockIdx.x;
  const float* vr = v + (long long)r * cols;
  float ss = 0.f;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) ss += vr[i] * vr[i];
  __shared__ float red[32];
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  const float scale = g[r] / sqrtf(red[0]);
  for (int i = threadIdx.x; i < cols; i += blockDim.x) out[(long long)r * cols + i] = vr[i] * scale;
}

__global__ void pack_conv_kernel(const float* __restrict__ src, float* __restrict__ dst, const int* __restrict__ co_map,
                                 const int* __restrict__ ci_map, int Cin, int K, int CoutPad, int src_cin) {
  const long long n = (long long)Cin * K * CoutPad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i % CoutPad);
    const int k = (int)((i / CoutPad) % K);
    const int ci = (int)(i / ((long long)CoutPad * K));
    const int co = co_map[p];
    const int sci = ci_map ? ci_map[ci] : ci;
    dst[i] = co < 0 ? 0.f : src[((long long)co * src_cin + sci) * K + k];
  }
}

__global__ void pack_convT_kernel(const float* __restrict__ src, float* __restrict__ dst, int Cin, int Cout, int CoutPad,
                                  int k, int u) {
  const int ntaps = k / u;
  const long long n = (long long)Cin * ntaps * CoutPad * u;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i % u);
    const int co = (int)((i / u) % CoutPad);
    const int tap = (int)((i / ((long long)u * CoutPad)) % ntaps);
    const int ci = (int)(i / ((long long)u * CoutPad * ntaps));
    dst[i] = co < Cout ? src[((long long)ci * Cout + co) * k + r + tap * u] : 0.f;
  }
}

// ConvTranspose1d weight [Cin][Cout][k] -> equivalent Conv1d weight [Cout*u][Cin][ntaps] of the polyphase
// form: W'[co*u + r][ci][k'] = W[ci][co][r + (ntaps-1-k')*u]; bias'[co*u + r] = bias[co]
__global__ void convT_as_conv_kernel(const float* __restrict__ src, const float* __restrict__ bias,
                                     float* __restrict__ dst, float* __restrict__ bias_out, int Cin, int Cout, int k, int u) {
  const int ntaps = k / u;
  const long long n = (long long)Cout * u * Cin * ntaps;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int kp = (int)(i % ntaps);
    const int ci = (int)((i / ntaps) % Cin);
    const int cp = (int)(i / ((long long)ntaps * Cin));
    const int co = cp / u, r = cp - co * u;
    dst[i] = src[((long long)ci * Cout + co) * k + r + (ntaps - 1 - kp) * u];
    if (ci == 0 && kp == 0) bias_out[cp] = bias[co];
  }
}

__global__ void gather_vec_kernel(const float* __restrict__ src, float* __restrict__ dst, const int* __restrict__ map,
                                  int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = map[i] < 0 ? 0.f : src[map[i]];
}

// ------------------------------------------------------------------ embeddings
__global__ void embed_kernel(const long long* __restrict__ ids, const long long* __restrict__ lengths,
                             const float* __restrict__ table, float* __restrict__ out, int Tx, int H, int n_vocab,
                             float scale) {
  // block: 32 time steps of one utterance; smem transpose so both sides are coalesced
  extern __shared__ float tile[];  // [32][H+1]
  const int b = blockIdx.y, t0 = blockIdx.x * 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const long long len = lengths[b];
  for (int tt = warp; tt < 32; tt += nw) {
    const int t = t0 + tt;
    long long id = (t < Tx) ? ids[(long long)b * Tx + t] : 0;
    if (id < 0) id = 0;
    if (id >= n_vocab) id = n_vocab - 1;
    const float m = (t < Tx && t < len) ? scale : 0.f;
    for (int c = lane; c < H; c += 32) tile[tt * (H + 1) + c] = table[id * H + c] * m;
  }
  __syncthreads();
  for (int c = warp; c < H; c += nw) {
    const int t = t0 + lane;
    if (t < Tx) out[((long long)b * H + c) * Tx + t] = tile[lane * (H + 1) + c];
  }
}

__global__ void speaker_embed_kernel(const long long* __restrict__ sid, const float* __restrict__ table,
                                     float* __restrict__ g, int gin, int n_speakers) {
  const int b = blockIdx.x;
  long long s = sid[b];
  if (s < 0) s = 0;
  if (s >= n_speakers) s = n_speakers - 1;
  for (int c = threadIdx.x; c < gin; c += blockDim.x) g[(long long)b * gin + c] = table[s * gin + c];
}

// ------------------------------------------------------------------ channel LayerNorm
// PT = channels per thread: 32 (C <= 256, every reference LayerNorm of the HiFi-GAN recipes) or 64 (C <= 512, Vocos)

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

template <int kLnMaxPerThread>
__global__ void __launch_bounds__(256) layernorm_kernel(const LnArgs a) {
  // block = 32 time steps x 8 channel groups; channel c handled by warp (c % 8)
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.y, t = blockIdx.x * 32 + lane;
  const int C = a.C, T = a.T;
  const bool tok = t < T;
  const long long len = a.lengths ? a.lengths[b] : (long long)T;
  const long long base = (long long)b * C * T;
  float v[kLnMaxPerThread];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxPerThread; ++i) {
    const int c = warp + 8 * i;
    float x = 0.f;
    if (c < C && tok) {
      const float* row = a.a + base + (long long)c * T;
      if (a.dww) {
        x = a.dwb[c];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int tt = t + (k - 1) * a.dil;
          if (tt >= 0 && tt < T && tt < len) x = fmaf(a.dww[c * 3 + k], row[tt], x);
        }
      } else {
        x = row[t];
        if (a.b) x += a.b[base + (long long)c * T + t];
      }
      sum += x;
    }
    v[i] = x;
  }
  red[warp][lane] = sum;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += red[w][lane];
  const float mean = tot / (float)C;
  __syncthreads();
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxPerThread; ++i) {
    const int c = warp + 8 * i;
    if (c < C) { const float d = v[i] - mean; sq = fmaf(d, d, sq); }
  }
  red[warp][lane] = sq;
  __syncthreads();
  float vtot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) vtot += red[w][lane];
  const float rstd = rsqrtf(vtot / (float)C + a.eps);
  if (!tok) return;
  const float msk = (t < len) ? 1.f : 0.f;
#pragma unroll
  for (int i = 0; i < kLnMaxPerThread; ++i) {
    const int c = warp + 8 * i;
    if (c >= C) continue;
    float y = (v[i] - mean) * rstd * a.gamma[c] + a.beta[c];
    if (a.act == 1) y = gelu_erf(y);
    const long long off = base + (long long)c * T + t;
    if (a.res) y += a.res[off];
    if (a.out_mask) y *= msk;
    a.out[off] = y;
  }
}

// ------------------------------------------------------------------ relative-position attention
constexpr int kAttQ = 16;    // queries per CTA
constexpr int kAttKT = 64;   // keys per staged tile
constexpr int kAttThreads = 128;

__global__ void __launch_bounds__(kAttThreads) rel_attention_kernel(const float* __restrict__ qkv,
                                                                    const float* __restrict__ emb_k,
                                                                    const float* __restrict__ emb_v,
                                                                    const long long* __restrict__ lengths,
                                                                    float* __restrict__ out, int C, int T, int n_heads,
                                                                    int window, int dk, int Tpad) {
  extern __shared__ __align__(16) float smem[];
  float* qs = smem;                        // [dk][kAttQ]   (scaled by 1/sqrt(dk))
  float* kt = qs + dk * kAttQ;             // [dk][kAttKT+1]  K tile, later V tile
  float* S = kt + dk * (kAttKT + 1);       // [kAttQ][Tpad]
  float* os = S + kAttQ * Tpad;            // [dk][kAttQ]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.x * kAttQ, h = blockIdx.y, b = blockIdx.z;
  const long long len = lengths[b];
  const float* qb = qkv + ((long long)b * 3 * C + h * dk) * T;
  const float* kb = qb + (long long)C * T;
  const float* vb = kb + (long long)C * T;
  const float scale = rsqrtf((float)dk);
  const int nrel = 2 * window + 1;

  for (int idx = tid; idx < dk * kAttQ; idx += kAttThreads) {
    const int d = idx / kAttQ, i = idx - d * kAttQ;
    qs[idx] = (i0 + i < T) ? qb[(long long)d * T + i0 + i] * scale : 0.f;
  }
  // ---- scores
  for (int j0 = 0; j0 < T; j0 += kAttKT) {
    __syncthreads();
    for (int idx = tid; idx < dk * kAttKT; idx += kAttThreads) {
      const int d = idx / kAttKT, jj = idx - d * kAttKT;
      kt[d * (kAttKT + 1) + jj] = (j0 + jj < T) ? kb[(long long)d * T + j0 + jj] : 0.f;
    }
    __syncthreads();
    const int jj = tid & (kAttKT - 1), ig = tid / kAttKT;  // ig in {0,1}: queries ig*8 .. ig*8+7
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.f;
    for (int d = 0; d < dk; ++d) {
      const float kv = kt[d * (kAttKT + 1) + jj];
      const float4 q0 = *reinterpret_cast<const float4*>(qs + d * kAttQ + ig * 8);
      const float4 q1 = *reinterpret_cast<const float4*>(qs + d * kAttQ + ig * 8 + 4);
      acc[0] = fmaf(q0.x, kv, acc[0]); acc[1] = fmaf(q0.y, kv, acc[1]);
      acc[2] = fmaf(q0.z, kv, acc[2]); acc[3] = fmaf(q0.w, kv, acc[3]);
      acc[4] = fmaf(q1.x, kv, acc[4]); acc[5] = fmaf(q1.y, kv, acc[5]);
      acc[6] = fmaf(q1.z, kv, acc[6]); acc[7] = fmaf(q1.w, kv, acc[7]);
    }
    if (j0 + jj < T) {
#pragma unroll
      for (int q = 0; q < 8; ++q) S[(ig * 8 + q) * Tpad + j0 + jj] = acc[q];
    }
  }
  __syncthreads();
  // ---- relative-key bias on the band |j-i| <= window, then masking (attentions.py:247-262)
  for (int idx = tid; idx < kAttQ * nrel; idx += kAttThreads) {
    const int i = idx / nrel, r = idx - i * nrel;
    const int ig_ = i0 + i, j = ig_ + r - window;
    if (emb_k && ig_ < T && j >= 0 && j < T) {      // emb_k == nullptr: plain attention (window_size=None)
      float s = 0.f;
      for (int d = 0; d < dk; ++d) s = fmaf(qs[d * kAttQ + i], emb_k[r * dk + d], s);
      S[i * Tpad + j] += s;
    }
  }
  __syncthreads();
  // ---- masked softmax, one warp per row
  for (int i = warp; i < kAttQ; i += kAttThreads / 32) {
    const int ig_ = i0 + i;
    if (ig_ >= T) continue;
    float* row = S + i * Tpad;
    const bool qvalid = ig_ < len;
    float mx = -CUDART_INF_F;
    for (int j = lane; j < T; j += 32) {
      float s = row[j];
      if (!qvalid || j >= len) { s = -1e4f; row[j] = s; }
      mx = fmaxf(mx, s);
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float e = expf(row[j] - mx);
      row[j] = e;
      sum += e;
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
    for (int j = lane; j < T; j += 32) row[j] *= inv;
  }
  // ---- O = P V : thread -> channels d = lane + 32*dd, queries qg*4 .. qg*4+3
  const int qg = warp;  // 4 warps x 4 queries
  float oacc[3][4];
#pragma unroll
  for (int dd = 0; dd < 3; ++dd)
#pragma unroll
    for (int q = 0; q < 4; ++q) oacc[dd][q] = 0.f;
  for (int j0 = 0; j0 < T; j0 += kAttKT) {
    __syncthreads();
    for (int idx = tid; idx < dk * kAttKT; idx += kAttThreads) {
      const int d = idx / kAttKT, jj = idx - d * kAttKT;
      kt[d * (kAttKT + 1) + jj] = (j0 + jj < T) ? vb[(long long)d * T + j0 + jj] : 0.f;
    }
    __syncthreads();
    const int jn = min(kAttKT, T - j0);
    for (int jj = 0; jj < jn; ++jj) {
      float p[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) p[q] = S[(qg * 4 + q) * Tpad + j0 + jj];
#pragma unroll
      for (int dd = 0; dd < 3; ++dd) {
        const int d = lane + 32 * dd;
        if (d < dk) {
          const float vv = kt[d * (kAttKT + 1) + jj];
#pragma unroll
          for (int q = 0; q < 4; ++q) oacc[dd][q] = fmaf(p[q], vv, oacc[dd][q]);
        }
      }
    }
  }
  // ---- relative values (attentions.py:273-279) and store
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = qg * 4 + q, ig_ = i0 + i;
    if (ig_ < T && emb_v) {
      for (int r = 0; r < nrel; ++r) {
        const int j = ig_ + r - window;
        if (j < 0 || j >= T) continue;
        const float p = S[i * Tpad + j];
#pragma unroll
        for (int dd = 0; dd < 3; ++dd) {
          const int d = lane + 32 * dd;
          if (d < dk) oacc[dd][q] = fmaf(p, emb_v[r * dk + d], oacc[dd][q]);
        }
      }
    }
#pragma unroll
    for (int dd = 0; dd < 3; ++dd) {
      const int d = lane + 32 * dd;
      if (d < dk) os[d * kAttQ + i] = oacc[dd][q];
    }
  }
  __syncthreads();
  float* ob = out + ((long long)b * C + h * dk) * T;
  for (int idx = tid; idx < dk * kAttQ; idx += kAttThreads) {
    const int d = idx / kAttQ, i = idx - d * kAttQ;
    if (i0 + i < T) ob[(long long)d * T + i0 + i] = os[idx];
  }
}

// ------------------------------------------------------------------ Vocos / VITS2 helpers (SURVEY.md 8f rank 4)
// out[b][c][j] = in[b][c][j == 0 ? 1 : j - 1] * (src < len)    (nn.ReflectionPad1d([1, 0]) after the frame mask)
__global__ void reflect_pad_left_kernel(const float* __restrict__ in, long long in_bs, int in_cs, const long long* __restrict__ lengths,
                                        float* __restrict__ out, int C, int T) {
  const int b = blockIdx.z, c = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > T) return;
  const int src = (j == 0) ? (T > 1 ? 1 : 0) : j - 1;
  float v = in[(long long)b * in_bs + (long long)c * in_cs + src];
  if (lengths && src >= lengths[b]) v = 0.f;
  out[((long long)b * C + c) * (T + 1) + j] = v;
}
// out[b][c][t] = in[b][c0 + c*cstep][t] (optionally * (t < len)): a channel slice / reversal of z (Flip folded in)
__global__ void gather_channels_kernel(const float* __restrict__ in, long long in_bs, int c0, int cstep,
                                       const long long* __restrict__ lengths, float* __restrict__ out, float* __restrict__ out_masked,
                                       int C, int T) {
  const int b = blockIdx.z, c = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float v = in[(long long)b * in_bs + (long long)(c0 + c * cstep) * T + t];
  const long long o = ((long long)b * C + c) * T + t;
  if (out) out[o] = v;
  if (out_masked) out_masked[o] = (lengths && t >= lengths[b]) ? 0.f : v;
}
// x [B][2K][F] (log-magnitudes, phases) -> in place [re | im]: mag = min(exp(m), 100)  (decoders.py:300-305)
__global__ void vocos_spec_kernel(float* __restrict__ x, int K, int F) {
  const int b = blockIdx.z, k = blockIdx.y, f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  float* pm = x + ((long long)b * 2 * K + k) * F + f;
  float* pp = pm + (long long)K * F;
  const float mag = fminf(expf(*pm), 100.f);
  float sn, cs;
  sincosf(*pp, &sn, &cs);
  *pm = mag * cs;
  *pp = mag * sn;
}
// inverse real DFT + synthesis window as a 1x1 conv weight [N][2K][1] (K = N/2 + 1): row n, column k (re) / K + k (im)
__global__ void idft_weight_kernel(float* __restrict__ w, int N) {
  const int K = N / 2 + 1;
  const long long total = (long long)N * 2 * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % (2 * K)), n = (int)(i / (2 * K));
    const int k = col < K ? col : col - K;
    const double ck = (k == 0 || k == N / 2) ? 1.0 : 2.0;
    const long long kn = ((long long)k * n) % N;                       // exact angle reduction
    const double ang = 6.283185307179586476925286766559 * (double)kn / (double)N;
    const double win = 0.5 - 0.5 * cos(6.283185307179586476925286766559 * (double)n / (double)N);   // periodic hann
    double v = (col < K) ? ck * cos(ang) : ((k == 0 || k == N / 2) ? 0.0 : -ck * sin(ang));
    w[i] = (float)(v * win / (double)N);
  }
}
// out[b][t] = sum_f frames[b][t + N/2 - f*hop][f] / sum_f win^2[t + N/2 - f*hop],  t < hop * (F - 1)   (torch.istft, center)
__global__ void istft_overlap_add_kernel(const float* __restrict__ frames, float* __restrict__ out, int N, int hop, int F) {
  const int b = blockIdx.y;
  const long long L = (long long)hop * (F - 1);
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t >= L) return;
  const long long s = t + N / 2;
  int f_hi = (int)(s / hop);
  if (f_hi > F - 1) f_hi = F - 1;
  float acc = 0.f, env = 0.f;
  for (int f = f_hi; f >= 0; --f) {
    const long long n = s - (long long)f * hop;
    if (n >= N) break;
    acc += frames[((long long)b * N + n) * F + f];
    const float wv = 0.5f - 0.5f * cospif(2.0f * (float)n / (float)N);
    env = fmaf(wv, wv, env);
  }
  out[(long long)b * L + t] = acc / env;
}
// ------------------------------------------------------------------ posterior encoder / linear spectrogram
// stats [B][2C][T] (m rows 0..C-1, logs rows C..2C-1, already masked) -> z = (m + noise * exp(logs)) * mask
// (encoders.py:97-98); m / logs / y_mask written when non-null (y_mask [B][1][T] by the c == 0 threads)
__global__ void posterior_sample_kernel(const float* __restrict__ stats, const float* __restrict__ noise,
                                        const long long* __restrict__ lengths, float* __restrict__ z, float* __restrict__ m_out,
                                        float* __restrict__ logs_out, float* __restrict__ y_mask, int C, int T) {
  const int b = blockIdx.z, c = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float msk = t < lengths[b] ? 1.f : 0.f;
  const long long o = ((long long)b * C + c) * T + t;
  const float m = stats[((long long)b * 2 * C + c) * T + t];
  const float ls = stats[((long long)b * 2 * C + C + c) * T + t];
  z[o] = (m + noise[o] * expf(ls)) * msk;
  if (m_out) m_out[o] = m;
  if (logs_out) logs_out[o] = ls;
  if (y_mask && c == 0) y_mask[(long long)b * T + t] = msk;
}
// frames[b][n][f] = audio[b][reflect(f*hop + n - pad)] for f < F_b (the frames torch.stft(center=False) takes from the
// utterance reflect-padded by `pad` at its own length L_b), 0 for f >= F_b.  The analysis window is in the DFT weight.
__global__ void spec_frames_kernel(const float* __restrict__ audio, long long L, const long long* __restrict__ lengths,
                                   float* __restrict__ frames, int N, int hop, int pad, int F) {
  const int b = blockIdx.z, n = blockIdx.y, f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const long long Lb = lengths[b];
  const long long Fb = 1 + (Lb + 2 * pad - N) / hop;
  float v = 0.f;
  if (f < Fb) {
    long long i = (long long)f * hop + n - pad;
    if (i < 0) i = -i;
    if (i >= Lb) i = 2 * (Lb - 1) - i;
    v = audio[(long long)b * L + i];
  }
  frames[((long long)b * N + n) * F + f] = v;
}
// forward real DFT x periodic hann window as a 1x1 conv weight [2K][N][1] (K = N/2 + 1): row k = re, row K + k = im
// (the forward twin of idft_weight_kernel)
__global__ void dft_weight_kernel(float* __restrict__ w, int N) {
  const int K = N / 2 + 1;
  const long long total = (long long)2 * K * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % N), row = (int)(i / N);
    const int k = row < K ? row : row - K;
    const long long kn = ((long long)k * n) % N;                       // exact angle reduction
    const double ang = 6.283185307179586476925286766559 * (double)kn / (double)N;
    const double win = 0.5 - 0.5 * cos(6.283185307179586476925286766559 * (double)n / (double)N);   // periodic hann
    w[i] = (float)((row < K ? cos(ang) : -sin(ang)) * win);
  }
}
// dft [B][2K][F] (re | im) -> spec [B][K][F] = sqrt(re^2 + im^2 + 1e-6) for f < F_b, exactly 0 beyond
// (mel_processing.py:91); spec_lengths[b] = F_b written by the (k == 0, f == 0) thread
__global__ void spec_magnitude_kernel(const float* __restrict__ dft, const long long* __restrict__ lengths, float* __restrict__ spec,
                                      long long* __restrict__ spec_lengths, int K, int F, int N, int hop, int pad) {
  const int b = blockIdx.z, k = blockIdx.y, f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const long long Fb = 1 + (lengths[b] + 2 * pad - N) / hop;
  float v = 0.f;
  if (f < Fb) {
    const float re = dft[((long long)b * 2 * K + k) * F + f];
    const float im = dft[((long long)b * 2 * K + K + k) * F + f];
    v = sqrtf(re * re + im * im + 1e-6f);
  }
  spec[((long long)b * K + k) * F + f] = v;
  if (spec_lengths && k == 0 && f == 0) spec_lengths[b] = Fb;
}

// w[r][*] *= s[r], b[r] *= s[r]   (ConvNeXt layer scale folded into pw_conv2, decoders.py:245)
__global__ void scale_rows_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ s,
                                  float* __restrict__ w_out, float* __restrict__ b_out, int rows, int cols) {
  const long long total = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    w_out[i] = w[i] * s[i / cols];
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) b_out[r] = bias[r] * s[r];
}

// ------------------------------------------------------------------ SDP pieces
__global__ void convflow_pre_kernel(const float* __restrict__ z, int src_ch, const float* __restrict__ w,
                                    const float* __restrict__ bias, const float* __restrict__ cond,
                                    float* __restrict__ out, int C, int T) {
  const int b = blockIdx.z, c = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const long long off = ((long long)b * C + c) * T + t;
  out[off] = fmaf(w[c], z[((long long)b * 2 + src_ch) * T + t], bias[c]) + cond[off];
}

__device__ __forceinline__ float softplusf_t(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// transforms.py:47-187 inverse branch for one scalar, 10 bins, linear tails at +-5.
__device__ float rqs_inverse_scalar(float y, const float* uw, const float* uh, const float* ud /*9*/) {
  constexpr int K = 10;
  constexpr float B = 5.f, MINW = 1e-3f, MINH = 1e-3f, MIND = 1e-3f;
  if (!(y >= -B && y <= B)) return y;
  float cw[K + 1], ch[K + 1];
  {
    float mx = uw[0];
#pragma unroll
    for (int k = 1; k < K; ++k) mx = fmaxf(mx, uw[k]);
    float e[K], s = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) { e[k] = expf(uw[k] - mx); s += e[k]; }
    float c = 0.f;
    cw[0] = -B;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      c += MINW + (1.f - MINW * K) * (e[k] / s);
      cw[k + 1] = 2.f * B * c + (-B);
    }
    cw[K] = B;
  }
  {
    float mx = uh[0];
#pragma unroll
    for (int k = 1; k < K; ++k) mx = fmaxf(mx, uh[k]);
    float e[K], s = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) { e[k] = expf(uh[k] - mx); s += e[k]; }
    float c = 0.f;
    ch[0] = -B;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      c += MINH + (1.f - MINH * K) * (e[k] / s);
      ch[k + 1] = 2.f * B * c + (-B);
    }
    ch[K] = B;
  }
  int bin = -1;
#pragma unroll
  for (int k = 0; k <= K; ++k) {
    const float edge = (k == K) ? ch[k] + 1e-6f : ch[k];
    bin += (y >= edge) ? 1 : 0;
  }
  bin = max(0, min(K - 1, bin));
  // boundary derivative parameter log(exp(1 - 1e-3) - 1), evaluated in double then stored
  // as fp32 exactly as the reference does (transforms.py:67-71)
  const float cst = (float)0.5397424172369522;
  float in_cw = 0.f, in_w = 0.f, in_ch = 0.f, in_h = 0.f, d0 = 0.f, d1 = 0.f;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    if (k == bin) {
      in_cw = cw[k]; in_w = cw[k + 1] - cw[k];
      in_ch = ch[k]; in_h = ch[k + 1] - ch[k];
      const float u0 = (k == 0) ? cst : ud[k - 1];
      const float u1 = (k == K - 1) ? cst : ud[k];
      d0 = MIND + softplusf_t(u0);
      d1 = MIND + softplusf_t(u1);
    }
  }
  const float delta = in_h / in_w;
  const float dy = y - in_ch;
  const float tt = dy * (d0 + d1 - 2.f * delta);
  const float a = tt + in_h * (delta - d0);
  const float bq = in_h * d0 - tt;
  const float c = -delta * dy;
  const float disc = bq * bq - 4.f * a * c;
  const float root = (2.f * c) / (-bq - sqrtf(disc));
  return root * in_w + in_cw;
}

__global__ void spline_flip_kernel(const float* __restrict__ zin, const float* __restrict__ u, float* __restrict__ zout,
                                   const long long* __restrict__ lengths, int T, float inv_sqrt_h) {
  const int b = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float msk = (t < lengths[b]) ? 1.f : 0.f;
  const float* ub = u + (long long)b * 29 * T + t;
  float uw[10], uh[10], ud[9];
#pragma unroll
  for (int k = 0; k < 10; ++k) uw[k] = ub[(long long)k * T] * inv_sqrt_h;
#pragma unroll
  for (int k = 0; k < 10; ++k) uh[k] = ub[(long long)(10 + k) * T] * inv_sqrt_h;
#pragma unroll
  for (int k = 0; k < 9; ++k) ud[k] = ub[(long long)(20 + k) * T];
  const float x0 = zin[((long long)b * 2 + 1) * T + t];
  const float x1 = zin[((long long)b * 2 + 0) * T + t];
  zout[((long long)b * 2 + 0) * T + t] = x0 * msk;
  zout[((long long)b * 2 + 1) * T + t] = rqs_inverse_scalar(x1, uw, uh, ud) * msk;
}

__global__ void scale_kernel(const float* __restrict__ in, float* __restrict__ out, float scale, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] * scale;
}

__global__ void sdp_final_kernel(const float* __restrict__ z, const float* __restrict__ m, const float* __restrict__ logs,
                                 const long long* __restrict__ lengths, float* __restrict__ logw, int T) {
  const int b = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float msk = (t < lengths[b]) ? 1.f : 0.f;
  logw[(long long)b * T + t] = (z[((long long)b * 2 + 1) * T + t] - m[0]) * expf(-logs[0]) * msk;
}

// ------------------------------------------------------------------ length regulation
__global__ void __launch_bounds__(256) length_regulate_kernel(const float* __restrict__ logw,
                                                              const long long* __restrict__ x_lengths,
                                                              const float* __restrict__ durations, float length_scale,
                                                              int Tx, float* __restrict__ w_ceil, int* __restrict__ cum,
                                                              long long* __restrict__ y_lengths) {
  // one CTA per utterance: d[t] = ceil(exp(logw)*mask*ls); inclusive scan; y_len = max(sum, 1)
  __shared__ int part[256];
  const int b = blockIdx.x, tid = threadIdx.x;
  const long long len = x_lengths[b];
  const int per = (Tx + 255) / 256;
  const int lo = tid * per, hi = min(Tx, lo + per);
  int local = 0;
  for (int t = lo; t < hi; ++t) {
    const float msk = (t < len) ? 1.f : 0.f;
    float w;
    if (durations) w = durations[(long long)b * Tx + t] * msk;
    else w = ceilf(expf(logw[(long long)b * Tx + t]) * msk * length_scale);
    w = fminf(fmaxf(w, 0.f), 1.0e6f);
    w_ceil[(long long)b * Tx + t] = w;
    local += (int)w;
  }
  part[tid] = local;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const int add = tid >= o ? part[tid - o] : 0;
    __syncthreads();
    part[tid] += add;
    __syncthreads();
  }
  int run = part[tid] - local;
  for (int t = lo; t < hi; ++t) {
    run += (int)w_ceil[(long long)b * Tx + t];
    cum[(long long)b * Tx + t] = run;
  }
  if (tid == 255) y_lengths[b] = part[255] > 1 ? part[255] : 1;
}

__global__ void __launch_bounds__(128) expand_prior_kernel(const float* __restrict__ m, const float* __restrict__ logs,
                                                           const int* __restrict__ cum,
                                                           const long long* __restrict__ y_lengths,
                                                           const float* __restrict__ noise, long long noise_bs,
                                                           long long noise_rs, float noise_scale, int C, int Tx, int Ty,
                                                           float* __restrict__ m_p, float* __restrict__ logs_p,
                                                           float* __restrict__ z_p, float* __restrict__ attn,
                                                           float* __restrict__ y_mask) {
  __shared__ int tsel[128];
  const int b = blockIdx.y, y0 = blockIdx.x * 128, y = y0 + threadIdx.x;
  const int* cb = cum + (long long)b * Tx;
  const long long ylen = y_lengths[b];
  int tph = -1;
  if (y < Ty && y < ylen && y < cb[Tx - 1]) {
    int lo = 0, hi = Tx;  // first t with cum[t] > y
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (cb[mid] > y) hi = mid; else lo = mid + 1;
    }
    tph = lo;
  }
  tsel[threadIdx.x] = tph;
  if (y < Ty) {
    if (y_mask) y_mask[(long long)b * Ty + y] = (y < ylen) ? 1.f : 0.f;
    for (int c = 0; c < C; ++c) {
      float mv = 0.f, lv = 0.f;
      if (tph >= 0) {
        mv = m[((long long)b * C + c) * Tx + tph];
        lv = logs[((long long)b * C + c) * Tx + tph];
      }
      const long long o = ((long long)b * C + c) * Ty + y;
      if (m_p) m_p[o] = mv;
      if (logs_p) logs_p[o] = lv;
      if (z_p) z_p[o] = mv + noise[b * noise_bs + c * noise_rs + y] * expf(lv) * noise_scale;
    }
  }
  if (attn) {
    __syncthreads();
    const int ny = min(128, Ty - y0);
    float* ab = attn + ((long long)b * Ty + y0) * Tx;
    for (int idx = threadIdx.x; idx < ny * Tx; idx += 128) {
      const int yy = idx / Tx, tx = idx - yy * Tx;
      ab[idx] = (tsel[yy] == tx) ? 1.f : 0.f;
    }
  }
}

__global__ void max_i64_kernel(const long long* __restrict__ v, int n, long long* __restrict__ out) {
  __shared__ long long red[32];
  long long mx = LLONG_MIN;
  for (int i = threadIdx.x; i < n; i += blockDim.x) mx = v[i] > mx ? v[i] : mx;
  for (int o = 16; o > 0; o >>= 1) {
    const long long other = __shfl_xor_sync(0xffffffffu, mx, o);
    mx = other > mx ? other : mx;
  }
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mx = red[w] > mx ? red[w] : mx;
    out[0] = mx;
  }
}

__global__ void transpose_blc_kernel(const float* __restrict__ in, float* __restrict__ out, int L, int C) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, l0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* ib = in + (long long)b * L * C;
  float* ob = out + (long long)b * L * C;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int l = l0 + r, c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (l < L && c < C) ? ib[(long long)l * C + c] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = c0 + r, l = l0 + threadIdx.x;
    if (c < C && l < L) ob[(long long)c * L + l] = tile[threadIdx.x][r];
  }
}

}  // namespace

// ------------------------------------------------------------------ launchers
void launch_weight_norm_fold(const float* v, const float* g, float* out, int rows, int cols, cudaStream_t s) {
  weight_norm_fold_kernel<<<rows, 256, 0, s>>>(v, g, out, rows, cols);
  count_launch();
}
void launch_pack_conv(const float* src, float* dst, const int* co_map, const int* ci_map, int Cin, int K, int CoutPad,
                      int src_cin, cudaStream_t s) {
  const long long n = (long long)Cin * K * CoutPad;
  pack_conv_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, co_map, ci_map, Cin,
                                                                                            K, CoutPad, src_cin);
  count_launch();
}
void launch_pack_convT(const float* src, float* dst, int Cin, int Cout, int CoutPad, int k, int u, cudaStream_t s) {
  const long long n = (long long)Cin * (k / u) * CoutPad * u;
  pack_convT_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, dst, Cin, Cout, CoutPad,
                                                                                             k, u);
  count_launch();
}
void launch_convT_as_conv(const float* src, const float* bias, float* dst, float* bias_out, int Cin, int Cout, int k, int u,
                          cudaStream_t s) {
  const long long n = (long long)Cout * u * Cin * (k / u);
  convT_as_conv_kernel<<<(int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256), 256, 0, s>>>(src, bias, dst, bias_out, Cin,
                                                                                               Cout, k, u);
  count_launch();
}
void launch_gather_vec(const float* src, float* dst, const int* map, int n, cudaStream_t s) {
  gather_vec_kernel<<<(n + 255) / 256, 256, 0, s>>>(src, dst, map, n);
  count_launch();
}
void launch_embed(const long long* ids, const long long* lengths, const float* table, float* out, int B, int Tx, int H,
                  int n_vocab, float scale, cudaStream_t s) {
  dim3 grid((Tx + 31) / 32, B);
  embed_kernel<<<grid, 256, sizeof(float) * 32 * (H + 1), s>>>(ids, lengths, table, out, Tx, H, n_vocab, scale);
  count_launch();
}
void launch_speaker_embed(const long long* sid, const float* table, float* g, int B, int gin, int n_speakers,
                          cudaStream_t s) {
  speaker_embed_kernel<<<B, 128, 0, s>>>(sid, table, g, gin, n_speakers);
  count_launch();
}
void launch_layernorm(const LnArgs& a, cudaStream_t s) {
  dim3 grid((a.T + 31) / 32, a.B);
  if (a.C <= 256) layernorm_kernel<32><<<grid, 256, 0, s>>>(a);
  else layernorm_kernel<64><<<grid, 256, 0, s>>>(a);
  count_launch();
}
void launch_rel_attention(const float* qkv, const float* emb_k, const float* emb_v, const long long* lengths, float* out,
                          int B, int C, int T, int n_heads, int window, cudaStream_t s) {
  const int dk = C / n_heads;
  const int Tpad = (T + 3) & ~3;
  const size_t smem = sizeof(float) * ((size_t)dk * kAttQ * 2 + (size_t)dk * (kAttKT + 1) + (size_t)kAttQ * Tpad);
  static DynSmemAttr attr;
  if (attr.ensure((const void*)rel_attention_kernel, smem) != cudaSuccess) return;
  dim3 grid((T + kAttQ - 1) / kAttQ, n_heads, B);
  rel_attention_kernel<<<grid, kAttThreads, smem, s>>>(qkv, emb_k, emb_v, lengths, out, C, T, n_heads, window, dk, Tpad);
  count_launch();
}
void launch_convflow_pre(const float* z, int src_ch, const float* w, const float* bias, const float* cond, float* out,
                         int B, int C, int T, cudaStream_t s) {
  dim3 grid((T + 127) / 128, C, B);
  convflow_pre_kernel<<<grid, 128, 0, s>>>(z, src_ch, w, bias, cond, out, C, T);
  count_launch();
}
void launch_spline_flip(const float* zin, const float* u, int, float* zout, const long long* lengths, int B, int T,
                        float inv_sqrt_h, cudaStream_t s) {
  dim3 grid((T + 127) / 128, B);
  spline_flip_kernel<<<grid, 128, 0, s>>>(zin, u, zout, lengths, T, inv_sqrt_h);
  count_launch();
}
void launch_scale(const float* in, float* out, float scale, long long n, cudaStream_t s) {
  scale_kernel<<<(int)((n + 255) / 256), 256, 0, s>>>(in, out, scale, n);
  count_launch();
}
void launch_sdp_final(const float* z, const float* m, const float* logs, const long long* lengths, float* logw, int B,
                      int T, cudaStream_t s) {
  dim3 grid((T + 127) / 128, B);
  sdp_final_kernel<<<grid, 128, 0, s>>>(z, m, logs, lengths, logw, T);
  count_launch();
}
void launch_length_regulate(const float* logw, const long long* x_lengths, const float* durations, float length_scale,
                            int B, int Tx, float* w_ceil, int* cum, long long* y_lengths, cudaStream_t s) {
  length_regulate_kernel<<<B, 256, 0, s>>>(logw, x_lengths, durations, length_scale, Tx, w_ceil, cum, y_lengths);
  count_launch();
}
void launch_expand_prior(const float* m, const float* logs, const int* cum, const long long*, const long long* y_lengths,
                         const float* noise, long long noise_bs, long long noise_rs, float noise_scale, int B, int C,
                         int Tx, int Ty, float* m_p, float* logs_p, float* z_p, float* attn, float* y_mask,
                         cudaStream_t s) {
  dim3 grid((Ty + 127) / 128, B);
  expand_prior_kernel<<<grid, 128, 0, s>>>(m, logs, cum, y_lengths, noise, noise_bs, noise_rs, noise_scale, C, Tx, Ty,
                                           m_p, logs_p, z_p, attn, y_mask);
  count_launch();
}
void launch_max_i64(const long long* v, int n, long long* out, cudaStream_t s) {
  max_i64_kernel<<<1, 256, 0, s>>>(v, n, out);
  count_launch();
}
// ------------------------------------------------------------------ output stage (callers' int16 conversion)
// peak[b] (or peak[0] for the batch-global mode) = max |audio| over the valid samples; non-negative floats order
// like their bit patterns, so the reduction is an integer atomicMax.
__global__ void __launch_bounds__(256) audio_peak_kernel(const float* __restrict__ audio, const long long* __restrict__ lengths,
                                                         long long L, int global_peak, float* __restrict__ peak) {
  const int b = blockIdx.y;
  const long long n = lengths ? (lengths[b] < L ? lengths[b] : L) : L;
  const float* row = audio + (long long)b * L;
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(row[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float wm[8];
  if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 8) {
    m = wm[threadIdx.x];
    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffu, m, o));
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<int*>(peak + (global_peak ? 0 : b)), __float_as_int(m));
  }
}
// out = int16(trunc(clip(audio * gain, +-32767))); gain = 32767 (mode 0) or 32767 / max(0.01, peak) * 0.6
// (inference.py:101-105: the same fp32 operation order)
__global__ void __launch_bounds__(256) audio_to_int16_kernel(const float* __restrict__ audio, const float* __restrict__ peak,
                                                             long long L, int mode, short* __restrict__ out) {
  const int b = blockIdx.y;
  float g = 32767.0f;
  if (mode != 0) g = 32767.0f / fmaxf(peak[mode == 2 ? 0 : b], 0.01f) * 0.6f;
  const float* row = audio + (long long)b * L;
  short* orow = out + (long long)b * L;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (long long)gridDim.x * blockDim.x) {
    const float v = fminf(fmaxf(row[i] * g, -32767.0f), 32767.0f);
    orow[i] = (short)__float2int_rz(v);
  }
}
void launch_audio_to_int16(const float* audio, const long long* lengths, int B, long long L, int mode, float* peak,
                           short* out, cudaStream_t s) {
  const int gx = (int)((L + 256 * 8 - 1) / (256 * 8) > 1024 ? 1024 : (L + 256 * 8 - 1) / (256 * 8));
  dim3 grid(gx < 1 ? 1 : gx, B);
  if (mode != 0) {
    cudaMemsetAsync(peak, 0, sizeof(float) * (mode == 2 ? 1 : B), s);
    audio_peak_kernel<<<grid, 256, 0, s>>>(audio, lengths, L, mode == 2, peak);
    count_launch();
  }
  audio_to_int16_kernel<<<grid, 256, 0, s>>>(audio, peak, L, mode, out);
  count_launch();
}

void launch_transpose_blc(const float* in, float* out, int B, int L, int C, cudaStream_t s) {
  dim3 grid((L + 31) / 32, (C + 31) / 32, B);
  transpose_blc_kernel<<<grid, dim3(32, 8), 0, s>>>(in, out, L, C);
  count_launch();
}

void launch_reflect_pad_left(const float* in, long long in_bs, int in_cs, const long long* lengths, float* out, int B, int C,
                             int T, cudaStream_t s) {
  dim3 grid((T + 1 + 127) / 128, C, B);
  reflect_pad_left_kernel<<<grid, 128, 0, s>>>(in, in_bs, in_cs, lengths, out, C, T);
  count_launch();
}
void launch_gather_channels(const float* in, long long in_bs, int c0, int cstep, const long long* lengths, float* out,
                            float* out_masked, int B, int C, int T, cudaStream_t s) {
  dim3 grid((T + 127) / 128, C, B);
  gather_channels_kernel<<<grid, 128, 0, s>>>(in, in_bs, c0, cstep, lengths, out, out_masked, C, T);
  count_launch();
}
void launch_vocos_spec(float* x, int B, int K, int F, cudaStream_t s) {
  dim3 grid((F + 127) / 128, K, B);
  vocos_spec_kernel<<<grid, 128, 0, s>>>(x, K, F);
  count_launch();
}
void launch_idft_weight(float* w, int N, cudaStream_t s) {
  idft_weight_kernel<<<1024, 256, 0, s>>>(w, N);
  count_launch();
}
void launch_istft_overlap_add(const float* frames, float* out, int B, int N, int hop, int F, cudaStream_t s) {
  const long long L = (long long)hop * (F - 1);
  dim3 grid((unsigned)((L + 255) / 256), B);
  istft_overlap_add_kernel<<<grid, 256, 0, s>>>(frames, out, N, hop, F);
  count_launch();
}
void launch_scale_rows(const float* w, const float* bias, const float* sc, float* w_out, float* b_out, int rows, int cols,
                       cudaStream_t s) {
  scale_rows_kernel<<<256, 256, 0, s>>>(w, bias, sc, w_out, b_out, rows, cols);
  count_launch();
}

void launch_posterior_sample(const float* stats, const float* noise, const long long* lengths, float* z, float* m, float* logs,
                             float* y_mask, int B, int C, int T, cudaStream_t s) {
  dim3 grid((T + 127) / 128, C, B);
  posterior_sample_kernel<<<grid, 128, 0, s>>>(stats, noise, lengths, z, m, logs, y_mask, C, T);
  count_launch();
}
void launch_spec_frames(const float* audio, long long L, const long long* lengths, float* frames, int B, int N, int hop, int pad,
                        int F, cudaStream_t s) {
  dim3 grid((F + 127) / 128, N, B);
  spec_frames_kernel<<<grid, 128, 0, s>>>(audio, L, lengths, frames, N, hop, pad, F);
  count_launch();
}
void launch_dft_weight(float* w, int N, cudaStream_t s) {
  dft_weight_kernel<<<1024, 256, 0, s>>>(w, N);
  count_launch();
}
void launch_spec_magnitude(const float* dft, const long long* lengths, float* spec, long long* spec_lengths, int B, int K, int F,
                           int N, int hop, int pad, cudaStream_t s) {
  dim3 grid((F + 127) / 128, K, B);
  spec_magnitude_kernel<<<grid, 128, 0, s>>>(dft, lengths, spec, spec_lengths, K, F, N, hop, pad);
  count_launch();
}

}  // namespace wetts
