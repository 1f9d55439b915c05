// Host side of libwetts_b200: checkpoint ingestion, weight-norm folding, weight re-layout,
// launch orchestration for every block of the VITS inference path, and the C ABI
// declared in include/wetts_b200.h.  No CPU compute path exists here: every tensor
// operation is a CUDA kernel from conv_kernels.cu / misc_kernels.cu.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/wetts_b200.h"
#include "kernels.cuh"

namespace wetts {

static thread_local std::string g_err;

// Effective options of the call in progress on this host thread: the handle's own setting when it has one
// (wetts_vits_set_option), else the process-wide default (wetts_set_option).  Set by CHECK_READY.
struct CallOpts {
  bool tc = true, fused = true, len_aware = false;
  int fmt = 16;   // operand format of the tensor-pipe kernels: 32 = 3xTF32 (kind::tf32), 16 = f16 split (kind::f16)
  bool attn_tc = false;
};
static std::atomic<int> g_tensor_format{16};
static std::atomic<int> g_attn_tc{1};   // text-encoder attention on the tensor pipe (attn_tc.cu) for 64 <= Tx <= 128

// Host-visible fault word of the device-side soft watchdog (tc_prims.cuh mbar_wait): one mapped pinned word per
// process, installed on every device a handle is created on.
static std::atomic<unsigned int*> g_fault_word{nullptr};
static int ensure_fault_word(int device) {
  unsigned int* w = g_fault_word.load();
  if (!w) {
    unsigned int* fresh = nullptr;
    if (cudaHostAlloc((void**)&fresh, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return 1;
    *fresh = 0;
    unsigned int* expected = nullptr;
    if (g_fault_word.compare_exchange_strong(expected, fresh)) w = fresh;
    else { cudaFreeHost(fresh); w = expected; }
  }
  (void)device;
  unsigned int* dptr = nullptr;
  if (cudaHostGetDevicePointer((void**)&dptr, w, 0) != cudaSuccess) return 1;
  return tc_conv_install_fault_word(dptr) | tc16_conv_install_fault_word(dptr) | fused_rb_install_fault_word(dptr) |
         fused_mrf16_install_fault_word(dptr) | attn_tc_install_fault_word(dptr) | tc16p_install_fault_word(dptr) | tc16r_install_fault_word(dptr);
}
// nonzero (and the word cleared) if a device-side pipeline wait timed out since the last check
static unsigned int take_fault() {
  unsigned int* w = g_fault_word.load();
  if (!w) return 0;
  const unsigned int v = *(volatile unsigned int*)w;
  if (v) *(volatile unsigned int*)w = 0;
  return v;
}
static thread_local CallOpts g_call;

static int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}

static unsigned int take_fault();
#define CUDA_OK(expr)                                                                        \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return fail("%s failed: %s%s (%s:%d)", #expr, cudaGetErrorString(_e),                  \
                  take_fault() ? " -- device pipeline watchdog fired (an mbarrier wait timed out)" : "", __FILE__, __LINE__); \
  } while (0)

struct Raw {
  float* d = nullptr;
  std::vector<int64_t> dims;
  size_t numel() const {
    size_t n = 1;
    for (auto v : dims) n *= (size_t)v;
    return n;
  }
};

struct Conv {
  float* w = nullptr;    // SIMT layout [Cin][K][CoutPad]
  float* b = nullptr;
  float* wtc = nullptr;  // tcgen05 layout (tc_conv_kernel.cu), hi/lo tf32 split
  uint16_t* wtc16 = nullptr;  // tcgen05 layout of the f16 split (tc16_conv_kernel.cu)
  const float* wraw = nullptr;  // folded source weight [Cout][Cin][K] (before any channel map)
  TcPlan tc, tc16;
  int Cin = 0, Cout = 0, CoutPad = 0, K = 1;
};
struct ConvT {
  float* w = nullptr;
  float* b = nullptr;
  int Cin = 0, Cout = 0, CoutPad = 0, k = 0, u = 1, ntaps = 2, pad = 0;
  Conv as_conv;  // polyphase form as a Conv1d with Cout*u channels (tensor-core path)
};
struct Ln {
  float* g = nullptr;
  float* b = nullptr;
  int C = 0;
};
struct Dds {
  float* dww[3];
  float* dwb[3];
  Conv c1x1[3];
  Ln n1[3], n2[3];
};

static int round_cout(int c) { return (c % 64 == 0) ? c : ((c + 31) / 32) * 32; }

// bump allocator over the caller's workspace
struct Arena {
  char* base;
  size_t cap, off = 0;
  bool dry;  // size query only
  Arena(void* p, size_t c) : base((char*)p), cap(c), dry(p == nullptr) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T* r = dry ? nullptr : (T*)(base + off);
    off += n * sizeof(T);
    return r;
  }
  bool ok() const { return dry || off <= cap; }
};

}  // namespace wetts

using namespace wetts;

struct wetts_vits_s {
  wetts_vits_config cfg;
  int device = 0;
  bool finalized = false;
  std::map<std::string, Raw> raw;
  std::vector<void*> owned;
  // per-handle options: -1 = follow the process-wide option (wetts_set_option)
  int opt_tc = -1, opt_fused = -1, opt_len_aware = 0, opt_fmt = -1, opt_attn_tc = -1;
  unsigned long long launches_at_create = 0;
  int U = 1;

  // text encoder
  float* emb = nullptr;
  struct EncLayer {
    Conv qkv, o, ffn1, ffn2;
    float *rel_k = nullptr, *rel_v = nullptr;
    Ln ln1, ln2;
  };
  std::vector<EncLayer> enc;
  Conv proj_m, proj_logs;
  // deterministic duration predictor
  Conv dp_cond, dp_c1, dp_c2, dp_proj;
  Ln dp_n1, dp_n2;
  // stochastic duration predictor
  Conv sdp_pre, sdp_proj, sdp_cond;
  Dds sdp_dds;
  struct ConvFlow {
    float *pre_w = nullptr, *pre_b = nullptr;
    Dds dds;
    Conv proj;
  } cf[3];  // flows 7, 5, 3 in application order
  float *ea_m = nullptr, *ea_logs = nullptr;
  // flow
  struct PlainEncLayer {   // attentions.Encoder layer with window_size=None (VITS2 pre_transformer)
    Conv qkv, o, ffn1, ffn2;
    Ln ln1, ln2;
  };
  struct Coupling {
    Conv pre, post, cond, in[4], rs[4];
    bool flipped = false;
    PlainEncLayer tf[2];   // flow_type 1 only
  } flow[4];  // application order: reference layers 6, 4, 2, 0
  // posterior encoder (enc_q, models.py:124-132; encoders.py:60-99): packed only when the checkpoint carries every key
  static constexpr int kPostLayers = 16;
  struct Posterior {
    Conv pre, cond, proj, in[kPostLayers], rs[kPostLayers];
    int S = 0;   // feature channels of enc_q.pre: filter_length / 2 + 1 (linear spectrogram) or n_mel_channels
  } post;
  bool has_post = false;
  std::string post_missing;   // first missing enc_q key when !has_post
  // linear spectrogram (mel_processing.py:42-93 with center=False): windowed real DFT as a constant 1x1 conv
  Conv spec_dft;
  int spec_nfft = 0;   // 0: the feature dimension is not n_fft/2 + 1 of a power-of-two n_fft (no spectrogram)
  // Vocos generator (vocoder_type 1)
  struct ConvNext {
    float *dww = nullptr, *dwb = nullptr;
    Ln norm;
    Conv pw1, pw2;   // pw2 carries the layer scale
  };
  Conv voc_in, voc_cond, voc_out, voc_idft;
  Ln voc_norm_pre, voc_norm_post;
  std::vector<ConvNext> voc_layers;
  // generator
  Conv conv_pre, dec_cond;
  std::vector<ConvT> ups;
  struct ResBlock {
    std::vector<Conv> c1, c2;  // type 2 uses c1 only
    std::vector<int> dil;
    int k = 3;
  };
  std::vector<ResBlock> rbs;
  std::vector<float*> fused_rb_w;  // per stage: packed weights of the fused MRF kernel (nullptr: per-layer path)
  std::vector<void*> fused16_w;    // per stage: packed f16-split weights of fused_mrf16_kernel (nullptr: not eligible)
  float* conv_post_w = nullptr;
  int c_last = 0;
  float* emb_g = nullptr;

  // ---------------------------------------------------------------- helpers
  template <typename T>
  int dalloc(T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T) + 16);
    if (e != cudaSuccess) return fail("cudaMalloc(%zu) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    owned.push_back(q);
    *p = (T*)q;
    return 0;
  }
  const Raw* find(const std::string& k) const {
    auto it = raw.find(k);
    return it == raw.end() ? nullptr : &it->second;
  }
  int need(const std::string& k, const Raw** out) const {
    *out = find(k);
    if (!*out) return fail("missing checkpoint tensor '%s'", k.c_str());
    return 0;
  }
  // plain weight for `prefix` (folds weight_g/weight_v when that is what the checkpoint has)
  int folded_weight(const std::string& prefix, Raw* out) {
    if (const Raw* w = find(prefix + ".weight")) {
      *out = *w;
      return 0;
    }
    const Raw *g, *v;
    if (need(prefix + ".weight_g", &g) || need(prefix + ".weight_v", &v)) return 1;
    const int rows = (int)v->dims[0];
    const int cols = (int)(v->numel() / rows);
    if ((int)g->numel() != rows) return fail("%s.weight_g has %zu elements, expected %d", prefix.c_str(), g->numel(), rows);
    float* f;
    if (dalloc(&f, v->numel())) return 1;
    launch_weight_norm_fold(v->d, g->d, f, rows, cols, 0);
    out->d = f;
    out->dims = v->dims;
    return 0;
  }
  int upload_ints(const std::vector<int>& h, int** d) {
    if (dalloc(d, h.size())) return 1;
    CUDA_OK(cudaMemcpy(*d, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice));
    return 0;
  }
  // Conv1d weight [Cout][Cin][K] -> packed [Cin'][K][CoutPad]; co_map: packed out channel -> source
  // out channel (empty: identity); ci_map: packed in channel -> source in channel (empty: identity)
  int pack_conv_from(const Raw& w, const float* bias_src, std::vector<int> co_map, const std::vector<int>& ci_map,
                     Conv* c, int tc_dil = 1) {
    if (w.dims.size() != 3) return fail("conv weight must be 3-D");
    const int src_cout = (int)w.dims[0], src_cin = (int)w.dims[1], K = (int)w.dims[2];
    if (co_map.empty()) {
      co_map.resize(src_cout);
      for (int i = 0; i < src_cout; ++i) co_map[i] = i;
    }
    c->Cout = (int)co_map.size();
    c->CoutPad = round_cout(c->Cout);
    c->Cin = ci_map.empty() ? src_cin : (int)ci_map.size();
    c->K = K;
    c->wraw = w.d;
    co_map.resize(c->CoutPad, -1);
    int *d_co = nullptr, *d_ci = nullptr;
    if (upload_ints(co_map, &d_co)) return 1;
    if (!ci_map.empty() && upload_ints(ci_map, &d_ci)) return 1;
    if (dalloc(&c->w, (size_t)c->Cin * K * c->CoutPad)) return 1;
    launch_pack_conv(w.d, c->w, d_co, d_ci, c->Cin, K, c->CoutPad, src_cin, 0);
    c->b = nullptr;
    if (bias_src) {
      if (dalloc(&c->b, (size_t)c->CoutPad)) return 1;
      launch_gather_vec(bias_src, c->b, d_co, c->CoutPad, 0);
    }
    c->wtc = nullptr;
    if (tc_dil > 0 && tc_conv_plan(c->Cin, c->Cout, K, tc_dil, &c->tc)) {
      if (getenv("WETTS_DEBUG_PLAN"))
        fprintf(stderr, "[tc plan] Cin=%d Cout=%d K=%d dil=%d -> mode=%d N=%d n_tiles=%d KC=%d chunks=%d MB=%d G=%d abuf=%d bbuf=%d smem=%zu\n",
                c->Cin, c->Cout, K, tc_dil, c->tc.mode, c->tc.N, c->tc.n_tiles, c->tc.KC, c->tc.n_chunks, c->tc.MB, c->tc.G,
                c->tc.n_abuf, c->tc.n_bbuf, tc_conv_smem_bytes(K, tc_dil, c->tc.N, c->tc.KC, c->tc.MB, c->tc.n_abuf, c->tc.n_bbuf));
      if (dalloc(&c->wtc, c->tc.packed_floats)) return 1;
      launch_pack_conv_tc(w.d, c->wtc, d_co, d_ci, c->Cout, c->Cin, K, src_cin, c->tc, 0);
    }
    c->wtc16 = nullptr;
    if (tc_dil > 0 && tc16_conv_plan(c->Cin, c->Cout, K, tc_dil, &c->tc16)) {
      if (getenv("WETTS_DEBUG_PLAN"))
        fprintf(stderr, "[tc16 plan] Cin=%d Cout=%d K=%d dil=%d -> mode=%d N=%d n_tiles=%d KC=%d chunks=%d MB=%d G=%d abuf=%d bbuf=%d smem=%zu\n",
                c->Cin, c->Cout, K, tc_dil, c->tc16.mode, c->tc16.N, c->tc16.n_tiles, c->tc16.KC, c->tc16.n_chunks, c->tc16.MB,
                c->tc16.G, c->tc16.n_abuf, c->tc16.n_bbuf,
                tc16_conv_smem_bytes(K, tc_dil, c->tc16.N, c->tc16.KC, c->tc16.MB, c->tc16.n_abuf, c->tc16.n_bbuf));
      if (dalloc(&c->wtc16, c->tc16.packed_floats + 64)) return 1;
      launch_pack_conv_tc16(w.d, c->wtc16, d_co, d_ci, c->Cout, c->Cin, K, src_cin, c->tc16, 0);
    }
    return 0;
  }
  int make_conv(const std::string& prefix, Conv* c, bool bias = true, std::vector<int> co_map = {},
                const std::vector<int>& ci_map = {}, int tc_dil = 1) {
    Raw w;
    if (folded_weight(prefix, &w)) return 1;
    const float* bsrc = nullptr;
    if (bias) {
      const Raw* b;
      if (need(prefix + ".bias", &b)) return 1;
      bsrc = b->d;
    }
    return pack_conv_from(w, bsrc, co_map, ci_map, c, tc_dil);
  }
  int make_ln(const std::string& prefix, Ln* l) {
    const Raw *g, *b;
    if (need(prefix + ".gamma", &g) || need(prefix + ".beta", &b)) return 1;
    l->g = g->d;
    l->b = b->d;
    l->C = (int)g->numel();
    if (l->C > 512) return fail("LayerNorm over %d channels not supported (max 512)", l->C);
    return 0;
  }
  int make_dds(const std::string& prefix, Dds* d) {
    for (int i = 0; i < 3; ++i) {
      const Raw *w, *b;
      const std::string p = prefix + ".convs_sep." + std::to_string(i);
      if (need(p + ".weight", &w) || need(p + ".bias", &b)) return 1;
      if (w->dims.size() != 3 || w->dims[2] != 3) return fail("%s: depthwise kernel size must be 3", p.c_str());
      d->dww[i] = w->d;
      d->dwb[i] = b->d;
      if (make_conv(prefix + ".convs_1x1." + std::to_string(i), &d->c1x1[i])) return 1;
      if (make_ln(prefix + ".norms_1." + std::to_string(i), &d->n1[i])) return 1;
      if (make_ln(prefix + ".norms_2." + std::to_string(i), &d->n2[i])) return 1;
    }
    return 0;
  }
};

// ================================================================== block launch helpers
namespace wetts {

static ConvArgs conv_args(const Conv& c, const float* in, long long in_bs, int in_cs, int B, int T, int dil = 1) {
  ConvArgs a;
  a.wtc = c.wtc;
  a.tc = c.tc;
  a.wtc16 = c.wtc16;
  a.tc16 = c.tc16;
  a.fmt = g_call.fmt;
  a.in = in;
  a.in_bs = in_bs;
  a.in_cs = in_cs;
  a.w = c.w;
  a.bias = c.b;
  a.B = B;
  a.Cin = c.Cin;
  a.Cout = c.Cout;
  a.CoutPad = c.CoutPad;
  a.T = T;
  a.K = c.K;
  a.dil = dil;
  a.pad_left = (c.K - 1) * dil / 2;
  a.ep.out_bs = (long long)c.Cout * T;
  a.use_tc = g_call.tc ? 1 : 0;
  return a;
}

// per-(b, co) vector from g: out[b][co] = W g[b] + bias   (a Conv1d over T == 1)
static void cond_vector(const Conv& c, const float* g, int B, float* out, cudaStream_t s) {
  if (c.K == 1 && c.Cin * 16 * sizeof(float) <= 48 * 1024) {
    launch_cond_vector(g, c.w, c.b, out, B, c.Cin, c.Cout, c.CoutPad, s);
    return;
  }
  ConvArgs a = conv_args(c, g, c.Cin, 1, B, 1);
  a.ep.out = out;
  a.ep.out_bs = c.Cout;
  launch_conv1d(a, s);
}

static void run_dds(const Dds& d, float* x, float* y, float* y2, const long long* lengths, int B, int C, int T,
                    cudaStream_t s) {
  // duration_predictors.py:45-57 (the caller applies the trailing `* x_mask` through in_mask of the next conv)
  int dil = 1;
  for (int i = 0; i < 3; ++i) {
    LnArgs l;
    l.a = x;
    l.dww = d.dww[i];
    l.dwb = d.dwb[i];
    l.dil = dil;
    l.gamma = d.n1[i].g;
    l.beta = d.n1[i].b;
    l.act = 1;
    l.out = y;
    l.lengths = lengths;
    l.B = B;
    l.C = C;
    l.T = T;
    launch_layernorm(l, s);
    ConvArgs a = conv_args(d.c1x1[i], y, (long long)C * T, T, B, T);
    a.ep.out = y2;
    launch_conv1d(a, s);
    LnArgs l2;
    l2.a = y2;
    l2.gamma = d.n2[i].g;
    l2.beta = d.n2[i].b;
    l2.act = 1;
    l2.res = x;
    l2.out = x;
    l2.B = B;
    l2.C = C;
    l2.T = T;
    launch_layernorm(l2, s);
    dil *= 3;
  }
}

// WN (modules.py:60-87) on the gated / res-skip epilogues: x [B][H][T] is the residual stream (updated in place and
// masked), skip [B][H][T] receives the unmasked sum of the skip outputs (the caller masks it through the next conv's
// in_mask).  gc: per-utterance cond vectors [B][2*H*n_layers] of the layer's cond_layer, or nullptr.
static void run_wn(const Conv* in, const Conv* rs, int n_layers, float* x, float* acts, float* skip, const float* gc,
                   const long long* len, int B, int H, int T, cudaStream_t s) {
  for (int i = 0; i < n_layers; ++i) {
    ConvArgs a = conv_args(in[i], x, (long long)H * T, T, B, T);
    a.ep.mode = EPI_GATE; a.ep.H = H; a.ep.out = acts; a.ep.out_bs = (long long)H * T;
    if (gc) { a.ep.cond = gc; a.ep.cond_bs = 2 * H * n_layers; a.ep.cond_off = 2 * H * i; }
    launch_conv1d(a, s);
    a = conv_args(rs[i], acts, (long long)H * T, T, B, T);
    a.lengths = len;
    a.ep.mode = EPI_RES_SKIP; a.ep.H = H; a.ep.x = x; a.ep.skip = skip; a.ep.out_bs = (long long)H * T;
    a.ep.skip_init = (i == 0); a.ep.last = (i == n_layers - 1);
    launch_conv1d(a, s);
  }
}

}  // namespace wetts

// ================================================================== C ABI
extern "C" {

const char* wetts_last_error(void) { return g_err.c_str(); }
const char* wetts_version(void) { return "wetts_b200 0.1 (sm_100a, fp32 SIMT path)"; }

int wetts_vits_create(const wetts_vits_config* cfg, int device, wetts_vits_t* out) {
  if (!cfg || !out) return fail("null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("no CUDA device: wetts_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail("device %d out of range (have %d)", device, ndev);
  CUDA_OK(cudaSetDevice(device));
  const wetts_vits_config& c = *cfg;
  if (c.hidden_channels % c.n_heads) return fail("hidden_channels %% n_heads != 0");
  if (c.hidden_channels / c.n_heads > 96) return fail("head dim %d > 96 not supported", c.hidden_channels / c.n_heads);
  if (c.hidden_channels > 256 || c.inter_channels % 2) return fail("unsupported channel configuration");
  if (c.vocoder_type != 0 && c.vocoder_type != 1) return fail("vocoder_type must be 0 (HiFi-GAN) or 1 (Vocos)");
  if (c.flow_type != 0 && c.flow_type != 1) return fail("flow_type must be 0 or 1 ('pre_conv')");
  if (c.vocoder_type == 1) {
    if (c.vocos_channels < 16 || c.vocos_channels > 512) return fail("vocos_channels must be in [16, 512]");
    if (c.vocos_n_fft < 16 || (c.vocos_n_fft & (c.vocos_n_fft - 1)) || c.vocos_out_channels != c.vocos_n_fft + 2)
      return fail("Vocos: n_fft must be a power of two and out_channels = n_fft + 2");
    if (c.vocos_hop_length < 1 || c.vocos_n_fft % c.vocos_hop_length) return fail("Vocos: hop_length must divide n_fft");
    if (c.vocos_num_layers < 1 || c.vocos_h_channels < 16) return fail("bad Vocos layer configuration");
  }
  int U = 1;
  if (c.vocoder_type == 1) {
    U = c.vocos_hop_length;
  } else {
    if (c.n_upsamples < 1 || c.n_upsamples > WETTS_MAX_UPSAMPLES) return fail("bad n_upsamples");
    if (c.n_resblock_kernels < 1 || c.n_resblock_kernels > WETTS_MAX_RESBLOCK_KERNELS) return fail("bad n_resblock_kernels");
    if (c.resblock_type != 1 && c.resblock_type != 2) return fail("resblock_type must be 1 or 2");
    for (int i = 0; i < c.n_upsamples; ++i) {
      const int u = c.upsample_rates[i], k = c.upsample_kernel_sizes[i];
      if (u < 1 || 32 % u) return fail("upsample rate %d must divide 32", u);
      if (k % u || (k - u) % 2) return fail("upsample kernel %d incompatible with rate %d", k, u);
      U *= u;
    }
    for (int j = 0; j < c.n_resblock_kernels; ++j) {
      if (c.resblock_kernel_sizes[j] % 2 == 0) return fail("resblock kernel sizes must be odd");
      if (c.resblock_n_dilations[j] < 1 || c.resblock_n_dilations[j] > WETTS_MAX_DILATIONS) return fail("bad dilation count");
    }
  }
  if (c.kernel_size % 2 == 0) return fail("FFN kernel_size must be odd");
  wetts_vits_s* h = new wetts_vits_s();
  h->cfg = c;
  h->device = device;
  h->U = U;
  h->launches_at_create = kernel_launch_counter();
  if (ensure_fault_word(device)) {
    delete h;
    return fail("could not install the watchdog fault word");
  }
  *out = h;
  return 0;
}

void wetts_vits_destroy(wetts_vits_t h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (void* p : h->owned) cudaFree(p);
  for (auto& kv : h->raw) cudaFree(kv.second.d);
  delete h;
}

int wetts_vits_upsample_factor(wetts_vits_t h) { return h ? h->U : 0; }

int wetts_set_option(const char* name, int value) {
  if (!name) return fail("null option name");
  if (!strcmp(name, "fused_resblock")) {
    set_fused_resblock_enabled(value != 0);
    return 0;
  }
  if (!strcmp(name, "tensor_cores")) {
    set_tensor_cores_enabled(value != 0);
    return 0;
  }
  if (!strcmp(name, "tensor_format")) {
    if (value != 16 && value != 32) return fail("tensor_format must be 16 (f16 split) or 32 (3xTF32)");
    g_tensor_format.store(value);
    return 0;
  }
  if (!strcmp(name, "attention_tensor_cores")) {
    g_attn_tc.store(value != 0);
    return 0;
  }
  if (!strcmp(name, "mrf_item_rows")) {
    if (set_mrf16_item_rows(value)) return fail("mrf_item_rows must be 0 (policy), 128, 256 or 384");
    return 0;
  }
  return fail("unknown option '%s'", name);
}
int wetts_get_option(const char* name, int* value) {
  if (!name || !value) return fail("null argument");
  if (!strcmp(name, "tensor_cores")) {
    *value = tensor_cores_enabled() ? 1 : 0;
    return 0;
  }
  if (!strcmp(name, "fused_resblock")) {
    *value = fused_resblock_enabled() ? 1 : 0;
    return 0;
  }
  if (!strcmp(name, "tensor_format")) {
    *value = g_tensor_format.load();
    return 0;
  }
  if (!strcmp(name, "attention_tensor_cores")) {
    *value = g_attn_tc.load();
    return 0;
  }
  if (!strcmp(name, "mrf_item_rows")) {
    *value = mrf16_item_rows_option();
    return 0;
  }
  if (!strcmp(name, "mrf_item_rows_last")) {
    *value = mrf16_last_item_rows();
    return 0;
  }
  return fail("unknown option '%s'", name);
}
int wetts_vits_set_option(wetts_vits_t h, const char* name, int value) {
  if (!h || !name) return fail("null argument");
  if (!strcmp(name, "tensor_cores")) h->opt_tc = value < 0 ? -1 : (value != 0);
  else if (!strcmp(name, "fused_resblock")) h->opt_fused = value < 0 ? -1 : (value != 0);
  else if (!strcmp(name, "length_aware")) h->opt_len_aware = value != 0;
  else if (!strcmp(name, "tensor_format")) {
    if (value != 16 && value != 32 && value >= 0) return fail("tensor_format must be 16, 32 or -1 (process default)");
    h->opt_fmt = value;
  } else if (!strcmp(name, "attention_tensor_cores")) h->opt_attn_tc = value < 0 ? -1 : (value != 0);
  else return fail("unknown option '%s'", name);
  return 0;
}
int wetts_vits_get_option(wetts_vits_t h, const char* name, int* value) {
  if (!h || !name || !value) return fail("null argument");
  if (!strcmp(name, "tensor_cores")) *value = h->opt_tc >= 0 ? h->opt_tc : (tensor_cores_enabled() ? 1 : 0);
  else if (!strcmp(name, "fused_resblock")) *value = h->opt_fused >= 0 ? h->opt_fused : (fused_resblock_enabled() ? 1 : 0);
  else if (!strcmp(name, "length_aware")) *value = h->opt_len_aware;
  else if (!strcmp(name, "tensor_format")) *value = h->opt_fmt > 0 ? h->opt_fmt : g_tensor_format.load();
  else if (!strcmp(name, "attention_tensor_cores")) *value = h->opt_attn_tc >= 0 ? h->opt_attn_tc : g_attn_tc.load();
  else return fail("unknown option '%s'", name);
  return 0;
}
int wetts_audio_to_int16(const float* audio, const int64_t* lengths, int B, int64_t L, int mode, float* peak_scratch,
                         int16_t* out, void* stream) {
  if (!audio || !out || B <= 0 || L <= 0) return fail("wetts_audio_to_int16: empty input");
  if (mode < 0 || mode > 2) return fail("wetts_audio_to_int16: unknown mode %d", mode);
  if (mode != 0 && !peak_scratch) return fail("wetts_audio_to_int16: the peak modes need a float[B] scratch buffer");
  launch_audio_to_int16(audio, (const long long*)lengths, B, (long long)L, mode, peak_scratch, (short*)out,
                        (cudaStream_t)stream);
  CUDA_OK(cudaGetLastError());
  return 0;
}

int wetts_vits_check_fault(wetts_vits_t h, void* stream, int synchronize) {
  if (!h) return fail("null handle");
  CUDA_OK(cudaSetDevice(h->device));
  if (synchronize) CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  CUDA_OK(cudaGetLastError());
  if (take_fault()) return fail("device pipeline watchdog fired (an mbarrier wait timed out)");
  return 0;
}

uint64_t wetts_vits_launch_count(wetts_vits_t h) { return h ? kernel_launch_counter() - h->launches_at_create : 0; }

int wetts_vits_set_tensor(wetts_vits_t h, const char* name, const void* data, const int64_t* dims, int ndim) {
  if (!h || !name || !data || (!dims && ndim > 0)) return fail("null argument");
  if (h->finalized) return fail("handle is finalized (immutable)");
  CUDA_OK(cudaSetDevice(h->device));
  Raw r;
  r.dims.assign(dims, dims + ndim);
  for (auto d : r.dims)
    if (d <= 0) return fail("tensor '%s' has a non-positive dimension", name);
  const size_t n = r.numel();
  CUDA_OK(cudaMalloc((void**)&r.d, n * sizeof(float) + 16));
  cudaError_t e = cudaMemcpy(r.d, data, n * sizeof(float), cudaMemcpyDefault);
  if (e != cudaSuccess) {
    cudaFree(r.d);
    return fail("copy of '%s' failed: %s", name, cudaGetErrorString(e));
  }
  auto it = h->raw.find(name);
  if (it != h->raw.end()) cudaFree(it->second.d);
  h->raw[name] = r;
  return 0;
}

int wetts_vits_finalize(wetts_vits_t h) {
  if (!h) return fail("null handle");
  if (h->finalized) return 0;
  CUDA_OK(cudaSetDevice(h->device));
  const wetts_vits_config& c = h->cfg;
  const int H = c.hidden_channels, Cc = c.inter_channels, half = Cc / 2, gin = c.gin_channels;
  const Raw* r;
  // ---- text encoder
  if (h->need("enc_p.emb.weight", &r)) return 1;
  if (r->dims.size() != 2 || r->dims[0] != c.n_vocab || r->dims[1] != H)
    return fail("enc_p.emb.weight has shape [%lld,%lld], config says [%d,%d]", (long long)r->dims[0],
                (long long)(r->dims.size() > 1 ? r->dims[1] : 0), c.n_vocab, H);
  h->emb = r->d;
  h->enc.resize(c.n_layers);
  for (int i = 0; i < c.n_layers; ++i) {
    auto& L = h->enc[i];
    const std::string a = "enc_p.encoder.attn_layers." + std::to_string(i);
    // q, k, v fused into one 1x1 conv with 3H output channels
    Raw wq, wk, wv;
    if (h->folded_weight(a + ".conv_q", &wq) || h->folded_weight(a + ".conv_k", &wk) || h->folded_weight(a + ".conv_v", &wv))
      return 1;
    const Raw *bq, *bk, *bv;
    if (h->need(a + ".conv_q.bias", &bq) || h->need(a + ".conv_k.bias", &bk) || h->need(a + ".conv_v.bias", &bv)) return 1;
    Raw cat;
    cat.dims = {3 * H, H, 1};
    float* catb;
    if (h->dalloc(&cat.d, (size_t)3 * H * H) || h->dalloc(&catb, (size_t)3 * H)) return 1;
    const Raw* ws[3] = {&wq, &wk, &wv};
    const Raw* bs[3] = {bq, bk, bv};
    for (int j = 0; j < 3; ++j) {
      if ((int)ws[j]->numel() != H * H) return fail("%s: unexpected q/k/v weight size", a.c_str());
      CUDA_OK(cudaMemcpy(cat.d + (size_t)j * H * H, ws[j]->d, sizeof(float) * H * H, cudaMemcpyDeviceToDevice));
      CUDA_OK(cudaMemcpy(catb + (size_t)j * H, bs[j]->d, sizeof(float) * H, cudaMemcpyDeviceToDevice));
    }
    if (h->pack_conv_from(cat, catb, {}, {}, &L.qkv)) return 1;
    if (h->make_conv(a + ".conv_o", &L.o)) return 1;
    if (h->need(a + ".emb_rel_k", &r)) return 1;
    if (r->dims.size() != 3 || r->dims[0] != 1 || r->dims[1] != 9 || r->dims[2] != H / c.n_heads)
      return fail("%s.emb_rel_k: only shared-head window-4 tables are supported", a.c_str());
    L.rel_k = r->d;
    if (h->need(a + ".emb_rel_v", &r)) return 1;
    L.rel_v = r->d;
    if (h->make_ln("enc_p.encoder.norm_layers_1." + std::to_string(i), &L.ln1)) return 1;
    if (h->make_ln("enc_p.encoder.norm_layers_2." + std::to_string(i), &L.ln2)) return 1;
    if (h->make_conv("enc_p.encoder.ffn_layers." + std::to_string(i) + ".conv_1", &L.ffn1)) return 1;
    if (h->make_conv("enc_p.encoder.ffn_layers." + std::to_string(i) + ".conv_2", &L.ffn2)) return 1;
  }
  {
    std::vector<int> lo(Cc), hi(Cc);
    for (int i = 0; i < Cc; ++i) { lo[i] = i; hi[i] = Cc + i; }
    if (h->make_conv("enc_p.proj", &h->proj_m, true, lo) || h->make_conv("enc_p.proj", &h->proj_logs, true, hi)) return 1;
  }
  // ---- duration predictor
  if (c.use_sdp) {
    if (h->make_conv("dp.pre", &h->sdp_pre) || h->make_conv("dp.proj", &h->sdp_proj)) return 1;
    if (gin && h->make_conv("dp.cond", &h->sdp_cond)) return 1;
    if (h->make_dds("dp.convs", &h->sdp_dds)) return 1;
    const int order[3] = {7, 5, 3};
    for (int j = 0; j < 3; ++j) {
      const std::string p = "dp.flows." + std::to_string(order[j]);
      const Raw *pw, *pb;
      if (h->need(p + ".pre.weight", &pw) || h->need(p + ".pre.bias", &pb)) return 1;
      h->cf[j].pre_w = pw->d;
      h->cf[j].pre_b = pb->d;
      if (h->make_dds(p + ".convs", &h->cf[j].dds)) return 1;
      if (h->make_conv(p + ".proj", &h->cf[j].proj)) return 1;
      if (h->cf[j].proj.Cout != 29) return fail("%s.proj must have 29 output channels (10 bins)", p.c_str());
    }
    const Raw *m, *ls;
    if (h->need("dp.flows.0.m", &m) || h->need("dp.flows.0.logs", &ls)) return 1;
    h->ea_m = m->d;
    h->ea_logs = ls->d;
  } else {
    if (gin && h->make_conv("dp.cond", &h->dp_cond)) return 1;
    if (h->make_conv("dp.conv_1", &h->dp_c1) || h->make_conv("dp.conv_2", &h->dp_c2) || h->make_conv("dp.proj", &h->dp_proj))
      return 1;
    if (h->make_ln("dp.norm_1", &h->dp_n1) || h->make_ln("dp.norm_2", &h->dp_n2)) return 1;
  }
  // ---- flow (application order 6,4,2,0; odd number of preceding Flips => channels reversed)
  {
    const int order[4] = {6, 4, 2, 0};
    std::vector<int> gate(2 * H);
    for (int p = 0; p < 2 * H; ++p) gate[p] = (p & 1) ? H + (p >> 1) : (p >> 1);
    for (int j = 0; j < 4; ++j) {
      auto& F = h->flow[j];
      F.flipped = (j % 2 == 0);
      const std::string p = "flow.flows." + std::to_string(order[j]);
      std::vector<int> ci;
      if (F.flipped) {
        ci.resize(half);
        for (int q = 0; q < half; ++q) ci[q] = half - 1 - q;
      }
      if (c.flow_type == 1) {
        // VITS2 'pre_conv' coupling layer: x0 is materialised in the layer's own channel order (gather kernel), so the
        // pre_transformer and `pre` take it unpermuted
        ci.clear();
        for (int i = 0; i < 2; ++i) {
          auto& L = F.tf[i];
          const std::string a = p + ".pre_transformer.attn_layers." + std::to_string(i);
          Raw wq, wk, wv;
          if (h->folded_weight(a + ".conv_q", &wq) || h->folded_weight(a + ".conv_k", &wk) || h->folded_weight(a + ".conv_v", &wv))
            return 1;
          const Raw *bq, *bk, *bv;
          if (h->need(a + ".conv_q.bias", &bq) || h->need(a + ".conv_k.bias", &bk) || h->need(a + ".conv_v.bias", &bv)) return 1;
          Raw cat;
          cat.dims = {3 * half, half, 1};
          float* catb;
          if (h->dalloc(&cat.d, (size_t)3 * half * half) || h->dalloc(&catb, (size_t)3 * half)) return 1;
          const Raw* ws[3] = {&wq, &wk, &wv};
          const Raw* bs[3] = {bq, bk, bv};
          for (int q = 0; q < 3; ++q) {
            if ((int)ws[q]->numel() != half * half) return fail("%s: unexpected q/k/v weight size", a.c_str());
            CUDA_OK(cudaMemcpy(cat.d + (size_t)q * half * half, ws[q]->d, sizeof(float) * half * half, cudaMemcpyDeviceToDevice));
            CUDA_OK(cudaMemcpy(catb + (size_t)q * half, bs[q]->d, sizeof(float) * half, cudaMemcpyDeviceToDevice));
          }
          if (h->pack_conv_from(cat, catb, {}, {}, &L.qkv)) return 1;
          if (h->make_conv(a + ".conv_o", &L.o)) return 1;
          if (h->make_ln(p + ".pre_transformer.norm_layers_1." + std::to_string(i), &L.ln1)) return 1;
          if (h->make_ln(p + ".pre_transformer.norm_layers_2." + std::to_string(i), &L.ln2)) return 1;
          if (h->make_conv(p + ".pre_transformer.ffn_layers." + std::to_string(i) + ".conv_1", &L.ffn1)) return 1;
          if (h->make_conv(p + ".pre_transformer.ffn_layers." + std::to_string(i) + ".conv_2", &L.ffn2)) return 1;
          if (L.ffn1.K != 3 || L.ffn2.K != 3) return fail("%s: FFN kernel size must be 3", p.c_str());
        }
      }
      if (h->make_conv(p + ".pre", &F.pre, true, {}, ci)) return 1;
      if (h->make_conv(p + ".post", &F.post)) return 1;
      if (F.post.Cout != half) return fail("%s.post: only mean_only couplings are supported", p.c_str());
      if (gin && h->make_conv(p + ".enc.cond_layer", &F.cond)) return 1;
      for (int i = 0; i < 4; ++i) {
        if (h->make_conv(p + ".enc.in_layers." + std::to_string(i), &F.in[i], true, gate)) return 1;
        if (F.in[i].K != 5) return fail("%s: WN kernel size must be 5", p.c_str());
        if (h->make_conv(p + ".enc.res_skip_layers." + std::to_string(i), &F.rs[i])) return 1;
      }
    }
  }
  // ---- Vocos generator (decoders.py:250-307)
  if (c.vocoder_type == 1) {
    const int vc = c.vocos_channels;
    if (h->make_conv("dec.in_conv", &h->voc_in)) return 1;
    if (gin && h->make_conv("dec.cond", &h->voc_cond)) return 1;
    if (h->make_ln("dec.norm_pre", &h->voc_norm_pre) || h->make_ln("dec.norm_post", &h->voc_norm_post)) return 1;
    h->voc_layers.resize(c.vocos_num_layers);
    for (int i = 0; i < c.vocos_num_layers; ++i) {
      auto& L = h->voc_layers[i];
      const std::string p = "dec.layers." + std::to_string(i);
      const Raw *w, *b, *sc;
      if (h->need(p + ".dw_conv.weight", &w) || h->need(p + ".dw_conv.bias", &b)) return 1;
      if (w->dims.size() != 3 || w->dims[0] != vc || w->dims[1] != 1 || w->dims[2] != 3)
        return fail("%s.dw_conv: expected a depthwise kernel [%d,1,3]", p.c_str(), vc);
      L.dww = w->d;
      L.dwb = b->d;
      if (h->make_ln(p + ".norm", &L.norm) || h->make_conv(p + ".pw_conv1", &L.pw1)) return 1;
      // x = res + scale * pw_conv2(.): the layer scale is folded into pw_conv2's rows
      Raw w2;
      const Raw* b2;
      if (h->folded_weight(p + ".pw_conv2", &w2) || h->need(p + ".pw_conv2.bias", &b2) || h->need(p + ".scale", &sc)) return 1;
      if ((int)sc->numel() != vc || (int)w2.dims[0] != vc) return fail("%s.scale: unexpected shape", p.c_str());
      Raw ws;
      ws.dims = w2.dims;
      float* bsc;
      if (h->dalloc(&ws.d, w2.numel()) || h->dalloc(&bsc, (size_t)vc)) return 1;
      launch_scale_rows(w2.d, b2->d, sc->d, ws.d, bsc, vc, (int)(w2.numel() / vc), 0);
      if (h->pack_conv_from(ws, bsc, {}, {}, &L.pw2)) return 1;
    }
    if (h->make_conv("dec.out_conv", &h->voc_out)) return 1;
    if (h->voc_out.Cout != c.vocos_out_channels) return fail("dec.out_conv: shape does not match the config");
    {
      Raw wi;   // inverse real DFT x periodic hann window as a constant 1x1 conv: [n_fft][n_fft + 2][1]
      wi.dims = {(int64_t)c.vocos_n_fft, (int64_t)c.vocos_n_fft + 2, 1};
      if (h->dalloc(&wi.d, wi.numel())) return 1;
      launch_idft_weight(wi.d, c.vocos_n_fft, 0);
      if (h->pack_conv_from(wi, nullptr, {}, {}, &h->voc_idft)) return 1;
    }
    h->c_last = vc;
  } else
  // ---- generator
  {
    if (h->make_conv("dec.conv_pre", &h->conv_pre)) return 1;
    if (gin && h->make_conv("dec.cond", &h->dec_cond)) return 1;
    int ch = c.upsample_initial_channel;
    h->ups.resize(c.n_upsamples);
    for (int i = 0; i < c.n_upsamples; ++i) {
      const std::string p = "dec.ups." + std::to_string(i);
      Raw w;
      if (h->folded_weight(p, &w)) return 1;
      const Raw* b;
      if (h->need(p + ".bias", &b)) return 1;
      ConvT& t = h->ups[i];
      t.Cin = (int)w.dims[0];
      t.Cout = (int)w.dims[1];
      t.k = (int)w.dims[2];
      t.u = c.upsample_rates[i];
      if (t.Cin != ch || t.k != c.upsample_kernel_sizes[i]) return fail("%s: shape does not match the config", p.c_str());
      t.ntaps = t.k / t.u;
      t.pad = (t.k - t.u) / 2;
      t.CoutPad = round_cout(t.Cout);
      if (h->dalloc(&t.w, (size_t)t.Cin * t.ntaps * t.CoutPad * t.u)) return 1;
      launch_pack_convT(w.d, t.w, t.Cin, t.Cout, t.CoutPad, t.k, t.u, 0);
      std::vector<int> idm(t.CoutPad, -1);
      for (int q = 0; q < t.Cout; ++q) idm[q] = q;
      int* dmap;
      if (h->upload_ints(idm, &dmap) || h->dalloc(&t.b, (size_t)t.CoutPad)) return 1;
      launch_gather_vec(b->d, t.b, dmap, t.CoutPad, 0);
      {
        Raw eq;
        eq.dims = {(int64_t)t.Cout * t.u, (int64_t)t.Cin, (int64_t)t.ntaps};
        float* eqb;
        if (h->dalloc(&eq.d, eq.numel()) || h->dalloc(&eqb, (size_t)t.Cout * t.u)) return 1;
        launch_convT_as_conv(w.d, b->d, eq.d, eqb, t.Cin, t.Cout, t.k, t.u, 0);
        if (h->pack_conv_from(eq, eqb, {}, {}, &t.as_conv, 1)) return 1;
      }
      ch = t.Cout;
      for (int j = 0; j < c.n_resblock_kernels; ++j) {
        wetts_vits_s::ResBlock rb;
        rb.k = c.resblock_kernel_sizes[j];
        const std::string rp = "dec.resblocks." + std::to_string(i * c.n_resblock_kernels + j);
        for (int n = 0; n < c.resblock_n_dilations[j]; ++n) {
          rb.dil.push_back(c.resblock_dilations[j][n]);
          Conv a, bq;
          if (c.resblock_type == 1) {
            if (h->make_conv(rp + ".convs1." + std::to_string(n), &a, true, {}, {}, rb.dil.back()) ||
                h->make_conv(rp + ".convs2." + std::to_string(n), &bq))
              return 1;
            rb.c1.push_back(a);
            rb.c2.push_back(bq);
          } else {
            if (h->make_conv(rp + ".convs." + std::to_string(n), &a, true, {}, {}, rb.dil.back())) return 1;
            rb.c1.push_back(a);
          }
          if (a.K != rb.k || a.Cin != ch) return fail("%s: shape does not match the config", rp.c_str());
        }
        h->rbs.push_back(rb);
      }
      // f16-split fused MRF stage kernel (fused_mrf16_kernel.cuh): ResBlock1 and ResBlock2 stages with 32 / 64 channels
      h->fused16_w.push_back(nullptr);
      if (c.n_resblock_kernels <= kMrfMaxRb) {
        const int nk = c.n_resblock_kernels;
        const int nconv = (c.resblock_type == 1) ? 6 : 2;
        int ks[kMrfMaxRb] = {0, 0, 0}, dil[kMrfMaxRb][kMrfMaxConv] = {};
        bool ok = true;
        size_t halfs = 0;
        for (int j = 0; j < nk && ok; ++j) {
          const auto& rb = h->rbs[(size_t)i * nk + j];
          ks[j] = rb.k;
          if (c.resblock_type == 1) {
            ok = rb.dil.size() == 3 && rb.c1.size() == 3 && rb.c2.size() == 3;
            for (int n = 0; n < 3 && ok; ++n) { dil[j][2 * n] = rb.dil[n]; dil[j][2 * n + 1] = 1; ok = rb.c1[n].b && rb.c2[n].b; }
          } else {
            ok = rb.dil.size() == 2 && rb.c1.size() == 2 && rb.c1[0].b && rb.c1[1].b;
            if (ok) { dil[j][0] = rb.dil[0]; dil[j][1] = rb.dil[1]; }
          }
          halfs += (size_t)nconv * fused_mrf16_conv_halfs(ch, rb.k);
        }
        if (ok && fused_mrf16_supported(ch, c.resblock_type, nk, ks, dil, nconv)) {
          uint16_t* fw;
          if (h->dalloc(&fw, halfs + 64)) return 1;
          size_t off = 0;
          for (int j = 0; j < nk; ++j) {
            const auto& rb = h->rbs[(size_t)i * nk + j];
            for (int cc = 0; cc < nconv; ++cc) {
              const Conv& cv = (c.resblock_type == 1) ? ((cc & 1) ? rb.c2[cc / 2] : rb.c1[cc / 2]) : rb.c1[cc];
              launch_fused_mrf16_pack(cv.wraw, fw + off, ch, cv.K, 0);
              off += fused_mrf16_conv_halfs(ch, cv.K);
            }
          }
          h->fused16_w.back() = fw;
          uint32_t smem_base = 0;
          if (dyn_smem_offset(&smem_base, 0)) return fail("dynamic shared memory probe failed");
        }
      }
      // fused ResBlock2/MRF stage kernel (fused_rb_kernel.cuh) when the stage is eligible
      h->fused_rb_w.push_back(nullptr);
      if (c.resblock_type == 2 && c.n_resblock_kernels <= 3) {
        const int nk = c.n_resblock_kernels;
        int ks[3] = {0, 0, 0}, d1[3] = {0, 0, 0}, d2[3] = {0, 0, 0};
        bool ok = true;
        size_t floats = 0;
        for (int j = 0; j < nk; ++j) {
          const auto& rb = h->rbs[(size_t)i * nk + j];
          ok = ok && rb.dil.size() == 2 && rb.c1.size() == 2 && rb.c1[0].b && rb.c1[1].b;
          if (!ok) break;
          ks[j] = rb.k; d1[j] = rb.dil[0]; d2[j] = rb.dil[1];
          floats += 2 * fused_rb_conv_floats(ch, rb.k);
        }
        if (ok && fused_rb_supported(ch, nk, ks, d1, d2)) {
          float* fw;
          if (h->dalloc(&fw, floats)) return 1;
          size_t off = 0;
          for (int j = 0; j < nk; ++j)
            for (int n = 0; n < 2; ++n) {
              const Conv& cv = h->rbs[(size_t)i * nk + j].c1[n];
              launch_fused_rb_pack(cv.wraw, fw + off, ch, cv.K, 0);
              off += fused_rb_conv_floats(ch, cv.K);
            }
          h->fused_rb_w.back() = fw;
          uint32_t smem_base = 0;   // probe the dynamic shared-memory base now, not inside the first timed call
          if (dyn_smem_offset(&smem_base, 0)) return fail("dynamic shared memory probe failed");
        }
      }
    }
    h->c_last = ch;
    if (h->need("dec.conv_post.weight", &r)) return 1;
    if (r->dims.size() != 3 || r->dims[0] != 1 || r->dims[1] != ch) return fail("dec.conv_post.weight: unexpected shape");
    h->conv_post_w = r->d;
  }
  // ---- posterior encoder (voice conversion only; infer never reads it)
  {
    const int nl = wetts_vits_s::kPostLayers;
    auto has_conv = [&](const std::string& p) { return h->find(p + ".weight") || (h->find(p + ".weight_g") && h->find(p + ".weight_v")); };
    std::vector<std::string> convs = {"enc_q.pre"};
    for (int i = 0; i < nl; ++i) convs.push_back("enc_q.enc.in_layers." + std::to_string(i));
    for (int i = 0; i < nl; ++i) convs.push_back("enc_q.enc.res_skip_layers." + std::to_string(i));
    if (gin) convs.push_back("enc_q.enc.cond_layer");
    convs.push_back("enc_q.proj");
    for (const auto& p : convs) {
      if (!has_conv(p)) { h->post_missing = p + (h->find(p + ".weight_g") ? ".weight_v" : h->find(p + ".weight_v") ? ".weight_g" : ".weight"); break; }
      if (!h->find(p + ".bias")) { h->post_missing = p + ".bias"; break; }
    }
    if (h->post_missing.empty()) {
      auto& P = h->post;
      std::vector<int> gate(2 * H);
      for (int q = 0; q < 2 * H; ++q) gate[q] = (q & 1) ? H + (q >> 1) : (q >> 1);
      if (h->make_conv("enc_q.pre", &P.pre)) return 1;
      if (P.pre.K != 1 || P.pre.Cout != H) return fail("enc_q.pre: expected a 1x1 conv to %d channels", H);
      P.S = P.pre.Cin;
      if (gin && h->make_conv("enc_q.enc.cond_layer", &P.cond)) return 1;
      if (gin && P.cond.Cout != 2 * H * nl) return fail("enc_q.enc.cond_layer: expected %d output channels", 2 * H * nl);
      for (int i = 0; i < nl; ++i) {
        if (h->make_conv("enc_q.enc.in_layers." + std::to_string(i), &P.in[i], true, gate)) return 1;
        if (P.in[i].K != 5 || P.in[i].Cin != H) return fail("enc_q.enc.in_layers.%d: expected [%d,%d,5]", i, 2 * H, H);
        if (h->make_conv("enc_q.enc.res_skip_layers." + std::to_string(i), &P.rs[i])) return 1;
        if (P.rs[i].Cout != (i < nl - 1 ? 2 * H : H)) return fail("enc_q.enc.res_skip_layers.%d: unexpected shape", i);
      }
      if (h->make_conv("enc_q.proj", &P.proj)) return 1;
      if (P.proj.K != 1 || P.proj.Cout != 2 * Cc || P.proj.Cin != H) return fail("enc_q.proj: expected [%d,%d,1]", 2 * Cc, H);
      h->has_post = true;
      // linear spectrogram front end: n_fft = 2 (S - 1) for a power-of-two n_fft, hop = the upsample factor
      const int N = 2 * (P.S - 1);
      if (P.S >= 9 && !((P.S - 1) & (P.S - 2)) && h->U <= N && (N - h->U) % 2 == 0) {
        Raw wd;
        wd.dims = {(int64_t)N + 2, (int64_t)N, 1};
        if (h->dalloc(&wd.d, wd.numel())) return 1;
        launch_dft_weight(wd.d, N, 0);
        if (h->pack_conv_from(wd, nullptr, {}, {}, &h->spec_dft)) return 1;
        h->spec_nfft = N;
      }
    }
  }
  if (c.n_speakers > 0) {
    if (h->need("emb_g.weight", &r)) return 1;
    if (r->dims.size() != 2 || r->dims[0] != c.n_speakers || r->dims[1] != gin) return fail("emb_g.weight: unexpected shape");
    h->emb_g = r->d;
  }
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaGetLastError());
  h->finalized = true;
  return 0;
}

#define CHECK_READY(h)                                                                        \
  if (!(h)) return fail("null handle");                                                       \
  if (!(h)->finalized) return fail("handle not finalized");                                   \
  CUDA_OK(cudaSetDevice((h)->device));                                                        \
  g_call.tc = ((h)->opt_tc >= 0 ? (h)->opt_tc != 0 : tensor_cores_enabled());                 \
  g_call.fused = ((h)->opt_fused >= 0 ? (h)->opt_fused != 0 : fused_resblock_enabled());      \
  g_call.len_aware = (h)->opt_len_aware != 0;                                                 \
  g_call.fmt = ((h)->opt_fmt > 0 ? (h)->opt_fmt : g_tensor_format.load());                     \
  g_call.attn_tc = ((h)->opt_attn_tc >= 0 ? (h)->opt_attn_tc != 0 : g_attn_tc.load() != 0);

#define CHECK_LAUNCH()                                                                                   \
  do {                                                                                                   \
    cudaError_t _le = take_launcher_error();                                                             \
    if (_le != cudaSuccess) return fail("kernel attribute setup failed: %s", cudaGetErrorString(_le)); \
    CUDA_OK(cudaGetLastError());                                                                         \
  } while (0)

// ------------------------------------------------------------------ speaker embedding
int wetts_speaker_embedding(wetts_vits_t h, const int64_t* sid, int B, float* g, void* stream) {
  CHECK_READY(h);
  if (!h->emb_g) return fail("model has no speaker embedding (n_speakers == 0)");
  launch_speaker_embed((const long long*)sid, h->emb_g, g, B, h->cfg.gin_channels, h->cfg.n_speakers, (cudaStream_t)stream);
  CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ text encoder
struct TextEncWs {
  float *qkv, *att, *y, *f;
};
static size_t text_enc_layout(const wetts_vits_config& c, int B, int Tx, Arena& A, TextEncWs* w) {
  const size_t H = c.hidden_channels, F = c.filter_channels, n = (size_t)B * Tx;
  w->qkv = A.take<float>(3 * H * n);
  w->att = A.take<float>(H * n);
  w->y = A.take<float>(H * n);
  w->f = A.take<float>(F * n);
  return A.off;
}
size_t wetts_text_encoder_workspace_bytes(wetts_vits_t h, int B, int Tx) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  TextEncWs w;
  return text_enc_layout(h->cfg, B, Tx, A, &w) + 256;
}
int wetts_text_encoder_forward(wetts_vits_t h, const int64_t* ids, const int64_t* lengths, int B, int Tx, float* h_out,
                               float* m_out, float* logs_out, void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (B <= 0 || Tx <= 0) return fail("empty batch");
  if (Tx > 3000) return fail("Tx=%d exceeds the attention kernel limit (3000)", Tx);
  const wetts_vits_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  TextEncWs w;
  text_enc_layout(c, B, Tx, A, &w);
  if (!workspace || !A.ok()) return fail("text encoder workspace too small: need %zu bytes", A.off);
  const int H = c.hidden_channels, F = c.filter_channels;
  const long long* len = (const long long*)lengths;
  float* x = h_out;
  launch_embed((const long long*)ids, len, h->emb, x, B, Tx, H, c.n_vocab, sqrtf((float)H), s);
  for (int i = 0; i < c.n_layers; ++i) {
    auto& L = h->enc[i];
    ConvArgs a = conv_args(L.qkv, x, (long long)H * Tx, Tx, B, Tx);
    a.ep.out = w.qkv;
    launch_conv1d(a, s);
    if (g_call.tc && g_call.attn_tc && rel_attention_tc_supported(H, Tx, c.n_heads, 4)) {
      if (launch_rel_attention_tc(w.qkv, L.rel_k, L.rel_v, len, w.att, B, H, Tx, c.n_heads, 4, s))
        return fail("tensor-pipe attention launch failed");
    } else {
      launch_rel_attention(w.qkv, L.rel_k, L.rel_v, len, w.att, B, H, Tx, c.n_heads, 4, s);
    }
    a = conv_args(L.o, w.att, (long long)H * Tx, Tx, B, Tx);
    a.ep.out = w.y;
    launch_conv1d(a, s);
    LnArgs l;
    l.a = x; l.b = w.y; l.gamma = L.ln1.g; l.beta = L.ln1.b; l.out = x; l.B = B; l.C = H; l.T = Tx;
    launch_layernorm(l, s);
    a = conv_args(L.ffn1, x, (long long)H * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.act = 1; a.ep.out = w.f;
    launch_conv1d(a, s);
    a = conv_args(L.ffn2, w.f, (long long)F * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.out_mask = 1; a.ep.out = w.y;
    launch_conv1d(a, s);
    LnArgs l2;
    l2.a = x; l2.b = w.y; l2.gamma = L.ln2.g; l2.beta = L.ln2.b; l2.out = x; l2.B = B; l2.C = H; l2.T = Tx;
    l2.lengths = len; l2.out_mask = (i == c.n_layers - 1);
    launch_layernorm(l2, s);
  }
  ConvArgs a = conv_args(h->proj_m, x, (long long)H * Tx, Tx, B, Tx);
  a.lengths = len; a.ep.out_mask = 1; a.ep.out = m_out;
  launch_conv1d(a, s);
  a = conv_args(h->proj_logs, x, (long long)H * Tx, Tx, B, Tx);
  a.lengths = len; a.ep.out_mask = 1; a.ep.out = logs_out;
  launch_conv1d(a, s);
  CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ duration predictors
struct DurWs {
  float *cvec, *x, *y, *y2, *xc, *hb, *u, *z0, *z1;
};
static size_t dur_layout(const wetts_vits_config& c, int B, int Tx, Arena& A, DurWs* w) {
  const size_t n = (size_t)B * Tx;
  if (c.use_sdp) {
    const size_t H = c.hidden_channels;
    w->cvec = A.take<float>((size_t)B * H);
    w->x = A.take<float>(H * n);
    w->y = A.take<float>(H * n);
    w->y2 = A.take<float>(H * n);
    w->xc = A.take<float>(H * n);
    w->hb = A.take<float>(H * n);
    w->u = A.take<float>(29 * n);
    w->z0 = A.take<float>(2 * n);
    w->z1 = A.take<float>(2 * n);
  } else {
    w->cvec = A.take<float>((size_t)B * c.hidden_channels);
    w->x = A.take<float>((size_t)c.hidden_channels * n);
    w->y = A.take<float>(256 * n);
    w->y2 = A.take<float>(256 * n);
    w->xc = w->hb = w->u = w->z0 = w->z1 = nullptr;
  }
  return A.off;
}
size_t wetts_duration_workspace_bytes(wetts_vits_t h, int B, int Tx) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  DurWs w;
  return dur_layout(h->cfg, B, Tx, A, &w) + 256;
}
}  // extern "C"

namespace wetts {
__global__ void add_channel_vec_kernel(const float* __restrict__ in, const float* __restrict__ vec, float* __restrict__ out,
                                       int C, int T) {
  const int b = blockIdx.z, c = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < T) {
    const long long o = ((long long)b * C + c) * T + t;
    out[o] = in[o] + vec[(long long)b * C + c];
  }
}
}  // namespace wetts

extern "C" {
int wetts_duration_forward(wetts_vits_t h, const float* h_in, const int64_t* lengths, const float* g, const float* noise_w,
                           float noise_scale_w, int B, int Tx, float* logw, void* workspace, size_t workspace_bytes,
                           void* stream) {
  CHECK_READY(h);
  const wetts_vits_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  DurWs w;
  dur_layout(c, B, Tx, A, &w);
  if (!workspace || !A.ok()) return fail("duration workspace too small: need %zu bytes", A.off);
  const int H = c.hidden_channels;
  const long long* len = (const long long*)lengths;
  const bool has_g = g && c.gin_channels > 0;
  if (!c.use_sdp) {
    const float* x = h_in;
    if (has_g) {
      cond_vector(h->dp_cond, g, B, w.cvec, s);
      dim3 grid((Tx + 127) / 128, H, B);
      add_channel_vec_kernel<<<grid, 128, 0, s>>>(h_in, w.cvec, w.x, H, Tx);
      count_launch();
      x = w.x;
    }
    ConvArgs a = conv_args(h->dp_c1, x, (long long)H * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.act = 1; a.ep.out = w.y;
    launch_conv1d(a, s);
    LnArgs l;
    l.a = w.y; l.gamma = h->dp_n1.g; l.beta = h->dp_n1.b; l.out = w.y; l.B = B; l.C = h->dp_n1.C; l.T = Tx;
    launch_layernorm(l, s);
    a = conv_args(h->dp_c2, w.y, (long long)h->dp_c1.Cout * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.act = 1; a.ep.out = w.y2;
    launch_conv1d(a, s);
    l.a = w.y2; l.gamma = h->dp_n2.g; l.beta = h->dp_n2.b; l.out = w.y2; l.C = h->dp_n2.C;
    launch_layernorm(l, s);
    a = conv_args(h->dp_proj, w.y2, (long long)h->dp_c2.Cout * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.out_mask = 1; a.ep.out = logw;
    launch_conv1d(a, s);
    CHECK_LAUNCH();
    return 0;
  }
  if (!noise_w) return fail("stochastic duration predictor needs noise_w [B,2,Tx]");
  // x = pre(h) + cond(g)
  ConvArgs a = conv_args(h->sdp_pre, h_in, (long long)H * Tx, Tx, B, Tx);
  if (has_g) {
    cond_vector(h->sdp_cond, g, B, w.cvec, s);
    a.ep.cond = w.cvec;
    a.ep.cond_bs = H;
  }
  a.ep.out = w.x;
  launch_conv1d(a, s);
  run_dds(h->sdp_dds, w.x, w.y, w.y2, len, B, H, Tx, s);
  a = conv_args(h->sdp_proj, w.x, (long long)H * Tx, Tx, B, Tx);
  a.lengths = len; a.in_mask = 1; a.ep.out_mask = 1; a.ep.out = w.xc;
  launch_conv1d(a, s);
  launch_scale(noise_w, w.z0, noise_scale_w, (long long)B * 2 * Tx, s);
  float *zc = w.z0, *zn = w.z1;
  for (int j = 0; j < 3; ++j) {
    auto& F = h->cf[j];
    launch_convflow_pre(zc, 1, F.pre_w, F.pre_b, w.xc, w.hb, B, H, Tx, s);
    run_dds(F.dds, w.hb, w.y, w.y2, len, B, H, Tx, s);
    a = conv_args(F.proj, w.hb, (long long)H * Tx, Tx, B, Tx);
    a.lengths = len; a.in_mask = 1; a.ep.out_mask = 1; a.ep.out = w.u;
    launch_conv1d(a, s);
    launch_spline_flip(zc, w.u, 29, zn, len, B, Tx, 1.f / sqrtf((float)H), s);
    float* t = zc; zc = zn; zn = t;
  }
  launch_sdp_final(zc, h->ea_m, h->ea_logs, len, logw, B, Tx, s);
  CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ length regulation / prior expansion
int wetts_length_regulate(wetts_vits_t h, const float* logw, const int64_t* x_lengths, const float* durations,
                          float length_scale, int B, int Tx, float* w_ceil, int32_t* cum, int64_t* y_lengths, void* stream) {
  CHECK_READY(h);
  launch_length_regulate(logw, (const long long*)x_lengths, durations, length_scale, B, Tx, w_ceil, cum,
                         (long long*)y_lengths, (cudaStream_t)stream);
  CHECK_LAUNCH();
  return 0;
}

int wetts_expand_prior(wetts_vits_t h, const float* m, const float* logs, const int32_t* cum, const int64_t* x_lengths,
                       const int64_t* y_lengths, const float* noise_z, int64_t noise_bs, int64_t noise_rs,
                       float noise_scale, int B, int Tx, int Ty, float* m_p_out, float* logs_p_out, float* z_p_out,
                       float* attn, float* y_mask, void* stream) {
  CHECK_READY(h);
  if (z_p_out && !noise_z) return fail("z_p requested without noise_z");
  launch_expand_prior(m, logs, cum, (const long long*)x_lengths, (const long long*)y_lengths, noise_z, noise_bs, noise_rs,
                      noise_scale, B, h->cfg.inter_channels, Tx, Ty, m_p_out, logs_p_out, z_p_out, attn, y_mask,
                      (cudaStream_t)stream);
  CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ flow
struct FlowWs {
  float *gc, *hb, *acts, *skip;
  float *x0, *xt, *qkv, *att, *y, *f;   // VITS2 'pre_conv' flows: x0 in layer order, encoder state and scratch (half channels)
};
static size_t flow_layout(const wetts_vits_config& c, int B, int Ty, Arena& A, FlowWs* w) {
  const size_t H = c.hidden_channels, n = (size_t)B * Ty;
  w->gc = A.take<float>((size_t)B * 8 * H);
  w->hb = A.take<float>(H * n);
  w->acts = A.take<float>(H * n);
  w->skip = A.take<float>(H * n);
  w->x0 = w->xt = w->qkv = w->att = w->y = w->f = nullptr;
  if (c.flow_type == 1) {
    const size_t half = c.inter_channels / 2;
    w->x0 = A.take<float>(half * n);
    w->xt = A.take<float>(half * n);
    w->qkv = A.take<float>(3 * half * n);
    w->att = A.take<float>(half * n);
    w->y = A.take<float>(half * n);
    w->f = A.take<float>(half * n);
  }
  return A.off;
}
size_t wetts_flow_workspace_bytes(wetts_vits_t h, int B, int Ty) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  FlowWs w;
  return flow_layout(h->cfg, B, Ty, A, &w) + 256;
}
}  // extern "C"

// The four coupling layers of the flow.  Inverse (infer): reference layers 6, 4, 2, 0, each x1 = (x1 - m) * mask.
// Forward (voice conversion): layers 0, 2, 4, 6, each x1 = m + x1 * mask (flows.py:494-513, mean_only).  The Flips between
// them are folded into channel maps; a layer sees z reversed (`flipped`) in both directions alike.
static int flow_run(wetts_vits_t h, float* z, const int64_t* y_lengths, const float* g, int B, int Ty, void* workspace,
                    size_t workspace_bytes, cudaStream_t s, bool forward) {
  const wetts_vits_config& c = h->cfg;
  Arena A(workspace, workspace_bytes);
  FlowWs w;
  flow_layout(c, B, Ty, A, &w);
  if (!workspace || !A.ok()) return fail("flow workspace too small: need %zu bytes", A.off);
  const int H = c.hidden_channels, Cc = c.inter_channels, half = Cc / 2;
  const long long* len = (const long long*)y_lengths;
  const bool has_g = g && c.gin_channels > 0;
  for (int step = 0; step < 4; ++step) {
    auto& F = h->flow[forward ? 3 - step : step];
    if (has_g) cond_vector(F.cond, g, B, w.gc, s);
    ConvArgs a;
    if (c.flow_type == 1) {
      // flows.py:146-151: x0_ = pre_transformer(x0 * mask, mask) + x0 ; h = pre(x0_) * mask.  x0 = the layer's first half
      // in ITS channel order (after the Flips applied so far: the reversed second half of z when F.flipped)
      if (Ty > 3000) return fail("Ty=%d exceeds the attention kernel limit (3000) of the transformer flow", Ty);
      launch_gather_channels(z, (long long)Cc * Ty, F.flipped ? Cc - 1 : 0, F.flipped ? -1 : 1, len, w.x0, w.xt, B, half, Ty, s);
      for (int i = 0; i < 2; ++i) {
        auto& L = F.tf[i];
        ConvArgs q = conv_args(L.qkv, w.xt, (long long)half * Ty, Ty, B, Ty);
        q.ep.out = w.qkv;
        launch_conv1d(q, s);
        launch_rel_attention(w.qkv, nullptr, nullptr, len, w.att, B, half, Ty, 2, 0, s);
        q = conv_args(L.o, w.att, (long long)half * Ty, Ty, B, Ty);
        q.ep.out = w.y;
        launch_conv1d(q, s);
        LnArgs l;
        l.a = w.xt; l.b = w.y; l.gamma = L.ln1.g; l.beta = L.ln1.b; l.out = w.xt; l.B = B; l.C = half; l.T = Ty;
        launch_layernorm(l, s);
        q = conv_args(L.ffn1, w.xt, (long long)half * Ty, Ty, B, Ty);
        q.lengths = len; q.in_mask = 1; q.ep.act = 1; q.ep.out = w.f;
        launch_conv1d(q, s);
        q = conv_args(L.ffn2, w.f, (long long)half * Ty, Ty, B, Ty);
        q.lengths = len; q.in_mask = 1; q.ep.out_mask = 1; q.ep.out = w.y;
        launch_conv1d(q, s);
        LnArgs l2;
        l2.a = w.xt; l2.b = w.y; l2.gamma = L.ln2.g; l2.beta = L.ln2.b; l2.out = w.xt; l2.B = B; l2.C = half; l2.T = Ty;
        l2.lengths = len;
        if (i == 1) { l2.res = w.x0; l2.out_mask = 1; }   // (LN + x0) * mask: equals pre()'s masked input on every valid frame
        launch_layernorm(l2, s);
      }
      a = conv_args(F.pre, w.xt, (long long)half * Ty, Ty, B, Ty);
    } else {
      // h = pre(x0) * mask
      a = conv_args(F.pre, z + (F.flipped ? (long long)half * Ty : 0), (long long)Cc * Ty, Ty, B, Ty);
    }
    a.lengths = len; a.ep.out_mask = 1; a.ep.out = w.hb;
    launch_conv1d(a, s);
    run_wn(F.in, F.rs, 4, w.hb, w.acts, w.skip, has_g ? w.gc : nullptr, len, B, H, Ty, s);
    // m = post(out * mask) * mask ; x1 = (x1 - m) * mask  (forward: x1 = m + x1 * mask)
    a = conv_args(F.post, w.skip, (long long)H * Ty, Ty, B, Ty);
    a.lengths = len; a.in_mask = 1;
    a.ep.mode = EPI_COUPLING; a.ep.out = z; a.ep.out_bs = (long long)Cc * Ty;
    a.ep.z_c0 = F.flipped ? half - 1 : half;
    a.ep.z_cstep = F.flipped ? -1 : 1;
    a.ep.z_forward = forward ? 1 : 0;
    launch_conv1d(a, s);
  }
  CHECK_LAUNCH();
  return 0;
}

extern "C" {
int wetts_flow_reverse(wetts_vits_t h, float* z, const int64_t* y_lengths, const float* g, int B, int Ty, void* workspace,
                       size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  return flow_run(h, z, y_lengths, g, B, Ty, workspace, workspace_bytes, (cudaStream_t)stream, false);
}
int wetts_flow_forward(wetts_vits_t h, float* z, const int64_t* y_lengths, const float* g, int B, int Ty, void* workspace,
                       size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  return flow_run(h, z, y_lengths, g, B, Ty, workspace, workspace_bytes, (cudaStream_t)stream, true);
}

// ------------------------------------------------------------------ generator
struct GenWs {
  float *cvec, *x[2], *xu, *r, *t;
  void* item_map;   // length-aware mode: work-item list of the fused stage being launched
};
struct VocosWs {
  float *cvec, *zp, *x, *y, *hid, *spec, *frames;
};
static size_t vocos_layout(const wetts_vits_config& c, int B, int T, Arena& A, VocosWs* w) {
  const size_t n = (size_t)B * (T + 1);
  w->cvec = A.take<float>((size_t)B * c.vocos_channels);
  w->zp = A.take<float>((size_t)c.inter_channels * n);
  w->x = A.take<float>((size_t)c.vocos_channels * n);
  w->y = A.take<float>((size_t)c.vocos_channels * n);
  w->hid = A.take<float>((size_t)c.vocos_h_channels * n);
  w->spec = A.take<float>((size_t)c.vocos_out_channels * n);
  w->frames = A.take<float>((size_t)c.vocos_n_fft * n);
  return A.off;
}
// VocosGenerator.forward (decoders.py:287-307): reflection pad, in_conv + cond, LayerNorm, ConvNeXt layers (:239-247),
// LayerNorm, out_conv, exp / cos / sin, inverse STFT (inverse real DFT as a constant 1x1 conv on the tensor pipe,
// overlap-add with the squared-window envelope)
static int vocos_forward(wetts_vits_t h, const float* z, int64_t z_bs, int64_t z_cs, const int64_t* y_lengths, const float* g,
                         int B, int T, float* audio, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  const wetts_vits_config& c = h->cfg;
  Arena A(workspace, workspace_bytes);
  VocosWs w;
  vocos_layout(c, B, T, A, &w);
  if (!workspace || !A.ok()) return fail("generator workspace too small: need %zu bytes", A.off);
  const int F = T + 1, vc = c.vocos_channels;
  launch_reflect_pad_left(z, (long long)z_bs, (int)z_cs, (const long long*)y_lengths, w.zp, B, c.inter_channels, T, s);
  ConvArgs a = conv_args(h->voc_in, w.zp, (long long)c.inter_channels * F, F, B, F);
  if (g && c.gin_channels > 0) {
    cond_vector(h->voc_cond, g, B, w.cvec, s);
    a.ep.cond = w.cvec;
    a.ep.cond_bs = vc;
  }
  a.ep.out = w.x;
  launch_conv1d(a, s);
  LnArgs l;
  l.a = w.x; l.gamma = h->voc_norm_pre.g; l.beta = h->voc_norm_pre.b; l.out = w.x; l.B = B; l.C = vc; l.T = F;
  launch_layernorm(l, s);
  for (auto& L : h->voc_layers) {
    LnArgs d;   // LayerNorm(dw_conv(x)): depthwise k3 front-end of the norm kernel
    d.a = w.x; d.dww = L.dww; d.dwb = L.dwb; d.dil = 1; d.gamma = L.norm.g; d.beta = L.norm.b; d.out = w.y;
    d.B = B; d.C = vc; d.T = F;
    launch_layernorm(d, s);
    a = conv_args(L.pw1, w.y, (long long)vc * F, F, B, F);
    a.ep.act = 2; a.ep.out = w.hid;
    launch_conv1d(a, s);
    a = conv_args(L.pw2, w.hid, (long long)c.vocos_h_channels * F, F, B, F);
    a.ep.mode = EPI_RESID; a.ep.resid = w.x; a.ep.out = w.x;      // x = res + scale * pw_conv2(.)  (scale folded)
    launch_conv1d(a, s);
  }
  l.gamma = h->voc_norm_post.g; l.beta = h->voc_norm_post.b;
  launch_layernorm(l, s);
  a = conv_args(h->voc_out, w.x, (long long)vc * F, F, B, F);
  a.ep.out = w.spec;
  launch_conv1d(a, s);
  launch_vocos_spec(w.spec, B, c.vocos_out_channels / 2, F, s);
  a = conv_args(h->voc_idft, w.spec, (long long)c.vocos_out_channels * F, F, B, F);
  a.ep.out = w.frames;
  launch_conv1d(a, s);
  launch_istft_overlap_add(w.frames, audio, B, c.vocos_n_fft, c.vocos_hop_length, F, s);
  CHECK_LAUNCH();
  return 0;
}

static size_t gen_layout(wetts_vits_t h, int B, int T, Arena& A, GenWs* w) {
  const wetts_vits_config& c = h->cfg;
  if (c.vocoder_type == 1) {
    VocosWs vw;
    return vocos_layout(c, B, T, A, &vw);
  }
  size_t mx = (size_t)c.upsample_initial_channel * T;
  size_t ch = c.upsample_initial_channel, len = T;
  for (int i = 0; i < c.n_upsamples; ++i) {
    ch /= 2;
    len *= c.upsample_rates[i];
    if (ch * len > mx) mx = ch * len;
  }
  mx *= (size_t)B;
  w->cvec = A.take<float>((size_t)B * c.upsample_initial_channel);
  w->x[0] = A.take<float>(mx);
  w->x[1] = A.take<float>(mx);
  w->xu = A.take<float>(mx);
  w->r = A.take<float>(mx);
  w->t = c.resblock_type == 1 ? A.take<float>(mx) : nullptr;
  w->item_map = A.take<char>(mrf_item_map_bytes(B, (int)len));
  return A.off;
}
size_t wetts_generator_workspace_bytes(wetts_vits_t h, int B, int T) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  GenWs w;
  return gen_layout(h, B, T, A, &w) + 256;
}
int wetts_generator_forward(wetts_vits_t h, const float* z, const int64_t* y_lengths, const float* g, int B, int T,
                            float* audio, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("null handle");
  return wetts_generator_forward_view(h, z, (int64_t)h->cfg.inter_channels * T, T, y_lengths, g, B, T, audio, workspace,
                                      workspace_bytes, stream);
}
int wetts_generator_forward_view(wetts_vits_t h, const float* z, int64_t z_batch_stride, int64_t z_channel_stride,
                                 const int64_t* y_lengths, const float* g, int B, int T, float* audio, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (B <= 0 || T <= 0) return fail("empty batch");
  if (z_channel_stride < T || z_channel_stride > 0x7fffffff) return fail("bad channel stride");
  if (h->cfg.vocoder_type == 1)
    return vocos_forward(h, z, z_batch_stride, z_channel_stride, y_lengths, g, B, T, audio, workspace, workspace_bytes,
                         (cudaStream_t)stream);
  const wetts_vits_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  GenWs w;
  gen_layout(h, B, T, A, &w);
  if (!workspace || !A.ok()) return fail("generator workspace too small: need %zu bytes", A.off);
  const int Cc = c.inter_channels;
  const bool has_g = g && c.gin_channels > 0;
  (void)Cc;
  ConvArgs a = conv_args(h->conv_pre, z, (long long)z_batch_stride, (int)z_channel_stride, B, T);
  if (y_lengths) { a.lengths = (const long long*)y_lengths; a.in_mask = 1; }
  if (has_g) {
    cond_vector(h->dec_cond, g, B, w.cvec, s);
    a.ep.cond = w.cvec;
    a.ep.cond_bs = c.upsample_initial_channel;
  }
  // length-aware mode: frames beyond len + kLaMargin (> the generator's receptive field in frames) are not computed
  constexpr int kLaMargin = 16;
  const long long* la = (g_call.len_aware && y_lengths) ? (const long long*)y_lengths : nullptr;
  auto set_la = [&](ConvArgs& ca, int rate) { ca.la_len = la; ca.la_rate = rate; ca.la_margin = kLaMargin; };
  set_la(a, 1);
  int cur = 0;
  a.ep.out = w.x[cur];
  launch_conv1d(a, s);
  int len = T;
  const int nk = c.n_resblock_kernels;
  for (int i = 0; i < c.n_upsamples; ++i) {
    const ConvT& up = h->ups[i];
    ConvTArgs ta;
    ta.in = w.x[cur]; ta.w = up.w; ta.bias = up.b; ta.out = w.xu; ta.B = B; ta.Cin = up.Cin; ta.Cout = up.Cout;
    ta.CoutPad = up.CoutPad; ta.T = len; ta.u = up.u; ta.ntaps = up.ntaps; ta.pad = up.pad; ta.pre_slope = 0.1f;
    // polyphase form needs the tcgen05 kernel (EPI_CONVT / in_T exist only there) and exactly two taps per phase
    const bool up16 = up.as_conv.wtc16 && g_call.fmt == 16;
    if ((up.as_conv.wtc || up16) && g_call.tc && up.ntaps == 2 && len + up.ntaps - 1 >= 64) {
      // polyphase form on the tensor pipe: a 2-tap conv over the input frames with Cout*u packed channels
      ConvArgs ca = conv_args(up.as_conv, w.x[cur], (long long)up.Cin * len, len, B, len, 1);
      ca.T = len + up.ntaps - 1;       // frames q = 0 .. len + ntaps - 2 reach output samples
      ca.in_T = len;                   // valid input frames
      ca.pad_left = up.ntaps - 1;
      ca.pre_act = 1; ca.pre_slope = 0.1f;
      ca.ep.mode = EPI_CONVT; ca.ep.out = w.xu; ca.ep.out_bs = (long long)up.Cout * len * up.u;
      ca.ep.up_u = up.u; ca.ep.up_pad = up.pad; ca.ep.out_T = (long long)len * up.u;
      set_la(ca, len / T);
      if (up16) launch_conv1d_tc16(ca, s); else launch_conv1d_tc(ca, s);
    } else {
      launch_conv_transpose1d(ta, s);
    }
    len *= up.u;
    const int ch = up.Cout;
    const long long bs = (long long)ch * len;
    float* acc = w.x[cur ^ 1];
    if (h->fused16_w[i] && g_call.tc && g_call.fused && g_call.fmt == 16 && (len & 3) == 0) {
      FusedMrfArgs fa;
      fa.in = w.xu; fa.out = acc; fa.w = h->fused16_w[i];
      fa.B = B; fa.T = len; fa.nrb = nk; fa.slope = 0.1f; fa.div = (float)nk;
      fa.type = c.resblock_type; fa.nconv = (c.resblock_type == 1) ? 6 : 2;
      for (int j = 0; j < nk; ++j) {
        const auto& rb = h->rbs[i * nk + j];
        fa.k[j] = rb.k;
        for (int cc = 0; cc < fa.nconv; ++cc) {
          const Conv& cv = (c.resblock_type == 1) ? ((cc & 1) ? rb.c2[cc / 2] : rb.c1[cc / 2]) : rb.c1[cc];
          fa.dil[j][cc] = (c.resblock_type == 1) ? ((cc & 1) ? 1 : rb.dil[cc / 2]) : rb.dil[cc];
          fa.bias[j][cc] = cv.b;
        }
      }
      if (la) launch_mrf_item_map(la, B, len, len / T, kLaMargin, fused_mrf16_item_rows(ch, fa.type, B, (int)len), w.item_map, &fa.item_map, &fa.n_items_dev, s);
      if (launch_fused_mrf16(ch, fa, s)) return fail("fused MRF (f16) launch failed");
      cur ^= 1;
      continue;
    }
    if (h->fused_rb_w[i] && g_call.tc && g_call.fused && (len & 3) == 0) {   // 16 B row loads
      FusedRbArgs fa;
      fa.in = w.xu; fa.out = acc; fa.w = h->fused_rb_w[i];
      fa.B = B; fa.T = len; fa.nrb = nk; fa.slope = 0.1f; fa.div = (float)nk;
      for (int j = 0; j < nk; ++j) {
        const auto& rb = h->rbs[i * nk + j];
        fa.k[j] = rb.k; fa.d1[j] = rb.dil[0]; fa.d2[j] = rb.dil[1];
        fa.bias1[j] = rb.c1[0].b; fa.bias2[j] = rb.c1[1].b;
      }
      if (launch_fused_rb(ch, fa, s)) return fail("fused resblock launch failed");
      cur ^= 1;
      continue;
    }
    for (int j = 0; j < nk; ++j) {
      const auto& rb = h->rbs[i * nk + j];
      const int nd = (int)rb.dil.size();
      const int acc_mode = (nk == 1) ? 0 : (j == 0 ? 0 : (j < nk - 1 ? 1 : 2));
      const float* curp = w.xu;
      for (int n = 0; n < nd; ++n) {
        const bool last = (n == nd - 1);
        if (c.resblock_type == 1) {
          ConvArgs c1 = conv_args(rb.c1[n], curp, bs, len, B, len, rb.dil[n]);
          c1.pre_act = 1; c1.pre_slope = 0.1f; c1.ep.out = w.t;
          set_la(c1, len / T);
          launch_conv1d(c1, s);
          ConvArgs c2 = conv_args(rb.c2[n], w.t, bs, len, B, len, 1);
          c2.pre_act = 1; c2.pre_slope = 0.1f; c2.ep.resid = curp;
          if (last) { c2.ep.mode = EPI_MRF; c2.ep.acc_mode = acc_mode; c2.ep.div = (float)nk; c2.ep.out = acc; }
          else { c2.ep.mode = EPI_RESID; c2.ep.out = w.r; }
          set_la(c2, len / T);
          launch_conv1d(c2, s);
          curp = w.r;
        } else {
          // ResBlock2: x = x + c(lrelu(x)); intermediates ping-pong between r and t-less buffers
          ConvArgs c1 = conv_args(rb.c1[n], curp, bs, len, B, len, rb.dil[n]);
          c1.pre_act = 1; c1.pre_slope = 0.1f; c1.ep.resid = curp;
          float* dst = (curp == w.r) ? nullptr : w.r;
          if (last) { c1.ep.mode = EPI_MRF; c1.ep.acc_mode = acc_mode; c1.ep.div = (float)nk; c1.ep.out = acc; }
          else {
            if (!dst) return fail("ResBlock2 with more than 2 dilations is not supported");
            c1.ep.mode = EPI_RESID; c1.ep.out = dst;
          }
          set_la(c1, len / T);
          launch_conv1d(c1, s);
          curp = w.r;
        }
      }
    }
    cur ^= 1;
  }
  launch_conv_post_tanh(w.x[cur], h->conv_post_w, audio, B, h->c_last, len, 7, 0.01f, s, la, len / T, kLaMargin);
  CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------ whole path
struct InferWs {
  float *g, *hbuf, *m, *logs, *logw, *w_ceil, *zbuf;
  long long* scalar;   // per-call device scalar (max y_lengths): lives in the caller's workspace, not in the handle
  int* cum;
  void* scratch;
  size_t scratch_bytes;
};
static size_t infer_layout(wetts_vits_t h, int B, int Tx, int max_frames, Arena& A, InferWs* w) {
  const wetts_vits_config& c = h->cfg;
  const size_t n = (size_t)B * Tx;
  w->g = A.take<float>((size_t)B * (c.gin_channels > 0 ? c.gin_channels : 1));
  w->hbuf = A.take<float>((size_t)c.hidden_channels * n);
  w->m = A.take<float>((size_t)c.inter_channels * n);
  w->logs = A.take<float>((size_t)c.inter_channels * n);
  w->logw = A.take<float>(n);
  w->w_ceil = A.take<float>(n);
  w->cum = A.take<int>(n);
  w->scalar = A.take<long long>(8);
  w->zbuf = A.take<float>((size_t)B * c.inter_channels * max_frames);
  size_t s1 = wetts_text_encoder_workspace_bytes(h, B, Tx);
  size_t s2 = wetts_duration_workspace_bytes(h, B, Tx);
  size_t s3 = wetts_flow_workspace_bytes(h, B, max_frames);
  size_t s4 = wetts_generator_workspace_bytes(h, B, max_frames);
  size_t mx = s1 > s2 ? s1 : s2;
  mx = mx > s3 ? mx : s3;
  mx = mx > s4 ? mx : s4;
  w->scratch = A.take<char>(mx);
  w->scratch_bytes = mx;
  return A.off;
}
size_t wetts_vits_infer_workspace_bytes(wetts_vits_t h, int B, int Tx, int max_frames) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  InferWs w;
  return infer_layout(h, B, Tx, max_frames < 1 ? 1 : max_frames, A, &w) + 256;
}

int wetts_vits_infer_durations(wetts_vits_t h, const int64_t* ids, const int64_t* x_lengths, const int64_t* sid,
                               const float* scales3, const float* noise_w, const float* durations, int B, int Tx,
                               int64_t* y_lengths, float* logw_out, float* w_ceil_out, int* max_frames_host,
                               void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (!scales3 || !y_lengths || !max_frames_host) return fail("null argument");
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  InferWs w;
  infer_layout(h, B, Tx, 1, A, &w);  // stage 1 needs only the persistent part + Tx-sized scratch
  if (!workspace) return fail("null workspace");
  // the persistent prefix does not depend on max_frames; scratch starts after zbuf, so recompute it for this size
  if (!A.ok()) return fail("infer workspace too small: need at least %zu bytes", A.off);
  const wetts_vits_config& c = h->cfg;
  const float* g = nullptr;
  if (c.n_speakers > 0) {
    if (!sid) return fail("sid is required for a multi-speaker model");
    if (wetts_speaker_embedding(h, sid, B, w.g, stream)) return 1;
    g = w.g;
  }
  // Stage-1 scratch: use the tail of the caller's workspace (everything after the persistent prefix)
  char* tail = (char*)w.zbuf;
  const size_t tail_bytes = workspace_bytes - (size_t)(tail - (char*)workspace);
  if (wetts_text_encoder_forward(h, ids, x_lengths, B, Tx, w.hbuf, w.m, w.logs, tail, tail_bytes, stream)) return 1;
  if (wetts_duration_forward(h, w.hbuf, x_lengths, g, noise_w, scales3[2], B, Tx, w.logw, tail, tail_bytes, stream)) return 1;
  if (wetts_length_regulate(h, w.logw, x_lengths, durations, scales3[1], B, Tx, w.w_ceil, w.cum, y_lengths, stream)) return 1;
  launch_max_i64((const long long*)y_lengths, B, w.scalar, s);
  if (logw_out) CUDA_OK(cudaMemcpyAsync(logw_out, w.logw, sizeof(float) * B * Tx, cudaMemcpyDeviceToDevice, s));
  if (w_ceil_out) CUDA_OK(cudaMemcpyAsync(w_ceil_out, w.w_ceil, sizeof(float) * B * Tx, cudaMemcpyDeviceToDevice, s));
  // the one host sync of the path (Ty sizes the outputs): the landing zone is this call's stack, no handle state
  long long max_frames = 0;
  CUDA_OK(cudaMemcpyAsync(&max_frames, w.scalar, sizeof(long long), cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaStreamSynchronize(s));
  CHECK_LAUNCH();
  *max_frames_host = (int)max_frames;
  return 0;
}

int wetts_vits_infer_synthesize(wetts_vits_t h, const int64_t* x_lengths, const int64_t* y_lengths, const float* scales3,
                                const float* noise_z, int64_t noise_bs, int64_t noise_rs, int B, int Tx, int Ty,
                                int gen_frames, float* audio, float* attn, float* y_mask, float* z, float* z_p, float* m_p,
                                float* logs_p, void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (!audio || !scales3 || !noise_z) return fail("null argument");
  if (gen_frames <= 0 || gen_frames > Ty) gen_frames = Ty;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  InferWs w;
  infer_layout(h, B, Tx, Ty, A, &w);
  if (!workspace || !A.ok()) return fail("infer workspace too small: need %zu bytes for Ty=%d", A.off, Ty);
  const wetts_vits_config& c = h->cfg;
  const float* g = c.n_speakers > 0 ? w.g : nullptr;
  float* zb = z ? z : w.zbuf;
  float* zp_dst = z_p ? z_p : zb;
  if (wetts_expand_prior(h, w.m, w.logs, w.cum, x_lengths, y_lengths, noise_z, noise_bs, noise_rs, scales3[0], B, Tx, Ty,
                         m_p, logs_p, zp_dst, attn, y_mask, stream))
    return 1;
  if (zp_dst != zb)
    CUDA_OK(cudaMemcpyAsync(zb, zp_dst, sizeof(float) * (size_t)B * c.inter_channels * Ty, cudaMemcpyDeviceToDevice, s));
  if (wetts_flow_reverse(h, zb, y_lengths, g, B, Ty, w.scratch, w.scratch_bytes, stream)) return 1;
  // models.py:270-271: the vocoder sees (z * y_mask)[:, :, :max_len] -- the flow ran on all Ty frames
  if (wetts_generator_forward_view(h, zb, (int64_t)c.inter_channels * Ty, Ty, y_lengths, g, B, gen_frames, audio, w.scratch,
                                   w.scratch_bytes, stream))
    return 1;
  return 0;
}

// ------------------------------------------------------------------ voice conversion (models.py:369-376)
#define CHECK_POSTERIOR(h)                                                                                      \
  if (!(h)->has_post)                                                                                           \
    return fail("the checkpoint has no complete posterior encoder: missing checkpoint tensor '%s'", (h)->post_missing.c_str());

struct PostWs {
  float *gc, *hb, *acts, *skip, *stats;
};
static size_t post_layout(const wetts_vits_config& c, int B, int T, Arena& A, PostWs* w) {
  const size_t H = c.hidden_channels, n = (size_t)B * T;
  w->gc = A.take<float>((size_t)B * 2 * H * wetts_vits_s::kPostLayers);
  w->hb = A.take<float>(H * n);
  w->acts = A.take<float>(H * n);
  w->skip = A.take<float>(H * n);
  w->stats = A.take<float>((size_t)2 * c.inter_channels * n);
  return A.off;
}
size_t wetts_posterior_workspace_bytes(wetts_vits_t h, int B, int T) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  PostWs w;
  return post_layout(h->cfg, B, T, A, &w) + 256;
}
// PosteriorEncoder.forward (encoders.py:91-99): pre(y) * mask, WN(16 layers, g), proj(.) * mask, z = (m + noise*exp(logs)) * mask
static int posterior_run(wetts_vits_t h, const float* y, const int64_t* y_lengths, const float* g, const float* noise, int B,
                         int T, float* z, float* m, float* logs, float* y_mask, void* workspace, size_t workspace_bytes,
                         cudaStream_t s) {
  CHECK_POSTERIOR(h);
  if (!y || !y_lengths || !noise || !z) return fail("null argument");
  if (B <= 0 || T <= 0) return fail("empty batch");
  const wetts_vits_config& c = h->cfg;
  Arena A(workspace, workspace_bytes);
  PostWs w;
  post_layout(c, B, T, A, &w);
  if (!workspace || !A.ok()) return fail("posterior encoder workspace too small: need %zu bytes", A.off);
  const auto& P = h->post;
  const int H = c.hidden_channels;
  const long long* len = (const long long*)y_lengths;
  const bool has_g = g && c.gin_channels > 0;
  ConvArgs a = conv_args(P.pre, y, (long long)P.S * T, T, B, T);
  a.lengths = len; a.ep.out_mask = 1; a.ep.out = w.hb;
  launch_conv1d(a, s);
  if (has_g) cond_vector(P.cond, g, B, w.gc, s);
  run_wn(P.in, P.rs, wetts_vits_s::kPostLayers, w.hb, w.acts, w.skip, has_g ? w.gc : nullptr, len, B, H, T, s);
  a = conv_args(P.proj, w.skip, (long long)H * T, T, B, T);
  a.lengths = len; a.in_mask = 1; a.ep.out_mask = 1; a.ep.out = w.stats;
  launch_conv1d(a, s);
  launch_posterior_sample(w.stats, noise, len, z, m, logs, y_mask, B, c.inter_channels, T, s);
  CHECK_LAUNCH();
  return 0;
}
int wetts_posterior_encoder_forward(wetts_vits_t h, const float* y, const int64_t* y_lengths, const float* g, const float* noise,
                                    int B, int T, float* z, float* m, float* logs, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  CHECK_READY(h);
  return posterior_run(h, y, y_lengths, g, noise, B, T, z, m, logs, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- linear spectrogram (spectrogram_torch, mel_processing.py:42-93, center=False, per utterance)
struct SpecGeom {
  int N, K, hop, pad, F;
};
static int spec_geometry(wetts_vits_t h, int64_t L, SpecGeom* g) {
  CHECK_POSTERIOR(h);
  if (!h->spec_nfft)
    return fail("the posterior encoder takes %d feature channels, not n_fft/2+1 of a power-of-two n_fft: there is no linear "
                "spectrogram for it (a mel posterior encoder takes the caller's mel features)", h->post.S);
  g->N = h->spec_nfft;
  g->K = g->N / 2 + 1;
  g->hop = h->U;
  g->pad = (g->N - g->hop) / 2;
  if (L <= g->pad) return fail("audio of %lld samples is shorter than the %d + 1 the spectrogram's reflection padding needs",
                               (long long)L, g->pad);
  g->F = (int)(1 + (L + 2 * g->pad - g->N) / g->hop);
  return 0;
}
static size_t spec_layout(const SpecGeom& sg, int B, Arena& A, float** frames, float** dft) {
  *frames = A.take<float>((size_t)B * sg.N * sg.F);
  *dft = A.take<float>((size_t)B * 2 * sg.K * sg.F);
  return A.off;
}
size_t wetts_spectrogram_workspace_bytes(wetts_vits_t h, int B, int64_t L) {
  if (!h) return 0;
  SpecGeom sg;
  if (spec_geometry(h, L, &sg)) return 0;
  Arena A(nullptr, 0);
  float *f, *d;
  return spec_layout(sg, B, A, &f, &d) + 256;
}
int wetts_spectrogram(wetts_vits_t h, const float* audio, const int64_t* audio_lengths, int B, int64_t L, float* spec,
                      int64_t* spec_lengths, void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (!audio || !audio_lengths || !spec) return fail("null argument");
  if (B <= 0) return fail("empty batch");
  SpecGeom sg;
  if (spec_geometry(h, L, &sg)) return 1;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  float *frames, *dft;
  spec_layout(sg, B, A, &frames, &dft);
  if (!workspace || !A.ok()) return fail("spectrogram workspace too small: need %zu bytes", A.off);
  // every utterance must be longer than the reflection padding (torch's reflect pad rejects it otherwise): the lengths
  // are checked on the host, so this call synchronises `stream`
  std::vector<long long> lens(B);
  CUDA_OK(cudaMemcpyAsync(lens.data(), audio_lengths, sizeof(long long) * B, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaStreamSynchronize(s));
  for (int b = 0; b < B; ++b)
    if (lens[b] <= sg.pad || lens[b] > L)
      return fail("utterance %d has %lld samples: need %d < length <= %lld (the reflection padding of the spectrogram)", b,
                  lens[b], sg.pad, (long long)L);
  const long long* len = (const long long*)audio_lengths;
  launch_spec_frames(audio, (long long)L, len, frames, B, sg.N, sg.hop, sg.pad, sg.F, s);
  ConvArgs a = conv_args(h->spec_dft, frames, (long long)sg.N * sg.F, sg.F, B, sg.F);
  a.ep.out = dft;
  launch_conv1d(a, s);
  launch_spec_magnitude(dft, len, spec, (long long*)spec_lengths, B, sg.K, sg.F, sg.N, sg.hop, sg.pad, s);
  CHECK_LAUNCH();
  return 0;
}

// ---- the composite call: posterior encoder (g_src), forward flow (g_src), inverse flow (g_tgt), dec(z_hat * y_mask, g_tgt)
struct VcWs {
  float *g_src, *g_tgt, *z, *z_p, *z_hat;
  void* scratch;
  size_t scratch_bytes;
};
static size_t vc_layout(wetts_vits_t h, int B, int T, Arena& A, VcWs* w) {
  const wetts_vits_config& c = h->cfg;
  const size_t n = (size_t)B * c.inter_channels * T;
  w->g_src = A.take<float>((size_t)B * (c.gin_channels > 0 ? c.gin_channels : 1));
  w->g_tgt = A.take<float>((size_t)B * (c.gin_channels > 0 ? c.gin_channels : 1));
  w->z = A.take<float>(n);
  w->z_p = A.take<float>(n);
  w->z_hat = A.take<float>(n);
  size_t mx = wetts_posterior_workspace_bytes(h, B, T);
  const size_t s2 = wetts_flow_workspace_bytes(h, B, T), s3 = wetts_generator_workspace_bytes(h, B, T);
  mx = mx > s2 ? mx : s2;
  mx = mx > s3 ? mx : s3;
  w->scratch = A.take<char>(mx);
  w->scratch_bytes = mx;
  return A.off;
}
size_t wetts_vits_voice_conversion_workspace_bytes(wetts_vits_t h, int B, int T) {
  if (!h) return 0;
  Arena A(nullptr, 0);
  VcWs w;
  return vc_layout(h, B, T, A, &w) + 256;
}
int wetts_vits_voice_conversion(wetts_vits_t h, const float* y, const int64_t* y_lengths, const int64_t* sid_src,
                                const int64_t* sid_tgt, const float* noise, int B, int T, float* audio, float* y_mask, float* z,
                                float* z_p, float* z_hat, void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  CHECK_POSTERIOR(h);
  if (h->cfg.n_speakers <= 0) return fail("voice conversion needs a multi-speaker model (n_speakers == 0)");
  if (!y || !y_lengths || !sid_src || !sid_tgt || !noise || !audio) return fail("null argument");
  if (B <= 0 || T <= 0) return fail("empty batch");
  const wetts_vits_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  Arena A(workspace, workspace_bytes);
  VcWs w;
  vc_layout(h, B, T, A, &w);
  if (!workspace || !A.ok()) return fail("voice conversion workspace too small: need %zu bytes", A.off);
  const size_t zbytes = sizeof(float) * (size_t)B * c.inter_channels * T;
  float* zb = z ? z : w.z;
  float* zpb = z_p ? z_p : w.z_p;
  float* zhb = z_hat ? z_hat : w.z_hat;
  if (wetts_speaker_embedding(h, sid_src, B, w.g_src, stream) || wetts_speaker_embedding(h, sid_tgt, B, w.g_tgt, stream)) return 1;
  if (posterior_run(h, y, y_lengths, w.g_src, noise, B, T, zb, nullptr, nullptr, y_mask, w.scratch, w.scratch_bytes, s)) return 1;
  CUDA_OK(cudaMemcpyAsync(zpb, zb, zbytes, cudaMemcpyDeviceToDevice, s));
  if (wetts_flow_forward(h, zpb, y_lengths, w.g_src, B, T, w.scratch, w.scratch_bytes, stream)) return 1;
  CUDA_OK(cudaMemcpyAsync(zhb, zpb, zbytes, cudaMemcpyDeviceToDevice, s));
  if (wetts_flow_reverse(h, zhb, y_lengths, w.g_tgt, B, T, w.scratch, w.scratch_bytes, stream)) return 1;
  // models.py:376: the vocoder sees z_hat * y_mask over the full padded length
  return wetts_generator_forward(h, zhb, y_lengths, w.g_tgt, B, T, audio, w.scratch, w.scratch_bytes, stream);
}

// ------------------------------------------------------------------ L2 decoder contract
size_t wetts_vits_decoder_workspace_bytes(wetts_vits_t h, int B, int L) {
  if (!h) return 0;
  return wetts_generator_workspace_bytes(h, B, L) + sizeof(float) * ((size_t)B * h->cfg.inter_channels * L +
                                                                     (size_t)B * (h->cfg.gin_channels + 1)) + 1024;
}
int wetts_vits_forward_decoder(wetts_vits_t h, const float* z_blc, const int64_t* sid, int B, int L, float* audio,
                               void* workspace, size_t workspace_bytes, void* stream) {
  CHECK_READY(h);
  if (!workspace || workspace_bytes < wetts_vits_decoder_workspace_bytes(h, B, L))
    return fail("decoder workspace too small: need %zu bytes", wetts_vits_decoder_workspace_bytes(h, B, L));
  Arena A(workspace, workspace_bytes);
  float* zt = A.take<float>((size_t)B * h->cfg.inter_channels * L);
  float* g = A.take<float>((size_t)B * (h->cfg.gin_channels + 1));
  A.off = (A.off + 255) & ~(size_t)255;
  launch_transpose_blc(z_blc, zt, B, L, h->cfg.inter_channels, (cudaStream_t)stream);
  const float* gp = nullptr;
  if (h->cfg.n_speakers > 0) {
    if (!sid) return fail("sid is required for a multi-speaker model");
    if (wetts_speaker_embedding(h, sid, B, g, stream)) return 1;
    gp = g;
  }
  return wetts_generator_forward(h, zt, nullptr, gp, B, L, audio, (char*)workspace + A.off, workspace_bytes - A.off, stream);
}

}  // extern "C"
