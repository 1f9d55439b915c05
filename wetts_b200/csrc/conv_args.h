// Argument structs of the convolution kernels (plain C++, no CUDA dependency: shared by the SIMT kernels, the
// tcgen05 kernels, the engine and the host CTA emulator).
#pragma once
#include <stddef.h>
#include <stdint.h>

namespace wetts {

enum EpiMode : int {
  EPI_PLAIN = 0,     // out = act(v + cond) [* mask]
  EPI_RESID = 1,     // out = v + resid                         (ResBlock inner add)
  EPI_MRF = 2,       // val = v + resid; acc_mode 0: out=val, 1: out+=val, 2: out=(out+val)/div
  EPI_GATE = 3,      // paired channels -> tanh(a+ga)*sigmoid(b+gb)   (modules.py:76-77)
  EPI_RES_SKIP = 4,  // co<H: x=(x+v)*mask ; co>=H: skip(+)=v         (modules.py:81-86)
  EPI_COUPLING = 5,  // z1 = (z1 - v*mask)*mask  (flows.py:510); z_forward: z1 = (z1 + v*mask)*mask  (flows.py:505)
  EPI_CONVT = 6,     // polyphase ConvTranspose1d scatter (tensor-core path only)
};

struct ConvEpilogue {
  int mode = EPI_PLAIN;
  float* out = nullptr;      // [B][*][T], batch stride out_bs, channel stride T
  long long out_bs = 0;
  const float* resid = nullptr;  // same geometry as out
  const float* cond = nullptr;   // per (b, co) additive term, cond[b*cond_bs + cond_off + co]
  int cond_bs = 0;
  int cond_off = 0;
  int act = 0;               // 0 none, 1 relu, 2 gelu (erf)
  int out_mask = 0;          // multiply result by (t < lengths[b])
  int acc_mode = 0;          // EPI_MRF
  float div = 1.f;           // EPI_MRF final divisor
  int H = 0;                 // EPI_GATE / EPI_RES_SKIP hidden size
  float* x = nullptr;        // EPI_RES_SKIP residual stream (in place), batch stride out_bs
  float* skip = nullptr;     // EPI_RES_SKIP skip accumulator, batch stride out_bs
  int skip_init = 0;         // 1: skip = v (first layer), 0: skip += v
  int last = 0;              // last WN layer: all Cout channels go to skip
  int z_c0 = 0;              // EPI_COUPLING: target channel = z_c0 + co*z_cstep in `out`
  int z_cstep = 1;
  int z_forward = 0;         // EPI_COUPLING: 0 = inverse direction (subtract the mean), 1 = forward (add it)
  int up_u = 1, up_pad = 0;  // EPI_CONVT: stride and padding of the transposed conv
  long long out_T = 0;       // EPI_CONVT: output samples per channel
};

// tiling of the tcgen05 implicit-GEMM path (tc_conv_kernel.cu), fixed per conv at load time
struct TcPlan {
  int mode = 0, N = 0, n_tiles = 0, KC = 0, n_chunks = 0, MB = 0, G = 0, n_abuf = 2, n_bbuf = 0, R_pad = 0, dil = 1;
  int tmem_cols = 512;
  size_t packed_floats = 0;
};

struct ConvArgs {
  const float* wtc = nullptr;  // tensor-core packed weights, 3xTF32 layout (nullptr: not eligible)
  TcPlan tc;
  const void* wtc16 = nullptr; // tensor-core packed weights, f16-split layout (nullptr: not eligible)
  TcPlan tc16;
  int fmt = 32;               // operand format to use when both layouts exist: 16 = f16 split, 32 = 3xTF32
  const float* in = nullptr;  // [B][Cin][T] view: element (b,ci,t) at in + b*in_bs + ci*in_cs + t
  long long in_bs = 0;
  int in_cs = 0;
  const float* w = nullptr;   // packed [Cin][K][CoutPad]
  const float* bias = nullptr;  // packed [CoutPad] or nullptr
  int B = 0, Cin = 0, Cout = 0, CoutPad = 0, T = 0, K = 1, dil = 1, pad_left = 0;
  int in_T = 0;               // valid input length when it differs from T (0: same as T); tensor-core path only
  int pre_act = 0;            // 1: leaky_relu(pre_slope) applied to the input
  float pre_slope = 0.1f;
  const long long* lengths = nullptr;  // int64[B] or nullptr
  int in_mask = 0;            // multiply the input by (t < lengths[b])
  int use_tc = 1;             // 0: force the fp32 SIMT kernel for this call (per-handle / process option)
  // length-aware mode (optional): work whose first output row lies at or beyond (la_len[b] + la_margin) * la_rate is
  // skipped (la_len in frames of z, la_rate = rows of THIS conv's time axis per frame); the skipped output rows are
  // left unwritten
  const long long* la_len = nullptr;
  int la_rate = 1, la_margin = 0;
  ConvEpilogue ep;
};
struct TcConvArgs {
  ConvArgs c;
  const float* wtc;
  int N, n_tiles, KC, n_chunks, MB, G, n_abuf, n_bbuf, R_pad, tmem_cols;
  int nt_minor = 0;     // work items ordered (rows, N tile) instead of (N tile, rows): the tiles of one row block run side by side
  long long* prof = nullptr;   // pipelined kernel, profiling instantiation: [cta][role 0..3][9] cycle counters
  int acc_slots = 1;    // pipelined kernel: accumulator sets in TMEM (2 = the MMAs of the next item overlap the drain of this one)
  int all_warps = 0;    // pipelined kernel (tc16p): 1 = warps 2..15 stage and warps 4..15 drain, 0 = 6 stager + 8 epilogue warps
  int stagger = 0;      // per-layer kernel: CTA i starts (i % 8) * stagger / 8 cycles late, so that the CTAs' memory-bound phases
                        // (staging, epilogue) and tensor-bound phases (MMAs) do not all coincide on the chip
  int epi_preload = 0;  // per-layer kernel: the epilogue's residual / skip / coupling operand is loaded before the accumulators are waited for
  int debug_skip = 0;   // experiments only (WETTS_TC16_DEBUG_SKIP): 1 = no staging work, 2 = no epilogue work (wrong results)
  int l2_prefetch = 0;  // warm L2 one work item ahead (activations) and for this item's epilogue operands
};

}  // namespace wetts
