// Conv epilogues shared by the fp32 SIMT kernel and the tcgen05 kernel, so both paths have
// bit-identical post-accumulation semantics (see EpiMode in kernels.cuh).
#pragma once
#include "kernels.cuh"

namespace wetts {

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.f / (1.f + expf(-x)); }
// tanh(a) * sigmoid(b) of the WaveNet gate on the tensor-pipe kernels' epilogue: two ex2.approx + two rcp.approx instead
// of tanhf + expf + a division (45 -> 14 instructions per gated value; the gate was 19 % of the instructions of a flow
// in_layer launch).  |error| <= 2.1e-7 absolute on outputs in (-1, 1) (tools/split_precision_probe-style check in numpy:
// 3.7e-7 of the rms), far inside the 1e-4 block tolerance; the fp32 SIMT path keeps tanhf / expf.
__device__ __forceinline__ float gate_tanh_sigmoid_fast(float a, float b) {
  const float e = __expf(-2.f * fabsf(a));                 // in (0, 1]
  const float t = copysignf(__fdividef(1.f - e, 1.f + e), a);
  const float s = __fdividef(1.f, 1.f + __expf(-b));       // __expf(-b) = inf for b < -88: s = 0, as it should
  return t * s;
}
__device__ __forceinline__ float gelu_erf_acc(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

// bias (+ per-(b,co) conditioning for EPI_PLAIN) of packed output channel `co`
__device__ __forceinline__ float channel_term(const ConvArgs& a, int b, int co) {
  float bv = a.bias ? a.bias[co] : 0.f;
  if (a.ep.mode == EPI_PLAIN && a.ep.cond) bv += a.ep.cond[(long long)b * a.ep.cond_bs + a.ep.cond_off + co];
  return bv;
}

// Epilogues are split in two phases so a thread can issue the global loads of many outputs
// back to back (memory-level parallelism) before any dependent store: epilogue_load() only
// reads, epilogue_finish() computes and writes.
struct EpiLoad {
  float a = 0.f, b = 0.f;
};

__device__ __forceinline__ EpiLoad epilogue_load(const ConvArgs& a, int b, int co, int t) {
  const ConvEpilogue& e = a.ep;
  EpiLoad l;
  const long long off = (long long)b * e.out_bs + (long long)co * a.T + t;
  switch (e.mode) {
    case EPI_RESID:
      l.a = e.resid[off];
      break;
    case EPI_MRF:
      l.a = e.resid[off];
      if (e.acc_mode != 0) l.b = e.out[off];
      break;
    case EPI_RES_SKIP:
      if (!e.last && co < e.H) l.a = e.x[off];
      else if (!e.skip_init) l.a = e.skip[(long long)b * e.out_bs + (long long)(e.last ? co : co - e.H) * a.T + t];
      break;
    case EPI_COUPLING:
      l.a = e.out[(long long)b * e.out_bs + (long long)(e.z_c0 + co * e.z_cstep) * a.T + t];
      break;
    default:
      break;
  }
  return l;
}

// v already contains the bias term
__device__ __forceinline__ void epilogue_finish(const ConvArgs& a, int b, int co, int t, float v, float msk,
                                                const EpiLoad& l) {
  const ConvEpilogue& e = a.ep;
  const int T = a.T;
  const long long off = (long long)b * e.out_bs + (long long)co * T + t;
  switch (e.mode) {
    case EPI_PLAIN:
      if (e.act == 1) v = fmaxf(v, 0.f);
      else if (e.act == 2) v = gelu_erf_acc(v);
      if (e.out_mask) v *= msk;
      e.out[off] = v;
      break;
    case EPI_RESID:
      e.out[off] = v + l.a;
      break;
    case EPI_MRF: {
      v += l.a;
      if (e.acc_mode == 0) e.out[off] = v;
      else if (e.acc_mode == 1) e.out[off] = l.b + v;
      else e.out[off] = (l.b + v) / e.div;
      break;
    }
    case EPI_RES_SKIP: {
      if (!e.last && co < e.H) {
        e.x[off] = (l.a + v) * msk;
      } else {
        const int c2 = e.last ? co : co - e.H;
        e.skip[(long long)b * e.out_bs + (long long)c2 * T + t] = e.skip_init ? v : l.a + v;
      }
      break;
    }
    case EPI_COUPLING: {
      const int zc = e.z_c0 + co * e.z_cstep;
      if (e.z_forward) v = -v;   // exact: the inverse direction keeps its expression (and its FMA) bit for bit
      e.out[(long long)b * e.out_bs + (long long)zc * T + t] = (l.a - v * msk) * msk;
      break;
    }
    default:
      break;
  }
}

__device__ __forceinline__ void epilogue_store(const ConvArgs& a, int b, int co, int t, float v, float msk) {
  epilogue_finish(a, b, co, t, v, msk, epilogue_load(a, b, co, t));
}

// EPI_GATE: packed channels (co, co+1) = (tanh half j, sigmoid half j), j = co/2
__device__ __forceinline__ void gate_terms(const ConvArgs& a, int b, int co, float& ba, float& bb) {
  ba = 0.f;
  bb = 0.f;
  if (a.bias) { ba = a.bias[co]; bb = a.bias[co + 1]; }
  if (a.ep.cond) {
    const float* g = a.ep.cond + (long long)b * a.ep.cond_bs + a.ep.cond_off;
    ba += g[co >> 1];
    bb += g[a.ep.H + (co >> 1)];
  }
}
__device__ __forceinline__ void gate_store(const ConvArgs& a, int b, int co, int t, float va, float vb) {
  a.ep.out[(long long)b * a.ep.out_bs + (long long)(co >> 1) * a.T + t] = tanhf(va) * sigmoidf_acc(vb);
}

}  // namespace wetts
