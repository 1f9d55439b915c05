// Fused conv epilogues of the tensor-pipe kernels in host-compilable form (no CUDA dependency beyond the tc_prims.cuh
// wrappers): the same code runs on the device and in the host CTA emulator.  Semantics: EpiMode in conv_args.h.
#pragma once
#include <math.h>

#include "conv_args.h"
#include "tc_prims.cuh"

namespace wetts {

WETTS_DEVICE float ep_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }
WETTS_DEVICE float ep_gelu(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }
WETTS_DEVICE int ep_min(int a, int b) { return a < b ? a : b; }
WETTS_DEVICE int ep_max(int a, int b) { return a > b ? a : b; }
// tanh(a) * sigmoid(b) of the WaveNet gate with two fast exponentials and two fast divisions (device: ex2.approx /
// rcp.approx, |error| <= 2.1e-7 on outputs in (-1, 1); host emulator: libm): see gate_tanh_sigmoid_fast in epilogue.cuh
WETTS_DEVICE float ep_gate(float a, float b) {
#ifdef WETTS_EMULATE
  const float e = expf(-2.f * fabsf(a));
  return copysignf((1.f - e) / (1.f + e), a) * (1.f / (1.f + expf(-b)));
#else
  const float e = __expf(-2.f * fabsf(a));
  return copysignf(__fdividef(1.f - e, 1.f + e), a) * __fdividef(1.f, 1.f + __expf(-b));
#endif
}

// Warm L2 with what the epilogue of a work item (channels [c_lo, c_hi), rows [r_lo, r_hi) of utterance b) reads back.
WETTS_DEVICE void tc_epilogue_prefetch(const ConvArgs& a, int b, int c_lo, int c_hi, int r_lo, int r_hi, int tid, int nthreads) {
  const ConvEpilogue& e = a.ep;
  const long long T = a.T, ob = (long long)b * e.out_bs;
  if (e.mode == EPI_RESID || e.mode == EPI_MRF) {
    tc::l2_prefetch_rows(e.resid + ob + (long long)c_lo * T, T, c_hi - c_lo, r_lo, r_hi, tid, nthreads);
    if (e.mode == EPI_MRF && e.acc_mode != 0) tc::l2_prefetch_rows(e.out + ob + (long long)c_lo * T, T, c_hi - c_lo, r_lo, r_hi, tid, nthreads);
  } else if (e.mode == EPI_RES_SKIP) {
    if (!e.last && c_lo < e.H) tc::l2_prefetch_rows(e.x + ob + (long long)c_lo * T, T, ep_min(c_hi, e.H) - c_lo, r_lo, r_hi, tid, nthreads);
    if (!e.skip_init && (e.last || c_hi > e.H)) {
      const int s_lo = e.last ? c_lo : ep_max(c_lo, e.H) - e.H, s_hi = e.last ? c_hi : c_hi - e.H;
      tc::l2_prefetch_rows(e.skip + ob + (long long)s_lo * T, T, s_hi - s_lo, r_lo, r_hi, tid, nthreads);
    }
  } else if (e.mode == EPI_COUPLING) {
    tc::l2_prefetch_rows(e.out + ob + (long long)(e.z_c0 + c_lo * e.z_cstep) * T, (long long)e.z_cstep * T, c_hi - c_lo, r_lo, r_hi, tid, nthreads);
  }
}

// NE strided loads / stores (channel stride `step` floats): one 64-bit add per element and, for a full slice, no
// per-element predicate (the kernels around these epilogues are bound by instruction issue).
template <int NE>
WETTS_DEVICE void ep_ld_strided(const float* p, long long step, int nval, float (&r)[16]) {
  if (nval >= NE) {
#pragma unroll
    for (int i = 0; i < NE; ++i) { r[i] = *p; p += step; }
  } else {
#pragma unroll
    for (int i = 0; i < NE; ++i) { r[i] = (i < nval) ? *p : 0.f; p += step; }
  }
}
template <int NE>
WETTS_DEVICE void ep_st_strided(float* p, long long step, int nval, const float (&x)[16]) {
  if (nval >= NE) {
#pragma unroll
    for (int i = 0; i < NE; ++i) { *p = x[i]; p += step; }
  } else {
#pragma unroll
    for (int i = 0; i < NE; ++i) { if (i < nval) *p = x[i]; p += step; }
  }
}

// Fused epilogue of one 16-channel slice of one output row with the mode as a template parameter (branch-free per
// instantiation).  v[i] already contains bias (+ conditioning).
template <int MODE>
WETTS_DEVICE void tc_epilogue_slice_m(const ConvArgs& a, int b, int t, int co0, float* v, float msk) {
  const ConvEpilogue& e = a.ep;
  const size_t Ts = (size_t)a.T;
  const long long step = (long long)Ts;
  const size_t row = (size_t)b * (size_t)e.out_bs + (size_t)t;
  const int nval = ep_min(16, a.Cout - co0);
  float x[16], r[16];
  switch (MODE) {
    case EPI_PLAIN: {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        x[i] = v[i];
        if (e.act == 1) x[i] = fmaxf(x[i], 0.f);
        else if (e.act == 2) x[i] = ep_gelu(x[i]);
        if (e.out_mask) x[i] *= msk;
      }
      ep_st_strided<16>(e.out + row + (size_t)co0 * Ts, step, nval, x);
      break;
    }
    case EPI_RESID: {
      ep_ld_strided<16>(e.resid + row + (size_t)co0 * Ts, step, nval, r);
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = v[i] + r[i];
      ep_st_strided<16>(e.out + row + (size_t)co0 * Ts, step, nval, x);
      break;
    }
    case EPI_MRF: {
      float* op = e.out + row + (size_t)co0 * Ts;
      float o[16];
      ep_ld_strided<16>(e.resid + row + (size_t)co0 * Ts, step, nval, r);
      if (e.acc_mode != 0) ep_ld_strided<16>(op, step, nval, o);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        x[i] = v[i] + r[i];
        if (e.acc_mode == 1) x[i] = o[i] + x[i];
        else if (e.acc_mode == 2) x[i] = (o[i] + x[i]) / e.div;
      }
      ep_st_strided<16>(op, step, nval, x);
      break;
    }
    case EPI_GATE: {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = ep_gate(v[2 * i], v[2 * i + 1]);
      ep_st_strided<8>(e.out + row + (size_t)(co0 >> 1) * Ts, step, (nval + 1) >> 1, x);
      break;
    }
    case EPI_RES_SKIP: {
      if (!e.last && co0 < e.H) {  // residual stream (a 16-slice never straddles H: H % 16 == 0 is checked on the host)
        float* xp = e.x + row + (size_t)co0 * Ts;
        ep_ld_strided<16>(xp, step, nval, r);
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = (r[i] + v[i]) * msk;
        ep_st_strided<16>(xp, step, nval, x);
      } else {
        float* sp = e.skip + row + (size_t)(e.last ? co0 : co0 - e.H) * Ts;
        if (!e.skip_init) {
          ep_ld_strided<16>(sp, step, nval, r);
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = r[i] + v[i];
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = v[i];
        }
        ep_st_strided<16>(sp, step, nval, x);
      }
      break;
    }
    case EPI_CONVT: {
      // polyphase ConvTranspose1d: packed channel = co*u + r, row t = input frame q; output sample
      // n = q*u + r - pad of channel co.  The u phases of one (q, co) are u consecutive samples, so a slice of
      // 16 packed channels is 16/u runs of u contiguous floats: written with 8 / 16 B stores when the run is
      // inside the signal and suitably aligned (u = 4: pad 2 -> 8 B; u = 8: pad 4 -> 16 B), else sample by sample.
      const int u = e.up_u;
      const long long n0 = (long long)t * u - e.up_pad;
      float* ob = e.out + (size_t)b * (size_t)e.out_bs;
      const bool whole = (nval == 16) && (n0 >= 0) && (n0 + u <= e.out_T) && ((e.out_T & 3) == 0);
      if (u == 8 && whole && (co0 & 7) == 0 && (n0 & 3) == 0) {
#pragma unroll
        for (int i = 0; i < 16; i += 8) {
          float4* dst = reinterpret_cast<float4*>(ob + (size_t)((co0 + i) >> 3) * (size_t)e.out_T + (size_t)n0);
          dst[0] = make_float4(v[i + 0], v[i + 1], v[i + 2], v[i + 3]);
          dst[1] = make_float4(v[i + 4], v[i + 5], v[i + 6], v[i + 7]);
        }
      } else if (u == 4 && whole && (co0 & 3) == 0 && (n0 & 1) == 0) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          float2* dst = reinterpret_cast<float2*>(ob + (size_t)((co0 + i) >> 2) * (size_t)e.out_T + (size_t)n0);
          dst[0] = make_float2(v[i + 0], v[i + 1]);
          dst[1] = make_float2(v[i + 2], v[i + 3]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int cp = co0 + i;
          const int co = cp / u, r = cp - co * u;
          const long long n = n0 + r;
          if (i < nval && n >= 0 && n < e.out_T) ob[(size_t)co * (size_t)e.out_T + (size_t)n] = v[i];
        }
      }
      break;
    }
    case EPI_COUPLING: {
      float* zp = e.out + row + (size_t)(e.z_c0 + co0 * e.z_cstep) * Ts;
      const long long zstep = (long long)e.z_cstep * (long long)Ts;
      ep_ld_strided<16>(zp, zstep, nval, r);
      const float zsgn = e.z_forward ? -1.f : 1.f;   // forward direction: v * -1 (exact); inverse: v * 1 == v bit for bit
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = (r[i] - (v[i] * zsgn) * msk) * msk;
      ep_st_strided<16>(zp, zstep, nval, x);
      break;
    }
    default:
      break;
  }
}

// the same with the mode read at run time (pipelined kernel tc16p)
WETTS_DEVICE void tc_epilogue_slice_p(const ConvArgs& a, int b, int t, int co0, float* v, float msk) {
  switch (a.ep.mode) {
    case EPI_PLAIN: tc_epilogue_slice_m<EPI_PLAIN>(a, b, t, co0, v, msk); break;
    case EPI_RESID: tc_epilogue_slice_m<EPI_RESID>(a, b, t, co0, v, msk); break;
    case EPI_MRF: tc_epilogue_slice_m<EPI_MRF>(a, b, t, co0, v, msk); break;
    case EPI_GATE: tc_epilogue_slice_m<EPI_GATE>(a, b, t, co0, v, msk); break;
    case EPI_RES_SKIP: tc_epilogue_slice_m<EPI_RES_SKIP>(a, b, t, co0, v, msk); break;
    case EPI_COUPLING: tc_epilogue_slice_m<EPI_COUPLING>(a, b, t, co0, v, msk); break;
    case EPI_CONVT: tc_epilogue_slice_m<EPI_CONVT>(a, b, t, co0, v, msk); break;
    default: break;
  }
}

}  // namespace wetts
