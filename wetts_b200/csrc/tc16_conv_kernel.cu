// tcgen05 (5th-gen tensor core) implicit-GEMM Conv1d for sm_100a, fp32-accurate via the f16 operand split
// (tensor_format = 16; the 3xTF32 twin of this file is tc_conv_kernel.cu).  Same pipeline, different operand format:
//   x ~ hi + lo' * 2^-11,  hi = f16(x),  lo' = f16((x - hi) * 2^11)   (22 significand bits, |x| < 65504)
//   K = 16 input channels per tcgen05.mma (kind::f16): half the MMAs and half the operand bytes of the TF32 form;
//   two MMAs per k-step: A_hi x [B_hi | B_lo'] -> accumulator columns [0, 2N), A_lo' x B_hi -> columns [N, 2N);
//   the epilogue adds columns [N, 2N) scaled by 2^-11.  An N tile is therefore at most 128 channels (2N <= 256).
// Original header of the shared design:
// tcgen05 (5th-gen tensor core) implicit-GEMM Conv1d for sm_100a.
//
//   D[time, co] = sum_{tap, ci} A[time + tap*dil, ci] * W[co, ci, tap]
//
// * M = 128 time rows per MMA, N = C_out tile (<= 256), K = 8 input channels per tcgen05.mma
//   (kind::tf32).  Accumulators live in TMEM (512 columns = up to 8 resident 128xN tiles), read
//   back with tcgen05.ld for the fused epilogue (epilogue.cuh: bias / residual / MRF mean /
//   WaveNet gate / res-skip / coupling update).
// * Operands are staged in shared memory in the no-swizzle K-major canonical layout
//   (8 rows x 16 B core matrices): element (row r, channel c) at (c/4)*LBO + r*16 + (c%4)*4.
//   With SBO = 128 B all rows of a 4-channel group are contiguous at a 16 B pitch, so a conv tap
//   is just a +tap*dil*16 B shift of the descriptor start address: no im2col, one staged tile
//   serves every tap and dilation.
// * fp32 accuracy: x = hi + lo with hi = tf32(x), lo = tf32(x - hi); three MMAs per product
//   (hi*hi, hi*lo, lo*hi) accumulate in fp32 (error ~2^-21 relative, far inside the stated
//   tolerance; plain TF32 would not be).  Weights are split once at load time; activations are
//   split while they are staged (together with leaky-relu, masks and zero padding).
// * Weights arrive by cp.async.bulk (TMA 1-D bulk copy) + mbarrier; tcgen05.commit signals
//   buffer reuse and accumulator completion; one persistent CTA per SM loops over work items
//   and keeps the weight tile resident when it can.
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "epilogue.cuh"
#include "kernels.cuh"
#include "tc_prims.cuh"

namespace wetts {
namespace {


using namespace tc;   // PTX wrappers shared with the fused kernels (tc_prims.cuh)

// Fused epilogue of one 16-channel slice of one output row, specialised per mode with the switch
// hoisted out of the element loops: all global loads of the slice are issued before the first store.
// v[i] already contains bias (+ conditioning).
// N strided loads / stores (channel stride `step` floats) with one 64-bit add per element and, for a full slice, no
// per-element predicate (the per-element `i < nval` test + 64-bit multiply cost 13 instructions per store, and the kernel
// is issue bound: 79 k warp-instructions per 256-row item at 4 warps per scheduler).
template <int NE>
__device__ __forceinline__ void ld_strided(const float* p, long long step, int nval, float (&r)[16]) {
  if (nval >= NE) {
#pragma unroll
    for (int i = 0; i < NE; ++i) { r[i] = *p; p += step; }
  } else {
#pragma unroll
    for (int i = 0; i < NE; ++i) { r[i] = (i < nval) ? *p : 0.f; p += step; }
  }
}
template <int NE>
__device__ __forceinline__ void st_strided(float* p, long long step, int nval, const float (&x)[16]) {
  if (nval >= NE) {
#pragma unroll
    for (int i = 0; i < NE; ++i) { *p = x[i]; p += step; }
  } else {
#pragma unroll
    for (int i = 0; i < NE; ++i) { if (i < nval) *p = x[i]; p += step; }
  }
}

template <int MODE>
__device__ __forceinline__ void tc16_epilogue_slice(const ConvArgs& a, int b, int t, int co0, float* v, float msk) {
  const ConvEpilogue& e = a.ep;
  const size_t Ts = (size_t)a.T;
  const long long step = (long long)Ts;
  const size_t row = (size_t)b * (size_t)e.out_bs + (size_t)t;
  const int nval = min(16, a.Cout - co0);
  float x[16], r[16];
  switch (MODE) {
    case EPI_PLAIN: {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        x[i] = v[i];
        if (e.act == 1) x[i] = fmaxf(x[i], 0.f);
        else if (e.act == 2) x[i] = gelu_erf_acc(x[i]);
        if (e.out_mask) x[i] *= msk;
      }
      st_strided<16>(e.out + row + (size_t)co0 * Ts, step, nval, x);
      break;
    }
    case EPI_RESID: {
      ld_strided<16>(e.resid + row + (size_t)co0 * Ts, step, nval, r);
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = v[i] + r[i];
      st_strided<16>(e.out + row + (size_t)co0 * Ts, step, nval, x);
      break;
    }
    case EPI_MRF: {
      float* op = e.out + row + (size_t)co0 * Ts;
      float o[16];
      ld_strided<16>(e.resid + row + (size_t)co0 * Ts, step, nval, r);
      // one code path for "accumulate" (acc_mode 1: dv = 1, x / 1 == x bit for bit) and "accumulate and average" (2): a
      // three-way branch on acc_mode here made ptxas version the whole persistent loop and move the MMA descriptors through
      // predicated R2UR.BROADCAST in this instantiation (170 R2UR, 20 UTCHMMA; now 60 / 14 like the other modes)
      const float dv = (e.acc_mode == 2) ? e.div : 1.0f;
      if (e.acc_mode != 0) ld_strided<16>(op, step, nval, o);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        x[i] = v[i] + r[i];
        if (e.acc_mode != 0) x[i] = (o[i] + x[i]) / dv;
      }
      st_strided<16>(op, step, nval, x);
      break;
    }
    case EPI_GATE: {
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = gate_tanh_sigmoid_fast(v[2 * i], v[2 * i + 1]);
      st_strided<8>(e.out + row + (size_t)(co0 >> 1) * Ts, step, (nval + 1) >> 1, x);
      break;
    }
    case EPI_RES_SKIP: {
      if (!e.last && co0 < e.H) {  // residual stream (a 16-slice never straddles H: H % 16 == 0 is checked on the host)
        float* xp = e.x + row + (size_t)co0 * Ts;
        ld_strided<16>(xp, step, nval, r);
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = (r[i] + v[i]) * msk;
        st_strided<16>(xp, step, nval, x);
      } else {
        float* sp = e.skip + row + (size_t)(e.last ? co0 : co0 - e.H) * Ts;
        if (!e.skip_init) {
          ld_strided<16>(sp, step, nval, r);
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = r[i] + v[i];
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = v[i];
        }
        st_strided<16>(sp, step, nval, x);
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
      ld_strided<16>(zp, zstep, nval, r);
      const float zsgn = e.z_forward ? -1.f : 1.f;   // forward direction: v * -1 (exact); inverse: v * 1 == v bit for bit
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = (r[i] - (v[i] * zsgn) * msk) * msk;
      st_strided<16>(zp, zstep, nval, x);
      break;
    }
    default:
      break;
  }
}

// The operand a slice's epilogue adds to (residual, skip accumulator, residual stream, coupling target): pointer to
// its first element and the stride between channels; false when the mode reads nothing (or reads `out`, see EPI_MRF).
template <int MODE>
__device__ __forceinline__ bool tc16_epilogue_operand(const ConvArgs& a, int b, int t, int co0, const float*& ptr, long long& step) {
  const ConvEpilogue& e = a.ep;
  const size_t Ts = (size_t)a.T;
  const size_t row = (size_t)b * (size_t)e.out_bs + (size_t)t;
  step = (long long)Ts;
  switch (MODE) {
    case EPI_RESID:
    case EPI_MRF:
      ptr = e.resid + row + (size_t)co0 * Ts;
      return true;
    case EPI_RES_SKIP:
      if (!e.last && co0 < e.H) { ptr = e.x + row + (size_t)co0 * Ts; return true; }
      if (e.skip_init) return false;
      ptr = e.skip + row + (size_t)(e.last ? co0 : co0 - e.H) * Ts;
      return true;
    case EPI_COUPLING:
      ptr = e.out + row + (size_t)(e.z_c0 + co0 * e.z_cstep) * Ts;
      step = (long long)e.z_cstep * (long long)Ts;
      return true;
    default:
      return false;
  }
}

// issue the loads of one slice's operand (row t, channels co0 .. co0+15) into r; zeros where nothing is read
template <int MODE>
__device__ __forceinline__ void tc16_epilogue_preload(const ConvArgs& a, bool active, int b, int t, int co0, float (&r)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) r[i] = 0.f;
  const float* ptr = nullptr;
  long long step;
  if (active && t < a.T && co0 < a.Cout && tc16_epilogue_operand<MODE>(a, b, t, co0, ptr, step)) ld_strided<16>(ptr, step, min(16, a.Cout - co0), r);
}

// tc16_epilogue_slice with the operand already in registers (r[i] = 0 where it was not read): the loads were issued before
// the accumulators were waited for, so their latency overlaps the last MMAs instead of sitting between TMEM and the stores.
template <int MODE>
__device__ __forceinline__ void tc16_epilogue_slice_r(const ConvArgs& a, int b, int t, int co0, float* v, float msk, const float (&r)[16]) {
  const ConvEpilogue& e = a.ep;
  const size_t Ts = (size_t)a.T;
  const long long step = (long long)Ts;
  const size_t row = (size_t)b * (size_t)e.out_bs + (size_t)t;
  const int nval = min(16, a.Cout - co0);
  float x[16];
  switch (MODE) {
    case EPI_RESID: {
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = v[i] + r[i];
      st_strided<16>(e.out + row + (size_t)co0 * Ts, step, nval, x);
      break;
    }
    case EPI_MRF: {
      float* op = e.out + row + (size_t)co0 * Ts;
      float o[16];
      // one code path for "accumulate" (acc_mode 1: dv = 1, x / 1 == x bit for bit) and "accumulate and average" (2): a
      // three-way branch on acc_mode here made ptxas version the whole persistent loop and move the MMA descriptors through
      // predicated R2UR.BROADCAST in this instantiation (170 R2UR, 20 UTCHMMA; now 60 / 14 like the other modes)
      const float dv = (e.acc_mode == 2) ? e.div : 1.0f;
      if (e.acc_mode != 0) ld_strided<16>(op, step, nval, o);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        x[i] = v[i] + r[i];
        if (e.acc_mode != 0) x[i] = (o[i] + x[i]) / dv;
      }
      st_strided<16>(op, step, nval, x);
      break;
    }
    case EPI_RES_SKIP: {
      if (!e.last && co0 < e.H) {
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = (r[i] + v[i]) * msk;
        st_strided<16>(e.x + row + (size_t)co0 * Ts, step, nval, x);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = e.skip_init ? v[i] : r[i] + v[i];
        st_strided<16>(e.skip + row + (size_t)(e.last ? co0 : co0 - e.H) * Ts, step, nval, x);
      }
      break;
    }
    case EPI_COUPLING: {
      const float zsgn = e.z_forward ? -1.f : 1.f;   // forward direction: v * -1 (exact); inverse: v * 1 == v bit for bit
#pragma unroll
      for (int i = 0; i < 16; ++i) x[i] = (r[i] - (v[i] * zsgn) * msk) * msk;
      st_strided<16>(e.out + row + (size_t)(e.z_c0 + co0 * e.z_cstep) * Ts, (long long)e.z_cstep * (long long)Ts, nval, x);
      break;
    }
    default:
      tc16_epilogue_slice<MODE>(a, b, t, co0, v, msk);
      break;
  }
}

// Warp-specialised persistent kernel with THREADS threads (8 or 16 warps).  The last warp owns the
// tensor pipe during the main loop: one elected lane issues the weight bulk copies and every
// tcgen05.mma / tcgen05.commit; the other warps stage activations.  The roles meet only at mbarriers
// (a_full / a_free per activation buffer, b_full / b_free per weight buffer, acc per work item) --
// there is no CTA-wide barrier inside an item, so staging of the next tile, the MMAs of the current
// one and other warps' loads overlap.  All warps then share the epilogue.
// THREADS = 256 runs 2 CTAs/SM (256 TMEM columns each), THREADS = 512 one CTA/SM (512 columns).
// MODE = the epilogue (EpiMode) as a template parameter: one lean, branch-free epilogue per instantiation (a run-time switch
// inlined next to the operand preload tripled the kernel's code and spilled registers into the MMA issue loop).
template <int THREADS, int MIN_CTAS, int MODE>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) conv1d_tc16_kernel(const TcConvArgs p) {
  // The issue loop of tcgen05.mma is software-bound (~115 cycles per MMA measured with clock64 timers:
  // descriptor arithmetic + R2UR moves on one warp), and with N = 32..64 there are 36-84 MMAs per tile,
  // so NI warps issue, each owning the tiles g with g % NI == its index (an accumulator is therefore
  // always fed, in order, by the same warp).
  constexpr int NI = 1;   // 2 deadlocks on hardware (an issuer commit never lands; see DESIGN.md); kept parametric
  constexpr int STAGERS = THREADS - 32 * NI;   // threads that stage activations
  constexpr int FIRST_MMA_WARP = THREADS / 32 - NI;
  extern __shared__ __align__(128) uint8_t smem[];
  const ConvArgs& a = p.c;
  // Issue-path hygiene (see DESIGN.md 4.1 "Issue path"; verified in SASS: UTCHMMA operands without R2UR):
  //  * warp index and TMEM base are rebuilt from warp votes (provably uniform);
  //  * mbarrier waits are single asm statements (tc_prims.cuh);
  //  * the MMA warp and the staging warps keep SEPARATE pipeline counters (a_count / a_count_s): a variable
  //    that is also updated inside the thread-dependent staging loops is "divergent" for the compiler, and
  //    through it every descriptor of the MMA loop was (308 predicated R2UR before, 2 after).
  const int tid = threadIdx.x, lane = tid & 31, warp = (int)uniform_bits((uint32_t)(tid >> 5), 0, 4);
  const int K = a.K, dil = a.dil, T = a.T;
  const int N = p.N, KC = p.KC, MB = p.MB, MT = 128 * p.MB;
  const int R = MT + (K - 1) * dil;
  const int Rp = p.R_pad;
  const uint32_t a_half = (uint32_t)(KC / 8) * Rp * 16;       // bytes of one hi or lo' activation tile ([KC/8][Rp][8 halfs])
  const uint32_t a_bytes = 2 * a_half;
  const uint32_t b_bytes = (uint32_t)K * (KC / 8) * 2 * N * 16;   // one weight tile: [tap][KC/8][hi | lo' : 2N rows][8 halfs]
  const int nb = p.n_bbuf, na = p.n_abuf;
  const uint32_t tmem_cols = (uint32_t)p.tmem_cols;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 112);
  float* addv = reinterpret_cast<float*>(smem + 128);  // [2][N] bias + conditioning of the current item
  uint8_t* A0 = smem + 128 + 2 * 256 * 4;
  uint8_t* B0 = A0 + (size_t)na * a_bytes;
  const uint32_t bar_a_free = smem_u32(&bars[0]);   // [4]  MMA -> workers: activation buffer reusable
  const uint32_t bar_b_full = smem_u32(&bars[4]);   // [2]  TMA -> MMA: weight tile landed
  const uint32_t bar_b_free = smem_u32(&bars[6]);   // [2]  MMA -> MMA: weight buffer reusable
  const uint32_t bar_acc = smem_u32(&bars[8]);      //      MMA -> workers: accumulators complete
  const uint32_t bar_a_full = smem_u32(&bars[9]);   // [4]  workers -> MMA: activation tile staged
  const uint32_t A_addr = smem_u32(A0), B_addr = smem_u32(B0);

  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_slot), tmem_cols);
  }
  if (tid == 0) {
    for (int i = 0; i < 6; ++i) mbar_init(smem_u32(&bars[i]), 1);   // a_free[4], b_full[2]
    mbar_init(bar_b_free, NI);                                       // every issuer commits per chunk
    mbar_init(bar_b_free + 8, NI);
    mbar_init(bar_acc, NI);                                          // every issuer commits per item
    for (int i = 0; i < 4; ++i) mbar_init(bar_a_full + 8 * i, STAGERS / 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // Every CTA runs the same sequence of equally long items (stage -> MMAs -> epilogue): started together they hit DRAM
  // in the same bursts and leave it idle during the MMAs.  A start-up offset per CTA spreads the phases over time.
  if (p.stagger > 0) spin_cycles(((long long)(blockIdx.x & 7) * p.stagger) >> 3);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_bits(*tmem_slot, 5, 9);

  const int G = p.G;
  const int group_rows = G * MT;
  const int n_groups = (T + group_rows - 1) / group_rows;
  const int items_per_nt = a.B * n_groups;
  const int n_items = items_per_nt * p.n_tiles;

  // item -> (N tile, utterance, first row).  Layers whose weights stream per item anyway (several chunks) run the N tiles
  // of one row block in consecutive items, i.e. on neighbouring CTAs at the same time: the tiles read the same activation
  // rows, which then come from DRAM once (ncu, in_layer of the flow: 443 MB read for a 126 MB tensor in N-tile-major order).
  auto decode_item = [&](int it, int& nt_, int& b_, int& t0_) {
    int rem;
    if (p.nt_minor) {
      rem = it / p.n_tiles;
      nt_ = it - rem * p.n_tiles;
    } else {
      nt_ = it / items_per_nt;
      rem = it - nt_ * items_per_nt;
    }
    b_ = rem / n_groups;
    t0_ = (rem - b_ * n_groups) * group_rows;
  };

  // role-private pipeline state
  uint32_t b_loads0 = 0, b_loads1 = 0, b_count = 0;   // MMA lane
  // activation ring of na (1, 2 or 4) buffers used round-robin: buffer = count & (na - 1), earlier uses = count >> na_log
  const uint32_t na_mask = (uint32_t)na - 1u, na_log = (na == 4) ? 2u : (na == 2 ? 1u : 0u);
  int b_resident_nt = -1;
  uint32_t a_count = 0, a_count_s = 0, acc_count = 0, item_count = 0;
  const uint32_t idesc_n = idesc_f16_m128(N), idesc_2n = idesc_f16_m128(2 * N);
  const uint32_t a_lo_delta = a_half >> 4;
  const int nb16 = KC / 16;                 // KC is a multiple of 16 (one tcgen05.mma k-step)

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    int nt, b, t_group0;
    decode_item(item, nt, b, t_group0);
    // length-aware mode: a group wholly beyond (len + margin) frames runs with zero tiles (no staging, no MMAs, empty
    // epilogue; the per-item barriers still tick).  A select, not a branch (SASS-checked: a `continue` here, or votes
    // on the tile count, cost the issue loop its uniform datapath: R2UR 19 -> 162).
    int tiles = min(G, (T - t_group0 + MT - 1) / MT);
    if (a.la_len) tiles = ((long long)t_group0 >= (a.la_len[b] + a.la_margin) * (long long)a.la_rate) ? 0 : tiles;
    // a zero-tile item must not touch the weight pipeline either (the next chunk's prefetch is issued from inside the
    // tile loop): it runs zero chunks; only the per-item barriers tick
    const int n_chunks_item = (tiles > 0) ? p.n_chunks : 0;
    const long long len = a.lengths ? a.lengths[b] : (long long)T;
    // per-item additive term of every output channel (bias + speaker conditioning), double buffered
    float* av = addv + (item_count & 1) * 256;
    for (int n = tid; n < N; n += THREADS) {
      const int co = nt * N + n;
      float x = 0.f;
      if (co < a.Cout) {
        if (a.bias) x = a.bias[co];
        if (a.ep.cond) {
          const float* gp = a.ep.cond + (long long)b * a.ep.cond_bs + a.ep.cond_off;
          if (MODE == EPI_GATE) x += (co & 1) ? gp[a.ep.H + (co >> 1)] : gp[co >> 1];
          else if (MODE == EPI_PLAIN) x += gp[co];
        }
      }
      av[n] = x;
    }
    item_count += 1;
    // the previous item's TMEM reads (all warps) are ordered before this item's first MMA
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp >= FIRST_MMA_WARP) {
      // ============ tensor-pipe warps: uniform control flow, one elected lane per warp issues ============
      constexpr int iw = 0;   // NI == 1: the issuer index is a constant, not a function of the warp index
      static_assert(NI == 1, "one issuing warp");
      {
        for (int c = 0; c < n_chunks_item; ++c) {
          int bb = 0;
          bool load_b = true;
          if (p.n_chunks == 1) {
            load_b = (b_resident_nt != nt);
            b_resident_nt = nt;
          } else {
            bb = (nb == 2) ? (int)(b_count & 1) : 0;
          }
          // Weight tiles.  Single-chunk layers: one resident tile, reloaded only when the item's N tile
          // changes (the previous item's MMAs are complete: bar_acc + the item barrier).  Multi-chunk
          // layers: two buffers; chunk c+1 is requested as soon as the first tile of chunk c has been
          // issued (its buffer was last read by chunk c-1, whose commit we wait for), so the bulk copy
          // overlaps the remaining tiles of chunk c.
          auto issue_b_load = [&](int chunk, int buf, uint32_t loads_before) {
            if (iw == 0 && p.n_chunks > 1 && loads_before > 0) mbar_wait(bar_b_free + 8 * buf, (loads_before - 1) & 1);
            const uint8_t* src = reinterpret_cast<const uint8_t*>(p.wtc) + ((size_t)nt * p.n_chunks + chunk) * b_bytes;
            if (iw == 0 && elect_one()) {
              mbar_expect_tx(bar_b_full + 8 * buf, b_bytes);
              uint32_t off = 0;
              while (off < b_bytes) {
                const uint32_t n = min(b_bytes - off, 32768u);
                bulk_g2s(B_addr + buf * b_bytes + off, src + off, n, bar_b_full + 8 * buf);
                off += n;
              }
            }
            __syncwarp();
          };
          bool prefetched = false;
          if (p.n_chunks > 1) {
            load_b = true;
            if (c > 0 && nb == 2) prefetched = true;  // requested during the previous chunk
          }
          if (load_b && !prefetched) issue_b_load(c, bb, bb ? b_loads1 : b_loads0);
          bool b_ready = !load_b;
          for (int g = 0; g < tiles; ++g) {
            const int ab = (int)(a_count & na_mask);
            if (g % NI != iw) {   // another issuer's tile: only keep the pipeline counters in step
              a_count += 1;
              if (g == 0 && nb == 2 && c + 1 < p.n_chunks) { const int ob = bb ^ 1; issue_b_load(c + 1, ob, ob ? b_loads1 : b_loads0); }
              continue;
            }
            mbar_wait(bar_a_full + 8 * ab, (a_count >> na_log) & 1);
            if (!b_ready) { mbar_wait(bar_b_full + 8 * bb, (bb ? b_loads1 : b_loads0) & 1); b_ready = true; }
            tc_fence_after();
            const uint64_t adesc0 = make_desc(A_addr + ab * a_bytes, (uint32_t)Rp * 16, 128);
            const uint64_t bdesc0 = make_desc(B_addr + bb * b_bytes, (uint32_t)(2 * N) * 16, 128);
            const uint32_t alo0 = (uint32_t)adesc0, blo0 = (uint32_t)bdesc0;
            for (int mb = 0; mb < MB; ++mb) {
              const uint32_t d_tmem = tmem_base + (uint32_t)((g * MB + mb) * 2 * N);
              for (int tap = 0; tap < K; ++tap) {
                uint32_t al = alo0 + (uint32_t)(mb * 128 + tap * dil);                 // 16 B units
                uint32_t bl = blo0 + (uint32_t)tap * (uint32_t)((KC / 8) * 2 * N);
                for (int kk = 0; kk < KC / 16; ++kk) {
                  const uint32_t first = (c == 0 && tap == 0 && kk == 0) ? 0u : 1u;
                  tc_mma_f16_split2(d_tmem, d_tmem + (uint32_t)N, desc_with_lo(adesc0, al), desc_with_lo(adesc0, al + a_lo_delta),
                                    desc_with_lo(bdesc0, bl), idesc_2n, idesc_n, first);
                  al += 2u * (uint32_t)Rp;
                  bl += 2u * (uint32_t)(2 * N);
                }
              }
            }
            if (elect_one()) tc_commit(bar_a_free + 8 * ab);
            __syncwarp();
            a_count += 1;
            if (g == 0 && nb == 2 && c + 1 < p.n_chunks) {
              // prefetch the next chunk's weights into the other buffer (loads counted when consumed)
              const int ob = bb ^ 1;
              issue_b_load(c + 1, ob, ob ? b_loads1 : b_loads0);
            }
          }
          // every issuer reports "my MMAs that read this weight buffer are done" (also when it had no tile)
          if (p.n_chunks > 1 && elect_one()) tc_commit(bar_b_free + 8 * bb);
          __syncwarp();
          if (load_b) { if (bb) b_loads1 += 1; else b_loads0 += 1; }
          if (p.n_chunks > 1) b_count += 1;
        }
        if (elect_one()) tc_commit(bar_acc);
        __syncwarp();
      }
    } else {
      // =========================== staging warps ===========================
      const int Tin = a.in_T > 0 ? a.in_T : T;
      const int t_hi = a.in_mask ? (int)(len < Tin ? len : Tin) : Tin;
      const float* in_b = a.in + (long long)b * a.in_bs;
      const long long in_cs = a.in_cs;
      if (p.l2_prefetch) {
        // (1) the activation rows of this CTA's NEXT item: its staging loads (16 per thread and round, one round trip per
        // chunk on the critical path of the MMAs) then hit L2; (2) what this item's epilogue reads back.
        const int nxt = item + (int)gridDim.x;
        if (nxt < n_items) {
          int nt_n, b_n, t0_n;
          decode_item(nxt, nt_n, b_n, t0_n);
          const long long len_n = a.lengths ? a.lengths[b_n] : (long long)T;
          const int t_hi_n = a.in_mask ? (int)(len_n < Tin ? len_n : Tin) : Tin;
          const int lo = max(0, t0_n - a.pad_left), hi = min(t_hi_n, t0_n - a.pad_left + G * MT + (K - 1) * dil);
          l2_prefetch_rows(a.in + (long long)b_n * a.in_bs, a.in_cs, a.Cin, lo, hi, tid, STAGERS);
        }
        const ConvEpilogue& e = a.ep;
        const int c_lo = nt * N, c_hi = min(a.Cout, nt * N + N);
        const int r_lo = t_group0, r_hi = min(T, t_group0 + tiles * MT);
        const long long ob = (long long)b * e.out_bs;
        if (MODE == EPI_RESID || MODE == EPI_MRF) {
          l2_prefetch_rows(e.resid + ob + (long long)c_lo * T, T, c_hi - c_lo, r_lo, r_hi, tid, STAGERS);
          if (MODE == EPI_MRF && e.acc_mode != 0) l2_prefetch_rows(e.out + ob + (long long)c_lo * T, T, c_hi - c_lo, r_lo, r_hi, tid, STAGERS);
        } else if (MODE == EPI_RES_SKIP) {
          if (!e.last && c_lo < e.H) l2_prefetch_rows(e.x + ob + (long long)c_lo * T, T, min(c_hi, e.H) - c_lo, r_lo, r_hi, tid, STAGERS);
          if (!e.skip_init && (e.last || c_hi > e.H)) {
            const int s_lo = e.last ? c_lo : max(c_lo, e.H) - e.H, s_hi = e.last ? c_hi : c_hi - e.H;
            l2_prefetch_rows(e.skip + ob + (long long)s_lo * T, T, s_hi - s_lo, r_lo, r_hi, tid, STAGERS);
          }
        } else if (MODE == EPI_COUPLING) {
          l2_prefetch_rows(e.out + ob + (long long)(e.z_c0 + c_lo * e.z_cstep) * T, (long long)e.z_cstep * T, c_hi - c_lo, r_lo, r_hi, tid, STAGERS);
        }
      }
      for (int c = 0; c < n_chunks_item; ++c) {
        const int c0 = c * KC;
        const bool fast = (a.Cin - c0) >= KC;
        for (int g = 0; g < tiles; ++g) {
          const int ab = (int)(a_count_s & na_mask);
          const uint32_t a_uses = a_count_s >> na_log;
          uint8_t* Ah = A0 + (size_t)ab * a_bytes;
          const int t_in0 = t_group0 + g * MT - a.pad_left;
          bool waited = (a_uses == 0);
          // two (row, 16-channel) items per round: 32 independent global loads per thread in flight
          int q16 = 0, r = tid;
          while (r >= Rp) { r -= Rp; ++q16; }
          if (p.debug_skip & 1) q16 = nb16;
          while (q16 < nb16) {
            int q16b = q16, rb = r + STAGERS;
            while (rb >= Rp) { rb -= Rp; ++q16b; }
            const bool has_b = q16b < nb16;
            float v[2][16];
            int rr[2] = {r, rb}, qq[2] = {q16, q16b};
            // unit b under a branch, not a predicate: warps without a second unit (all of them when one round covers the
            // tile, e.g. 264 rows x 16 channels on 480 threads) skip its 16 address + load instructions
            auto load_unit = [&](int u2) {
              const int t = t_in0 + rr[u2];
              const bool rok = (rr[u2] < R) && (t >= 0) && (t < t_hi);
              const int ci0 = c0 + qq[u2] * 16;
              const float* src = in_b + (long long)ci0 * a.in_cs + t;
              if (fast) {      // one 64-bit add per load instead of a 64-bit multiply-add (issue-bound kernel)
                const float* sp = src;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  v[u2][e] = rok ? __ldg(sp) : 0.f;
                  sp += in_cs;
                }
              } else {
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  v[u2][e] = 0.f;
                  if (rok && (ci0 + e) < a.Cin) v[u2][e] = __ldg(src + (long long)e * a.in_cs);
                }
              }
            };
            load_unit(0);
            if (has_b) load_unit(1);
            if (!waited) {  // the MMAs that last read this buffer must be done before it is overwritten
              mbar_wait(bar_a_free + 8 * ab, (a_uses - 1) & 1);
              waited = true;
            }
#pragma unroll
            for (int u2 = 0; u2 < 2; ++u2) {
              if (u2 == 1 && !has_b) break;
#pragma unroll
              for (int g8 = 0; g8 < 2; ++g8) {
                float x[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  x[e] = v[u2][g8 * 8 + e];
                  if (a.pre_act) x[e] = x[e] > 0.f ? x[e] : x[e] * a.pre_slope;
                }
                uint4 hi, lo;
                f16_split2(x[0], x[1], hi.x, lo.x);
                f16_split2(x[2], x[3], hi.y, lo.y);
                f16_split2(x[4], x[5], hi.z, lo.z);
                f16_split2(x[6], x[7], hi.w, lo.w);
                const size_t o = ((size_t)(qq[u2] * 2 + g8) * Rp + rr[u2]) * 16;
                *reinterpret_cast<uint4*>(Ah + o) = hi;
                *reinterpret_cast<uint4*>(Ah + a_half + o) = lo;
              }
            }
            r = rb + STAGERS;
            q16 = q16b;
            while (r >= Rp) { r -= Rp; ++q16; }
          }
          if (!waited) mbar_wait(bar_a_free + 8 * ab, (a_uses - 1) & 1);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_a_full + 8 * ab);
          a_count_s += 1;
        }
      }
    }
    // ---------------- fused epilogue (all warps).  A thread owns one TMEM lane (output row) per M block and ncol columns:
    // G * MB * ncol / 16 = 4 slices of 16 channels per item whenever TMEM is fully used (every plan).
    {
      constexpr int COLSPLIT = THREADS / 128;     // warps sharing a TMEM lane quarter split the columns
      const int q = warp & 3, part = warp >> 2;
      const int ncol = N / COLSPLIT;
      const int spb = ncol >> 4;                  // slices per M block (1, 2 or 4)
      const int n_slices = ((p.debug_skip & 2) ? 0 : tiles) * MB * spb;
      // What the epilogue adds to is requested early: slices 0 and 1 BEFORE the accumulators are waited for (the loads
      // overlap the last MMAs), slices 2 and 3 as soon as the registers of slices 0 and 1 are free (two register sets:
      // four would spill).
      float R[2][16];
      const bool pre = p.epi_preload && n_slices <= 4;
      const int row0 = t_group0 + q * 32 + lane, colbase = nt * N + part * ncol;
#pragma unroll
      for (int sl = 0; sl < 2; ++sl) {
        const int blk = sl / spb, cs = sl - blk * spb;            // (g * MB + mb) * 128 == g * MT + mb * 128
        tc16_epilogue_preload<MODE>(a, pre && sl < n_slices, b, row0 + blk * 128, colbase + cs * 16, R[sl]);
      }
      mbar_wait(bar_acc, acc_count & 1);
      acc_count += 1;
      tc_fence_after();
#pragma unroll 1
      for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int sl = 2 * h + k;
        if (sl < n_slices) {
          const int blk = sl / spb, cs = sl - blk * spb;
          const int t = row0 + blk * 128;
          const float msk = (t < len) ? 1.f : 0.f;
          const int nl = part * ncol + cs * 16;
          const uint32_t col0 = (uint32_t)(blk * 2 * N + nl);
          float v[16], vs[16];
          tmem_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + col0, v);
          tmem_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + col0 + (uint32_t)N, vs);
          tmem_ld_wait();
          const float4* a4 = reinterpret_cast<const float4*>(av + nl);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 x = a4[i];
            v[4 * i + 0] = (v[4 * i + 0] + vs[4 * i + 0] * kF16LoInv) + x.x;
            v[4 * i + 1] = (v[4 * i + 1] + vs[4 * i + 1] * kF16LoInv) + x.y;
            v[4 * i + 2] = (v[4 * i + 2] + vs[4 * i + 2] * kF16LoInv) + x.z;
            v[4 * i + 3] = (v[4 * i + 3] + vs[4 * i + 3] * kF16LoInv) + x.w;
          }
          if (t < T && nt * N + nl < a.Cout) {
            if (!pre) tc16_epilogue_preload<MODE>(a, true, b, t, nt * N + nl, R[k]);     // not requested ahead: load now
            tc16_epilogue_slice_r<MODE>(a, b, t, nt * N + nl, v, msk, R[k]);
          }
        }
        if (h == 0) {   // this register set is free: request the operand of slice sl + 2
          const int blk = (sl + 2) / spb, cs = (sl + 2) - blk * spb;
          tc16_epilogue_preload<MODE>(a, pre && (sl + 2) < n_slices, b, row0 + blk * 128, colbase + cs * 16, R[k]);
        }
      }
      // (plans that leave TMEM partly unused would have more than 4 slices: none exists; they would take this loop)
      for (int sl = 4; sl < n_slices; ++sl) {
        const int blk = sl / spb, cs = sl - blk * spb;
        const int t = t_group0 + blk * 128 + q * 32 + lane;
        const float msk = (t < len) ? 1.f : 0.f;
        const int nl = part * ncol + cs * 16;
        const uint32_t col0 = (uint32_t)(blk * 2 * N + nl);
        float v[16], vs[16];
        tmem_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + col0, v);
        tmem_ld16_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + col0 + (uint32_t)N, vs);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = (v[i] + vs[i] * kF16LoInv) + av[nl + i];
        if (t < T && nt * N + nl < a.Cout) tc16_epilogue_slice<MODE>(a, b, t, nt * N + nl, v, msk);
      }
    }
  }
  __syncthreads();
  if (warp == 0) {
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------ weight packing
// dst (halfs) [nt][chunk][tap][kg = KC/8][hl: hi rows 0..N-1, lo' rows N..2N-1][8] from the folded weight src[co][ci][tap]
__global__ void pack_conv_tc16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, const int* __restrict__ co_map,
                                      const int* __restrict__ ci_map, int Cout, int Cin, int K, int src_cin, int N,
                                      int n_tiles, int KC, int n_chunks) {
  const long long total = (long long)n_tiles * n_chunks * K * (KC / 8) * 2 * N * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int e = (int)(r % 8); r /= 8;
    const int n = (int)(r % N); r /= N;
    const int hl = (int)(r % 2); r /= 2;
    const int kg = (int)(r % (KC / 8)); r /= (KC / 8);
    const int tap = (int)(r % K); r /= K;
    const int chunk = (int)(r % n_chunks); r /= n_chunks;
    const int nt = (int)r;
    const int co_p = nt * N + n, ci_p = chunk * KC + kg * 8 + e;
    float w = 0.f;
    if (co_p < Cout && ci_p < Cin) {
      const int co = co_map[co_p];
      const int ci = ci_map ? ci_map[ci_p] : ci_p;
      if (co >= 0) w = src[((long long)co * src_cin + ci) * K + tap];
    }
    uint32_t hi2, lo2;
    f16_split2(w, 0.f, hi2, lo2);
    dst[i] = (uint16_t)((hl ? lo2 : hi2) & 0xFFFFu);
  }
}

}  // namespace

size_t tc16_conv_smem_bytes(int K, int dil, int N, int KC, int MB, int n_abuf, int n_bbuf) {
  const int R = 128 * MB + (K - 1) * dil;
  const int Rp = (R + 7) & ~7;
  return 128 + 2048 + (size_t)n_abuf * (2 * (size_t)(KC / 8) * Rp * 16) + (size_t)n_bbuf * ((size_t)K * (KC / 8) * 2 * N * 16);
}

// Tiling for the f16 form.  An accumulator block takes 2N TMEM columns ([hi*hi | small terms]), and 2N <= 256 is also
// the widest MMA, so N <= 128.  mode 0 ("small"): <= 110 KB shared memory, 256 columns, 256 threads, two CTAs per SM,
// whole C_in in one chunk (weights stay resident).  mode 1 ("large"): <= 216 KB, 512 columns, 512 threads, one CTA
// per SM, C_in chunked with double-buffered weight tiles.
bool tc16_conv_plan(int Cin, int Cout, int K, int dil, TcPlan* plan) {
  if (Cin < 16 || Cout < 16) return false;
  const int cin16 = (Cin + 15) / 16 * 16;
  const int cout32 = (Cout + 31) / 32 * 32;
  auto fill = [&](int mode, int N, int n_tiles, int KC, int MB, int na, int nb) {
    const int R = 128 * MB + (K - 1) * dil;
    plan->mode = mode; plan->N = N; plan->n_tiles = n_tiles; plan->KC = KC; plan->n_chunks = (cin16 + KC - 1) / KC;
    plan->MB = MB; plan->tmem_cols = mode == 0 ? 256 : 512; plan->G = plan->tmem_cols / (MB * 2 * N);
    plan->n_abuf = na; plan->n_bbuf = nb; plan->R_pad = (R + 7) & ~7; plan->dil = dil;
    plan->packed_floats = (size_t)n_tiles * plan->n_chunks * K * (KC / 8) * 2 * N * 8;   // in HALFS for this format
  };
  // ---- small mode
  if (cout32 <= 128) {
    const int N = cout32;
    for (int na = 2; na >= 1; --na)
      for (int MB = 2; MB >= 1; --MB) {
        if (MB * 2 * N > 256) continue;
        if (tc16_conv_smem_bytes(K, dil, N, cin16, MB, na, 1) <= 112 * 1024) {
          fill(0, N, 1, cin16, MB, na, 1);
          return true;
        }
      }
  }
  // ---- mode 2 ("two CTAs", WETTS_TC16_TWO_CTAS=1 at load time): the large-mode tiling with one M block per item, 256 TMEM
  // columns, 256 threads and <= 112 KB, so that two CTAs share an SM and one's MMAs run during the other's staging and
  // epilogue (the phases of an item cannot overlap inside a CTA: its accumulators fill its TMEM).  Costs twice the weight
  // stream per output row.
  // Policy (measured per layer, profiles/r02o_*): it pays where the activations are re-staged for many N tiles and the
  // weights of one N tile are small enough to stream twice as often -- three or more N tiles, or two with K * C_in <= 512
  // (flow in_layer 0.48 -> 0.415 ms, text-encoder convs -11 %); single-tile and heavy layers (C=128 / C=256 resblocks)
  // lose 10 % and stay in the large mode.  WETTS_TC16_TWO_CTAS = 0 never, 1 wherever it fits, 2 (default) the policy.
  static const int two_ctas = getenv("WETTS_TC16_TWO_CTAS") ? atoi(getenv("WETTS_TC16_TWO_CTAS")) : 2;
  const int nt128 = ((Cout + 63) / 64 * 64 + 127) / 128;
  if (two_ctas == 1 || (two_ctas == 2 && (nt128 >= 3 || (nt128 == 2 && K * cin16 <= 512)))) {
    const int cout64b = (Cout + 63) / 64 * 64;
    for (int n_tiles = (cout64b + 127) / 128; n_tiles <= cout64b / 64; ++n_tiles) {
      const int N = ((cout64b + n_tiles - 1) / n_tiles + 63) / 64 * 64;
      if (N > 128) continue;
      for (int nch = 1; nch <= cin16 / 16; ++nch) {
        const int KC = ((cin16 + nch - 1) / nch + 15) / 16 * 16;
        const int nb = (cin16 + KC - 1) / KC == 1 ? 1 : 2;
        if (tc16_conv_smem_bytes(K, dil, N, KC, 1, 2, nb) <= 112 * 1024) {
          fill(1, N, n_tiles, KC, 1, 2, nb);
          plan->mode = 2; plan->tmem_cols = 256; plan->G = 256 / (2 * N);
          return true;
        }
      }
    }
  }
  // ---- large mode (N a multiple of 64 so that 16 warps split the columns in 16-wide pieces)
  // WETTS_TC16_NMAX=64 (read once, at load time): 64-wide N tiles, so that two items' accumulators fit in TMEM and the
  // pipelined kernel can drain one while the MMAs of the next run
  static const int n_max = getenv("WETTS_TC16_NMAX") ? atoi(getenv("WETTS_TC16_NMAX")) : 128;
  const int cout64 = (Cout + 63) / 64 * 64;
  for (int n_tiles = (cout64 + n_max - 1) / n_max; n_tiles <= cout64 / 64; ++n_tiles) {
    const int N = ((cout64 + n_tiles - 1) / n_tiles + 63) / 64 * 64;
    if (N > n_max) continue;
    for (int MB = 2; MB >= 1; --MB) {
      if (MB * 2 * N > 512) continue;
      for (int nch = 1; nch <= cin16 / 16; ++nch) {
        const int KC = ((cin16 + nch - 1) / nch + 15) / 16 * 16;
        const int nb = (cin16 + KC - 1) / KC == 1 ? 1 : 2;
        if (tc16_conv_smem_bytes(K, dil, N, KC, MB, 2, nb) <= 216 * 1024) {
          // a deeper activation ring hides the latency of the staging loads (the MMAs of a chunk are shorter than
          // one round trip to L2); WETTS_TC16_ABUF=2 keeps the double buffer (experiments)
          static const int max_na = getenv("WETTS_TC16_ABUF") ? atoi(getenv("WETTS_TC16_ABUF")) : 2;   // 4: opt-in until measured
          const int na = (max_na >= 4 && nb == 2 && tc16_conv_smem_bytes(K, dil, N, KC, MB, 4, nb) <= 216 * 1024) ? 4 : 2;
          fill(1, N, n_tiles, KC, MB, na, nb);
          return true;
        }
      }
    }
  }
  return false;
}

void launch_pack_conv_tc16(const float* src, void* dst, const int* co_map, const int* ci_map, int Cout, int Cin, int K,
                           int src_cin, const TcPlan& pl, cudaStream_t s) {
  const long long total = (long long)pl.packed_floats;
  const int blocks = (int)((total + 255) / 256 > 8192 ? 8192 : (total + 255) / 256);
  pack_conv_tc16_kernel<<<blocks, 256, 0, s>>>(src, reinterpret_cast<uint16_t*>(dst), co_map, ci_map, Cout, Cin, K, src_cin, pl.N,
                                               pl.n_tiles, pl.KC, pl.n_chunks);
  count_launch();
}

void launch_conv1d_tc16(const ConvArgs& a, cudaStream_t s) {
  if (tc16r_enabled() && launch_conv1d_tc16r(a, s)) return;
  if (tc16p_enabled() && launch_conv1d_tc16p(a, s)) return;
  const TcPlan& pl = a.tc16;
  TcConvArgs p;
  p.c = a;
  p.wtc = reinterpret_cast<const float*>(a.wtc16);
  // the packed layout depends on (N, KC, n_chunks) only; M-blocks per tile are chosen per launch
  const int MB = (a.T > 128 && pl.MB == 2) ? 2 : 1;
  const int R = 128 * MB + (a.K - 1) * a.dil;
  p.N = pl.N; p.n_tiles = pl.n_tiles; p.KC = pl.KC; p.n_chunks = pl.n_chunks; p.MB = MB;
  p.tmem_cols = pl.tmem_cols; p.G = pl.tmem_cols / (MB * 2 * pl.N);
  p.n_abuf = pl.n_abuf; p.n_bbuf = pl.n_bbuf; p.R_pad = (R + 7) & ~7;
  const size_t smem = tc16_conv_smem_bytes(a.K, a.dil, pl.N, pl.KC, MB, pl.n_abuf, pl.n_bbuf);
  static const int opt_nt_minor = getenv("WETTS_TC16_NTMINOR") ? atoi(getenv("WETTS_TC16_NTMINOR")) : 1;
  static const int opt_prefetch = getenv("WETTS_TC16_PREFETCH") ? atoi(getenv("WETTS_TC16_PREFETCH")) : 1;
  p.nt_minor = (opt_nt_minor && pl.n_chunks > 1 && pl.n_tiles > 1) ? 1 : 0;
  p.l2_prefetch = opt_prefetch;
  static const int opt_skip = getenv("WETTS_TC16_DEBUG_SKIP") ? atoi(getenv("WETTS_TC16_DEBUG_SKIP")) : 0;
  p.debug_skip = opt_skip;
  static const int opt_stagger = getenv("WETTS_TC16_STAGGER") ? atoi(getenv("WETTS_TC16_STAGGER")) : 0;
  static const int opt_pre = getenv("WETTS_TC16_EPI_PRELOAD") ? atoi(getenv("WETTS_TC16_EPI_PRELOAD")) : 1;
  p.epi_preload = opt_pre;
  static DynSmemAttr attr[2][7];
  const int n_sm = current_device_sm_count();
  if (n_sm <= 0) return;
  const int group_rows = p.G * 128 * MB;
  const long long items = (long long)a.B * ((a.T + group_rows - 1) / group_rows) * pl.n_tiles;
  p.stagger = (items > 2LL * n_sm) ? opt_stagger : 0;   // only launches with several items per CTA
  const bool two = (pl.mode == 0 || pl.mode == 2);      // 256-thread CTAs, two per SM
  const int grid = (int)(two ? (items < 2 * n_sm ? items : 2 * n_sm) : (items < n_sm ? items : n_sm));
  bool ok = false;
#define WETTS_TC16_LAUNCH(M)                                                                                     \
  case M:                                                                                                        \
    if (two) {                                                                                                   \
      if (attr[0][M].ensure((const void*)conv1d_tc16_kernel<256, 2, M>, smem) != cudaSuccess) return;            \
      conv1d_tc16_kernel<256, 2, M><<<grid, 256, smem, s>>>(p);                                                  \
    } else {                                                                                                     \
      if (attr[1][M].ensure((const void*)conv1d_tc16_kernel<512, 1, M>, smem) != cudaSuccess) return;            \
      conv1d_tc16_kernel<512, 1, M><<<grid, 512, smem, s>>>(p);                                                  \
    }                                                                                                            \
    ok = true;                                                                                                   \
    break;
  switch (a.ep.mode) {
    WETTS_TC16_LAUNCH(EPI_PLAIN)
    WETTS_TC16_LAUNCH(EPI_RESID)
    WETTS_TC16_LAUNCH(EPI_MRF)
    WETTS_TC16_LAUNCH(EPI_GATE)
    WETTS_TC16_LAUNCH(EPI_RES_SKIP)
    WETTS_TC16_LAUNCH(EPI_COUPLING)
    WETTS_TC16_LAUNCH(EPI_CONVT)
    default:
      break;
  }
#undef WETTS_TC16_LAUNCH
  if (!ok) return;
  count_launch();
}

int tc16_conv_install_fault_word(unsigned int* word) { return tc::install_fault_word_tu(word) == cudaSuccess ? 0 : 1; }

}  // namespace wetts
