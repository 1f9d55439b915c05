// tcgen05 (5th-gen tensor core) implicit-GEMM Conv1d for sm_100a, fp32-accurate via 3xTF32.
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
__device__ __forceinline__ void tc_epilogue_slice(const ConvArgs& a, int b, int t, int co0, float* v, float msk) {
  const ConvEpilogue& e = a.ep;
  const size_t Ts = (size_t)a.T;
  const size_t row = (size_t)b * (size_t)e.out_bs + (size_t)t;
  const int nval = min(16, a.Cout - co0);
  switch (e.mode) {
    case EPI_PLAIN: {
      float* op = e.out + row + (size_t)co0 * Ts;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float x = v[i];
        if (e.act == 1) x = fmaxf(x, 0.f);
        else if (e.act == 2) x = gelu_erf_acc(x);
        if (e.out_mask) x *= msk;
        if (i < nval) op[(size_t)i * Ts] = x;
      }
      break;
    }
    case EPI_RESID: {
      const float* rp = e.resid + row + (size_t)co0 * Ts;
      float* op = e.out + row + (size_t)co0 * Ts;
      float r[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) r[i] = (i < nval) ? rp[(size_t)i * Ts] : 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i < nval) op[(size_t)i * Ts] = v[i] + r[i];
      break;
    }
    case EPI_MRF: {
      const float* rp = e.resid + row + (size_t)co0 * Ts;
      float* op = e.out + row + (size_t)co0 * Ts;
      float r[16], o[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) r[i] = (i < nval) ? rp[(size_t)i * Ts] : 0.f;
      if (e.acc_mode != 0) {
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] = (i < nval) ? op[(size_t)i * Ts] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float x = v[i] + r[i];
        if (e.acc_mode == 1) x = o[i] + x;
        else if (e.acc_mode == 2) x = (o[i] + x) / e.div;
        if (i < nval) op[(size_t)i * Ts] = x;
      }
      break;
    }
    case EPI_GATE: {
      float* op = e.out + row + (size_t)(co0 >> 1) * Ts;
#pragma unroll
      for (int i = 0; i < 16; i += 2)
        if (i < nval) op[(size_t)(i >> 1) * Ts] = tanhf(v[i]) * sigmoidf_acc(v[i + 1]);
      break;
    }
    case EPI_RES_SKIP: {
      if (!e.last && co0 < e.H) {  // residual stream (a 16-slice never straddles H: H % 16 == 0 is checked on the host)
        float* xp = e.x + row + (size_t)co0 * Ts;
        float r[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = (i < nval) ? xp[(size_t)i * Ts] : 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (i < nval) xp[(size_t)i * Ts] = (r[i] + v[i]) * msk;
      } else {
        float* sp = e.skip + row + (size_t)(e.last ? co0 : co0 - e.H) * Ts;
        float r[16];
        if (!e.skip_init) {
#pragma unroll
          for (int i = 0; i < 16; ++i) r[i] = (i < nval) ? sp[(size_t)i * Ts] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (i < nval) sp[(size_t)i * Ts] = e.skip_init ? v[i] : r[i] + v[i];
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
      const long long step = (long long)e.z_cstep * (long long)Ts;
      float r[16];
      const float zsgn = e.z_forward ? -1.f : 1.f;   // forward direction: v * -1 (exact); inverse: v * 1 == v bit for bit
#pragma unroll
      for (int i = 0; i < 16; ++i) r[i] = (i < nval) ? zp[(long long)i * step] : 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i < nval) zp[(long long)i * step] = (r[i] - (v[i] * zsgn) * msk) * msk;
      break;
    }
    default:
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
template <int THREADS, int MIN_CTAS>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) conv1d_tc_kernel(const TcConvArgs p) {
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
  const uint32_t a_half = (uint32_t)KC * Rp * 4;       // bytes of one hi or lo activation tile
  const uint32_t a_bytes = 2 * a_half;
  const uint32_t b_half = (uint32_t)K * KC * N * 4;    // bytes of one hi or lo weight tile
  const uint32_t b_bytes = 2 * b_half;
  const int nb = p.n_bbuf, na = p.n_abuf;
  const uint32_t tmem_cols = (uint32_t)p.tmem_cols;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 96);
  float* addv = reinterpret_cast<float*>(smem + 128);  // [2][N] bias + conditioning of the current item
  uint8_t* A0 = smem + 128 + 2 * 256 * 4;
  uint8_t* B0 = A0 + (size_t)na * a_bytes;
  const uint32_t bar_a_free = smem_u32(&bars[0]);   // [2]  MMA -> workers: activation buffer reusable
  const uint32_t bar_b_full = smem_u32(&bars[2]);   // [2]  TMA -> MMA: weight tile landed
  const uint32_t bar_b_free = smem_u32(&bars[4]);   // [2]  MMA -> MMA: weight buffer reusable
  const uint32_t bar_acc = smem_u32(&bars[6]);      //      MMA -> workers: accumulators complete
  const uint32_t bar_a_full = smem_u32(&bars[8]);   // [2]  workers -> MMA: activation tile staged
  const uint32_t A_addr = smem_u32(A0), B_addr = smem_u32(B0);

  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_slot), tmem_cols);
  }
  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(smem_u32(&bars[i]), 1);   // a_free[2], b_full[2]
    mbar_init(bar_b_free, NI);                                       // every issuer commits per chunk
    mbar_init(bar_b_free + 8, NI);
    mbar_init(bar_acc, NI);                                          // every issuer commits per item
    mbar_init(bar_a_full, STAGERS / 32);
    mbar_init(bar_a_full + 8, STAGERS / 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform_bits(*tmem_slot, 5, 9);

  const int G = p.G;
  const int group_rows = G * MT;
  const int n_groups = (T + group_rows - 1) / group_rows;
  const int items_per_nt = a.B * n_groups;
  const int n_items = items_per_nt * p.n_tiles;

  // role-private pipeline state
  uint32_t a_fills0 = 0, a_fills1 = 0, b_loads0 = 0, b_loads1 = 0, b_count = 0;   // MMA lane
  int b_resident_nt = -1;
  uint32_t a_uses0 = 0, a_uses1 = 0;                                              // stagers
  uint32_t a_count = 0, a_count_s = 0, acc_count = 0, item_count = 0;
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
  const uint32_t a_lo_delta = a_half >> 4, b_lo_delta = b_half >> 4;
  const int nb16 = (KC + 15) / 16;
  const bool full16 = (KC % 16 == 0);

  for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int nt = item / items_per_nt;
    const int rem = item - nt * items_per_nt;
    const int b = rem / n_groups;
    const int t_group0 = (rem - b * n_groups) * group_rows;
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
          if (a.ep.mode == EPI_GATE) x += (co & 1) ? gp[a.ep.H + (co >> 1)] : gp[co >> 1];
          else if (a.ep.mode == EPI_PLAIN) x += gp[co];
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
            const int ab = (na == 2) ? (int)(a_count & 1) : 0;
            if (g % NI != iw) {   // another issuer's tile: only keep the pipeline counters in step
              if (ab) a_fills1 += 1; else a_fills0 += 1;
              a_count += 1;
              if (g == 0 && nb == 2 && c + 1 < p.n_chunks) { const int ob = bb ^ 1; issue_b_load(c + 1, ob, ob ? b_loads1 : b_loads0); }
              continue;
            }
            mbar_wait(bar_a_full + 8 * ab, (ab ? a_fills1 : a_fills0) & 1);
            if (!b_ready) { mbar_wait(bar_b_full + 8 * bb, (bb ? b_loads1 : b_loads0) & 1); b_ready = true; }
            tc_fence_after();
            const uint64_t adesc0 = make_desc(A_addr + ab * a_bytes, (uint32_t)Rp * 16, 128);
            const uint64_t bdesc0 = make_desc(B_addr + bb * b_bytes, (uint32_t)N * 16, 128);
            const uint32_t alo0 = (uint32_t)adesc0, blo0 = (uint32_t)bdesc0;
            for (int mb = 0; mb < MB; ++mb) {
              const uint32_t d_tmem = tmem_base + (uint32_t)((g * MB + mb) * N);
              for (int tap = 0; tap < K; ++tap) {
                uint32_t al = alo0 + (uint32_t)(mb * 128 + tap * dil);                 // 16 B units
                uint32_t bl = blo0 + (uint32_t)tap * (uint32_t)(KC * N * 4 / 16);
                for (int kk = 0; kk < KC / 8; ++kk) {
                  const uint64_t a_hi = desc_with_lo(adesc0, al), a_lo = desc_with_lo(adesc0, al + a_lo_delta);
                  const uint64_t b_hi = desc_with_lo(bdesc0, bl), b_lo = desc_with_lo(bdesc0, bl + b_lo_delta);
                  const uint32_t first = (c == 0 && tap == 0 && kk == 0) ? 0u : 1u;
                  tc_mma_tf32_x3(d_tmem, a_hi, a_lo, b_hi, b_lo, idesc, first);
                  al += 2u * (uint32_t)Rp;
                  bl += 2u * (uint32_t)N;
                }
              }
            }
            if (elect_one()) tc_commit(bar_a_free + 8 * ab);
            __syncwarp();
            if (ab) a_fills1 += 1; else a_fills0 += 1;
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
      for (int c = 0; c < n_chunks_item; ++c) {
        const int c0 = c * KC;
        const bool fast = full16 && (a.Cin - c0) >= KC;
        for (int g = 0; g < tiles; ++g) {
          const int ab = (na == 2) ? (int)(a_count_s & 1) : 0;
          const uint32_t a_uses = ab ? a_uses1 : a_uses0;
          uint8_t* Ah = A0 + (size_t)ab * a_bytes;
          const int t_in0 = t_group0 + g * MT - a.pad_left;
          bool waited = (a_uses == 0);
          // two (row, 16-channel) items per round: 32 independent global loads per thread in flight
          int q16 = 0, r = tid;
          while (r >= Rp) { r -= Rp; ++q16; }
          while (q16 < nb16) {
            int q16b = q16, rb = r + STAGERS;
            while (rb >= Rp) { rb -= Rp; ++q16b; }
            const bool has_b = q16b < nb16;
            float v[2][16];
            int rr[2] = {r, rb}, qq[2] = {q16, q16b};
#pragma unroll
            for (int u2 = 0; u2 < 2; ++u2) {
              const int t = t_in0 + rr[u2];
              const bool rok = (u2 == 0 || has_b) && (rr[u2] < R) && (t >= 0) && (t < t_hi);
              const int ci0 = c0 + qq[u2] * 16;
              const float* src = in_b + (long long)ci0 * a.in_cs + t;
              if (fast) {
#pragma unroll
                for (int e = 0; e < 16; ++e) v[u2][e] = rok ? __ldg(src + (long long)e * a.in_cs) : 0.f;
              } else {
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                  v[u2][e] = 0.f;
                  if (rok && (ci0 + e) < a.Cin && (qq[u2] * 16 + e) < KC) v[u2][e] = __ldg(src + (long long)e * a.in_cs);
                }
              }
            }
            if (!waited) {  // the MMAs that last read this buffer must be done before it is overwritten
              mbar_wait(bar_a_free + 8 * ab, (a_uses - 1) & 1);
              waited = true;
            }
#pragma unroll
            for (int u2 = 0; u2 < 2; ++u2) {
              if (u2 == 1 && !has_b) break;
#pragma unroll
              for (int cg = 0; cg < 4; ++cg) {
                if (fast || qq[u2] * 16 + cg * 4 < KC) {
                  float4 hi, lo;
                  float x0 = v[u2][cg * 4 + 0], x1 = v[u2][cg * 4 + 1], x2 = v[u2][cg * 4 + 2], x3 = v[u2][cg * 4 + 3];
                  if (a.pre_act) {
                    x0 = x0 > 0.f ? x0 : x0 * a.pre_slope; x1 = x1 > 0.f ? x1 : x1 * a.pre_slope;
                    x2 = x2 > 0.f ? x2 : x2 * a.pre_slope; x3 = x3 > 0.f ? x3 : x3 * a.pre_slope;
                  }
                  hi.x = tf32_rna(x0); lo.x = tf32_rna(x0 - hi.x);
                  hi.y = tf32_rna(x1); lo.y = tf32_rna(x1 - hi.y);
                  hi.z = tf32_rna(x2); lo.z = tf32_rna(x2 - hi.z);
                  hi.w = tf32_rna(x3); lo.w = tf32_rna(x3 - hi.w);
                  const size_t o = ((size_t)(qq[u2] * 4 + cg) * Rp + rr[u2]) * 16;
                  *reinterpret_cast<float4*>(Ah + o) = hi;
                  *reinterpret_cast<float4*>(Ah + a_half + o) = lo;
                }
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
          if (ab) a_uses1 += 1; else a_uses0 += 1;
          a_count_s += 1;
        }
      }
    }
    // ---------------- accumulators complete -> fused epilogue (all warps)
    mbar_wait(bar_acc, acc_count & 1);
    acc_count += 1;
    tc_fence_after();
    {
      constexpr int COLSPLIT = THREADS / 128;     // warps sharing a TMEM lane quarter split the columns
      const int q = warp & 3, part = warp >> 2;
      const int ncol = N / COLSPLIT;
      for (int g = 0; g < tiles; ++g) {
        for (int mb = 0; mb < MB; ++mb) {
          const int t = t_group0 + g * MT + mb * 128 + q * 32 + lane;
          const float msk = (t < len) ? 1.f : 0.f;
          const uint32_t col0 = (uint32_t)((g * MB + mb) * N + part * ncol);
          for (int cc = 0; cc < ncol; cc += 16) {
            float v[16];
            tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + col0 + cc, v);
            const int nl = part * ncol + cc;
            const float4* a4 = reinterpret_cast<const float4*>(av + nl);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 x = a4[i];
              v[4 * i + 0] += x.x; v[4 * i + 1] += x.y; v[4 * i + 2] += x.z; v[4 * i + 3] += x.w;
            }
            if (t < T && nt * N + nl < a.Cout) tc_epilogue_slice(a, b, t, nt * N + nl, v, msk);
          }
        }
      }
    }
  }
  __syncthreads();
  if (warp == 0) {
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------ weight packing
// dst[nt][chunk][hl][tap][kg][n][e] from the folded weight src[co][ci][tap]
__global__ void pack_conv_tc_kernel(const float* __restrict__ src, float* __restrict__ dst, const int* __restrict__ co_map,
                                    const int* __restrict__ ci_map, int Cout, int Cin, int K, int src_cin, int N,
                                    int n_tiles, int KC, int n_chunks) {
  const long long per_half = (long long)K * KC * N;
  const long long total = (long long)n_tiles * n_chunks * 2 * per_half;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int e = (int)(r % 4); r /= 4;
    const int n = (int)(r % N); r /= N;
    const int kg = (int)(r % (KC / 4)); r /= (KC / 4);
    const int tap = (int)(r % K); r /= K;
    const int hl = (int)(r % 2); r /= 2;
    const int chunk = (int)(r % n_chunks); r /= n_chunks;
    const int nt = (int)r;
    const int co_p = nt * N + n, ci_p = chunk * KC + kg * 4 + e;
    float w = 0.f;
    if (co_p < Cout && ci_p < Cin) {
      const int co = co_map[co_p];
      const int ci = ci_map ? ci_map[ci_p] : ci_p;
      if (co >= 0) w = src[((long long)co * src_cin + ci) * K + tap];
    }
    const float hi = tf32_rna(w);
    dst[i] = hl ? tf32_rna(w - hi) : hi;
  }
}

}  // namespace

size_t tc_conv_smem_bytes(int K, int dil, int N, int KC, int MB, int n_abuf, int n_bbuf) {
  const int R = 128 * MB + (K - 1) * dil;
  const int Rp = (R + 7) & ~7;
  return 128 + 2048 + (size_t)n_abuf * (2 * (size_t)KC * Rp * 4) + (size_t)n_bbuf * (2 * (size_t)K * KC * N * 4);
}

// Chooses the tiling.  mode 0 ("small"): <= 110 KB shared memory, 256 TMEM columns, 256 threads, two CTAs per
// SM, only if the whole C_in fits one chunk (weights then stay resident in the persistent CTA).  Otherwise
// mode 1 ("large"): <= 220 KB, 512 columns, 512 threads, one CTA per SM, C_in chunked with double-buffered
// weight tiles.
bool tc_conv_plan(int Cin, int Cout, int K, int dil, TcPlan* plan) {
  if (Cin < 8 || Cout < 16) return false;
  const int cin8 = (Cin + 7) / 8 * 8;
  const int cout32 = (Cout + 31) / 32 * 32;
  auto fill = [&](int mode, int N, int n_tiles, int KC, int MB, int na, int nb) {
    const int R = 128 * MB + (K - 1) * dil;
    plan->mode = mode; plan->N = N; plan->n_tiles = n_tiles; plan->KC = KC; plan->n_chunks = (cin8 + KC - 1) / KC;
    plan->MB = MB; plan->tmem_cols = mode == 0 ? 256 : 512; plan->G = plan->tmem_cols / (MB * N);
    plan->n_abuf = na; plan->n_bbuf = nb; plan->R_pad = (R + 7) & ~7; plan->dil = dil;
    plan->packed_floats = (size_t)n_tiles * plan->n_chunks * 2 * K * KC * N;
  };
  // ---- small mode
  if (cout32 <= 128) {
    const int N = cout32;
    for (int na = 2; na >= 1; --na)
      for (int MB = 2; MB >= 1; --MB) {
        if (MB * N > 256) continue;
        if (tc_conv_smem_bytes(K, dil, N, cin8, MB, na, 1) <= 112 * 1024) {
          fill(0, N, 1, cin8, MB, na, 1);
          return true;
        }
      }
  }
  // ---- large mode (N a multiple of 64 so that 16 warps split the columns in 16-wide pieces); prefer the
  // widest N tile, fall back to narrower tiles when the weight tile of one tap does not fit.
  // WETTS_TC_PLAN_VARIANT (experiments): bit 0 = try one 128-row block per tile first (smaller activation
  // buffers -> larger K chunks, more tiles per weight pass); bit 1 = cap the N tile at 128 columns.
  static const int variant = getenv("WETTS_TC_PLAN_VARIANT") ? atoi(getenv("WETTS_TC_PLAN_VARIANT")) : 0;
  const int cout64 = (Cout + 63) / 64 * 64;
  const int nt0 = (variant & 2) ? (cout64 + 127) / 128 : (cout64 + 255) / 256;
  for (int n_tiles = nt0; n_tiles <= cout64 / 64; ++n_tiles) {
    const int N = ((cout64 + n_tiles - 1) / n_tiles + 63) / 64 * 64;
    for (int mbi = 0; mbi < 2; ++mbi) {
      const int MB = (variant & 1) ? 1 + mbi : 2 - mbi;
      if (MB * N > 512) continue;
      for (int nch = 1; nch <= cin8 / 8; ++nch) {
        const int KC = ((cin8 + nch - 1) / nch + 7) / 8 * 8;
        const int nb = (cin8 + KC - 1) / KC == 1 ? 1 : 2;
        if (tc_conv_smem_bytes(K, dil, N, KC, MB, 2, nb) <= 216 * 1024) {
          fill(1, N, n_tiles, KC, MB, 2, nb);
          return true;
        }
      }
    }
  }
  return false;
}

void launch_pack_conv_tc(const float* src, float* dst, const int* co_map, const int* ci_map, int Cout, int Cin, int K,
                         int src_cin, const TcPlan& pl, cudaStream_t s) {
  const long long total = (long long)pl.packed_floats;
  const int blocks = (int)((total + 255) / 256 > 8192 ? 8192 : (total + 255) / 256);
  pack_conv_tc_kernel<<<blocks, 256, 0, s>>>(src, dst, co_map, ci_map, Cout, Cin, K, src_cin, pl.N, pl.n_tiles, pl.KC,
                                             pl.n_chunks);
  count_launch();
}

static std::atomic<bool> g_tc_enabled{true};
void set_tensor_cores_enabled(bool on) { g_tc_enabled = on; }
bool tensor_cores_enabled() { return g_tc_enabled; }

void launch_conv1d_tc(const ConvArgs& a, cudaStream_t s) {
  const TcPlan& pl = a.tc;
  TcConvArgs p;
  p.c = a;
  p.wtc = a.wtc;
  // the packed layout depends on (N, KC, n_chunks) only; M-blocks per tile are chosen per launch
  const int MB = (a.T > 128 && pl.MB == 2) ? 2 : 1;
  const int R = 128 * MB + (a.K - 1) * a.dil;
  p.N = pl.N; p.n_tiles = pl.n_tiles; p.KC = pl.KC; p.n_chunks = pl.n_chunks; p.MB = MB;
  p.tmem_cols = pl.tmem_cols; p.G = pl.tmem_cols / (MB * pl.N);
  p.n_abuf = pl.n_abuf; p.n_bbuf = pl.n_bbuf; p.R_pad = (R + 7) & ~7;
  const size_t smem = tc_conv_smem_bytes(a.K, a.dil, pl.N, pl.KC, MB, pl.n_abuf, pl.n_bbuf);
  static DynSmemAttr attr[2];
  const int n_sm = current_device_sm_count();
  if (n_sm <= 0) return;
  const int group_rows = p.G * 128 * MB;
  const long long items = (long long)a.B * ((a.T + group_rows - 1) / group_rows) * pl.n_tiles;
  if (pl.mode == 0) {
    if (attr[0].ensure((const void*)conv1d_tc_kernel<256, 2>, smem) != cudaSuccess) return;
    const int grid = (int)(items < 2 * n_sm ? items : 2 * n_sm);
    conv1d_tc_kernel<256, 2><<<grid, 256, smem, s>>>(p);
  } else {
    if (attr[1].ensure((const void*)conv1d_tc_kernel<512, 1>, smem) != cudaSuccess) return;
    const int grid = (int)(items < n_sm ? items : n_sm);
    conv1d_tc_kernel<512, 1><<<grid, 512, smem, s>>>(p);
  }
  count_launch();
}

int tc_conv_install_fault_word(unsigned int* word) { return tc::install_fault_word_tu(word) == cudaSuccess ? 0 : 1; }

}  // namespace wetts
