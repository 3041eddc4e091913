// dib_int16.cu -- the integration network (models.py:81-84,122) in the tensor-core mode: 16-bit activations in HBM
// (emb, g_k, dz_k as fp16 -> half the traffic of the fp32 layout), tcgen05.mma kind::f16 with fp32 accumulation.
//
//   * dib_int16_gemm_kernel<MODE>: TMA-fed, mbarrier-pipelined 128 x 128 tile GEMM (K step 64 = one 128-byte swizzle
//     span) with fused epilogues:  FWD  g = act(A W + b) -> fp16;  DGRAD  dz_in = (dz W^T) * act'(g_in) -> fp16;
//     WGRAD  dW = g^T dz over a batch slice -> fp32 split partial (scaled back by 1/S), db = colsum dz from the smem tiles.
//   * dib_int16_head_kernel: the narrow output layer (out <= 16) fused with everything around it -- logits, compiled
//     loss + accuracy, d loss / d logits, the dgrad into the last hidden layer (incl. its act') and the output layer's
//     own weight/bias gradients -- one pass over the last hidden activation.
// Gradient operands are scaled by the power-of-two loss scale S (see dib_enc_fused.cu) to stay inside fp16 range.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "dib_common.cuh"
#include "dib_kernels.h"
#include "dib_sm100.cuh"

int dib_int16_rb_enabled();
int dib_int16_head1_enabled();
int dib_int16_2sm_enabled();

namespace {

using namespace sm100;

constexpr int kBM = 128, kBN = 128, kBK = 64, kStages = 3;
constexpr int kABytes = kBM * 128, kBBytes = kBN * 128, kStageBytes = kABytes + kBBytes;
constexpr int kBarOff = kStages * kStageBytes;
constexpr int kSmemTotal = kBarOff + 128 + 1024;

struct Int16Args {
  float* out32; uint16_t* out16; int ldc;       // WGRAD partial base (fp32) | FWD/DGRAD output (fp16)
  const uint16_t* X; int ldx;                   // DGRAD: activation whose act' gates the gradient (or null)
  const float* bias;                          // FWD
  float* dbias;                               // DGRAD: column sums of the produced gradient per 128-row tile [tiles_r][C] (or null)
  int M, T, C, R, act;
  float alpha, out_scale;
  int nsplit, rows_per_split; long long split_stride;
  int dbg;                                    // measurement only (dib_debug_set_variant key 5): 1 = skip the epilogue's global stores
};

template <bool BF16>
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  uint32_t r;
  if constexpr (BF16) asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
template <bool BF16>
__device__ __forceinline__ void unpack_h2(uint32_t u, float& a, float& b) {
  if constexpr (BF16) { a = __uint_as_float(u << 16); b = __uint_as_float(u & 0xffff0000u); }
  else { const float2 f = __half22float2(*reinterpret_cast<__half2*>(&u)); a = f.x; b = f.y; }
}

// Persistent: each CTA walks tiles blockIdx.x, +gridDim.x, ...; the shared-memory stage ring runs across tiles and the
// fp32 accumulator is double-buffered in TMEM (2 x 128 columns), so the epilogue of tile i overlaps the mainloop of
// tile i+1.  Warp roles: 0 TMA producer | 1 MMA issuer (+ TMEM owner) | 2..5 epilogue.
template <int MODE, bool BF16>
__global__ void __launch_bounds__(192, 2)
dib_int16_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const Int16Args a,
                      const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapB2, const Int16Args a2) {
  // (a2, mapA2, mapB2): an optional SECOND weight-gradient problem walked by the same launch (a2.nsplit > 0, WGRAD only): the two
  // layers' tiles together fill one wave of CTAs, which neither fills alone
  constexpr bool A_MN = (MODE == DIB_GEMM_WGRAD), B_MN = (MODE != DIB_GEMM_DGRAD);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar_base = sb + kBarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int acc) { return bar_base + 8u * (2 * kStages + acc); };
  auto tempty_bar = [&](int acc) { return bar_base + 8u * (2 * kStages + 2 + acc); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 4);
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + kBarOff + 8 * (2 * kStages + 4));

  __shared__ float colsum_s[4][kBN];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R0 = (MODE == DIB_GEMM_WGRAD) ? a.R : a.M, C0 = a.C;
  const int tiles_r = DIB_CEIL_DIV(R0, kBM), tiles_c = DIB_CEIL_DIV(C0, kBN);
  const int nsp = (MODE == DIB_GEMM_WGRAD) ? a.nsplit : 1;
  const int ntile0 = tiles_r * tiles_c * nsp;
  const bool two = (MODE == DIB_GEMM_WGRAD) && a2.nsplit > 0;
  const int tiles_r2 = two ? DIB_CEIL_DIV(a2.R, kBM) : 0, tiles_c2 = two ? DIB_CEIL_DIV(a2.C, kBN) : 0;
  const int ntile = ntile0 + tiles_r2 * tiles_c2 * (two ? a2.nsplit : 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB);
    if (two) { tma_prefetch_desc(&mapA2); tma_prefetch_desc(&mapB2); }
    for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int acc = 0; acc < 2; ++acc) { mbar_init(tfull_bar(acc), 1); mbar_init(tempty_bar(acc), 4); }
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 2 * kBN); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_g;

  int prob = 0;                                     // which problem the tile last decoded belongs to (per thread)
  auto decode = [&](int tile, int& r0, int& c0, int& split, int& t_begin, int& nk) {
    prob = (two && tile >= ntile0) ? 1 : 0;
    if (prob) tile -= ntile0;
    const int tr = prob ? tiles_r2 : tiles_r, tcn = prob ? tiles_c2 : tiles_c;
    const int per = tr * tcn;
    split = tile / per;
    const int rem = tile - split * per;
    r0 = (rem / tcn) * kBM; c0 = (rem % tcn) * kBN;
    int t_end;
    if (MODE == DIB_GEMM_WGRAD) {
      const int rps = prob ? a2.rows_per_split : a.rows_per_split;
      t_begin = split * rps; t_end = min(a.M, t_begin + rps);
    } else { t_begin = 0; t_end = a.T; }
    nk = t_end > t_begin ? DIB_CEIL_DIV(t_end - t_begin, kBK) : 0;
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
        int r0, c0, split, t_begin, nk;
        decode(tile, r0, c0, split, t_begin, nk);
        for (int k = 0; k < nk; ++k) {
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), kStageBytes);
          const uint32_t a_dst = sb + s * kStageBytes, b_dst = a_dst + kABytes;
          const int t0 = t_begin + k * kBK;
          const CUtensorMap* mA = prob ? &mapA2 : &mapA;
          const CUtensorMap* mB = prob ? &mapB2 : &mapB;
          if constexpr (A_MN) tma_load_3d(a_dst, mA, full_bar(s), 0, t0, r0 / 64);
          else                tma_load_2d(a_dst, mA, full_bar(s), t0, r0);
          if constexpr (B_MN) tma_load_3d(b_dst, mB, full_bar(s), 0, t0, c0 / 64);
          else                tma_load_2d(b_dst, mB, full_bar(s), t0, c0);
          if (++s == kStages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {                                       // the whole warp runs the issue loop (uniform registers), one elected lane issues
      constexpr uint32_t idesc = umma_idesc(BF16 ? 1u : 0u, A_MN ? 1u : 0u, B_MN ? 1u : 0u, kBN);
      // K-major: 32 B inside the swizzle span; MN-major (16-bit, SWIZZLE_128B): 16 k-rows = 2048 B, panels 8 KB apart.
      // Only the start-address field of the descriptors moves (stage, 16-deep k step) -- see umma_desc_lo.
      const uint32_t a_lo0 = umma_desc_lo(sb, A_MN ? kBK * 128 : 16), b_lo0 = umma_desc_lo(sb + kABytes, B_MN ? kBK * 128 : 16);
      const uint32_t d_hi = umma_desc_hi(1024);
      constexpr uint32_t a_step = (A_MN ? 2048 : 32) >> 4, b_step = (B_MN ? 2048 : 32) >> 4, st_step = kStageBytes >> 4;
      uint32_t s = 0, ph = 0, lt = 0;
      for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
        int r0, c0, split, t_begin, nk;
        decode(tile, r0, c0, split, t_begin, nk);
        if (nk == 0) continue;
        const int acc = lt & 1;
        mbar_wait(tempty_bar(acc), ((lt >> 1) & 1) ^ 1);           // the epilogue has drained this accumulator
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * kBN;
        for (int k = 0; k < nk; ++k) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after_sync();
          const uint32_t a_lo = a_lo0 + s * st_step, b_lo = b_lo0 + s * st_step;
#pragma unroll
          for (int kk = 0; kk < kBK / 16; ++kk)
            umma_f16_w(d_tmem, umma_desc_join(a_lo + kk * a_step, d_hi), umma_desc_join(b_lo + kk * b_step, d_hi), idesc, (k > 0 || kk > 0) ? 1u : 0u);
          umma_commit_w(empty_bar(s));
          if (++s == kStages) { s = 0; ph ^= 1; }
        }
        umma_commit_w(tfull_bar(acc));
        ++lt;
      }
    }
  } else {
    const int q = warp & 3;
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
      int r0, c0, split, t_begin, nk;
      decode(tile, r0, c0, split, t_begin, nk);
      const int acc = lt & 1;
      const int r = r0 + q * 32 + lane;
      const int R = prob ? a2.R : R0, C = prob ? a2.C : C0;
      // the activation row that gates the gradient (DGRAD) is fetched one 32-column chunk ahead -- the first chunk before the wait
      // for the accumulator -- so that its L2 / HBM latency never sits on the per-chunk critical path
      uint32_t xpre[16], xnext[16];
      auto load_x = [&](int cc, uint32_t (&dst)[16]) {
        if (r < R && c0 + cc < C && a.X) {
          uint32_t xa[8], xb[8];
          dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc, xa);
          dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc + 16, xb);
#pragma unroll
          for (int j = 0; j < 8; ++j) { dst[j] = xa[j]; dst[8 + j] = xb[j]; }
        }
      };
      if constexpr (MODE == DIB_GEMM_DGRAD) load_x(0, xpre);
      if (nk > 0) { mbar_wait(tfull_bar(acc), (lt >> 1) & 1); tc_fence_after_sync(); }
#pragma unroll 1
      for (int cc = 0; cc < kBN; cc += 32) {
        // the bias slice (FWD) is fetched BEFORE the TMEM load so that its latency hides under it (it sat behind
        // tcgen05.wait::ld: 41 % of the FWD kernel's stall samples, profiles/r02_int16_ncu_full.txt)
        const bool live = r < R && c0 + cc < C;
        float4 bpre[8];
        if constexpr (MODE == DIB_GEMM_FWD) {
          if (live) {
#pragma unroll
            for (int j = 0; j < 8; ++j) bpre[j] = *reinterpret_cast<const float4*>(a.bias + c0 + cc + 4 * j);
          }
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) { if (cc + 32 < kBN) load_x(cc + 32, xnext); }
        uint32_t v[32];
        if (nk > 0) { tmem_ld_32x32b_x32(tmem_base + acc * kBN + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v); tmem_ld_wait(); }
        else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        if (r < R && c0 + cc < C && !(a.dbg & 1)) {          // C is a multiple of 64: a 32-column chunk is entirely inside or outside
          const int c = c0 + cc;
          if constexpr (MODE == DIB_GEMM_WGRAD) {
            float* dst = (prob ? a2.out32 : a.out32) + (long long)split * a.split_stride + (long long)r * (prob ? a2.ldc : a.ldc) + c;
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              dib_st_global_v8(dst + j, __float_as_uint(__uint_as_float(v[j]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 1]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 2]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 3]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 4]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 5]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 6]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 7]) * a.out_scale));
          } else {
            uint16_t* dst = a.out16 + (long long)r * a.ldc + c;
            uint32_t ow[16];
            const uint16_t* xs = (MODE == DIB_GEMM_DGRAD && a.X) ? a.X + (long long)r * a.ldx + c : nullptr;
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              float f[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) f[k] = __uint_as_float(v[j + k]);
              if constexpr (MODE == DIB_GEMM_FWD) {
                const float4 b0 = bpre[j >> 2], b1 = bpre[(j >> 2) + 1];
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int k = 0; k < 8; ++k) f[k] = dib_act16(a.act, f[k] + bb[k], a.alpha);
              } else if (xs) {
                const uint32_t xw[4] = {xpre[j >> 1], xpre[(j >> 1) + 1], xpre[(j >> 1) + 2], xpre[(j >> 1) + 3]};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  float h0, h1;
                  unpack_h2<BF16>(xw[k], h0, h1);
                  f[2 * k] *= dib_act_grad(a.act, h0, a.alpha);
                  f[2 * k + 1] *= dib_act_grad(a.act, h1, a.alpha);
                }
              }
              ow[(j >> 1)] = pack_h2<BF16>(f[0], f[1]); ow[(j >> 1) + 1] = pack_h2<BF16>(f[2], f[3]);
              ow[(j >> 1) + 2] = pack_h2<BF16>(f[4], f[5]); ow[(j >> 1) + 3] = pack_h2<BF16>(f[6], f[7]);
              if (j & 8) dib_st_global_v8(dst + j - 8, ow[(j >> 1) - 4], ow[(j >> 1) - 3], ow[(j >> 1) - 2], ow[(j >> 1) - 1], ow[(j >> 1)], ow[(j >> 1) + 1], ow[(j >> 1) + 2], ow[(j >> 1) + 3]);
              if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
                for (int k = 0; k < 8; ++k) v[j + k] = __float_as_uint(f[k]);     // keep the gated fp32 values for the column sums
              }
            }
          }
        } else if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;                                  // rows / columns outside the matrix add nothing
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) {
          if (a.dbias) {
            // bias gradient of the layer below = column sums of the gradient just produced: 32 values per lane are
            // transpose-reduced over the warp's 32 rows in 31 shuffles; lane L ends up with column L of this chunk
            float w[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __uint_as_float(v[j]);
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
#pragma unroll
              for (int i = 0; i < o; ++i) {
                const bool up = (lane & o) != 0;
                const float send = up ? w[i] : w[i + o], keep = up ? w[i + o] : w[i];
                w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
              }
            }
            colsum_s[q][cc + lane] = w[0];
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) xpre[j] = xnext[j];
        }
      }
      if constexpr (MODE == DIB_GEMM_DGRAD) {
        if (a.dbias) {
          asm volatile("bar.sync 1, 128;" ::: "memory");
          const int et = (warp - 2) * 32 + lane;               // one column of the tile per epilogue thread
          if (c0 + et < C)
            a.dbias[(long long)(r0 / kBM) * C + c0 + et] = (colsum_s[0][et] + colsum_s[1][et]) + (colsum_s[2][et] + colsum_s[3][et]);
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
      }
      if (nk > 0) {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
        ++lt;
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) { tc_fence_after_sync(); tmem_dealloc(tmem_base, 2 * kBN); }
}

// ====================================================================================================
// Resident-B variant for FWD / DGRAD (the B operand is a weight matrix): with M = 65 536 rows and 128-row tiles the old
// kernel re-fetched the [K x 128] weight tile from L2 for every one of the 512 row tiles -- at ~20 B/clk of L2
// bandwidth per SM that traffic (not the MMAs) set the kernel time (ncu: long_scoreboard 44-57 %).  Here each persistent
// CTA owns ONE column tile, loads its [K x BN] slice of the weights once (<= 128 KB of shared memory) and streams only
// the activation tiles through a deeper ring; BN = 256 (full output width of the hidden layers) reads A exactly once.
// Warp roles as above: 0 TMA producer | 1 MMA issuer (+ TMEM owner) | 2..5 epilogue.
// ====================================================================================================
constexpr int kRbStages = 5;
template <int BN> constexpr int rb_tmem_cols() { return 2 * BN; }

template <int MODE, bool BF16, int BN>
__global__ void __launch_bounds__(192, 1)
dib_int16_rb_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const Int16Args a, int nkb) {
  static_assert(MODE != DIB_GEMM_WGRAD, "resident-B variant: FWD / DGRAD only");
  constexpr bool B_MN = (MODE == DIB_GEMM_FWD);
  constexpr int kBPanel = BN * 128;                    // bytes of one 64-deep k-block of the resident B slice
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t sB = sb, sA = sb + nkb * kBPanel;      // resident B | A ring
  const int bar_off = nkb * kBPanel + kRbStages * kABytes;
  const uint32_t bar_base = sb + bar_off;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kRbStages + s); };
  auto tfull_bar = [&](int acc) { return bar_base + 8u * (2 * kRbStages + acc); };
  auto tempty_bar = [&](int acc) { return bar_base + 8u * (2 * kRbStages + 2 + acc); };
  const uint32_t bfull_bar = bar_base + 8u * (2 * kRbStages + 4);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kRbStages + 5);
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + bar_off + 8 * (2 * kRbStages + 5));

  __shared__ float colsum_s[4][BN];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int R = a.M, C = a.C;
  const int tiles_r = DIB_CEIL_DIV(R, kBM), tiles_c = DIB_CEIL_DIV(C, BN);
  // this CTA's fixed column tile and its row tiles: blockIdx.x = col + tiles_c * k  (gridDim.x is a multiple of tiles_c)
  const int ctile = blockIdx.x % tiles_c, c0 = ctile * BN;
  const int rfirst = blockIdx.x / tiles_c, rstep = gridDim.x / tiles_c;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB);
    for (int s = 0; s < kRbStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int acc = 0; acc < 2; ++acc) { mbar_init(tfull_bar(acc), 1); mbar_init(tempty_bar(acc), 4); }
    mbar_init(bfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, rb_tmem_cols<BN>()); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_g;

  if (warp == 0) {
    if (lane == 0) {
      // the weight slice of this column tile, once
      mbar_expect_tx(bfull_bar, (uint32_t)(nkb * kBPanel));
      for (int k = 0; k < nkb; ++k) {
        const uint32_t dst = sB + k * kBPanel;
        // one box per k-block: FWD [BN/64 panels][64 k-rows][128 B] (MN-major), DGRAD [BN rows][128 B] (K-major)
        if constexpr (B_MN) tma_load_3d(dst, &mapB, bfull_bar, 0, k * kBK, c0 / 64);
        else                tma_load_2d(dst, &mapB, bfull_bar, k * kBK, c0);
      }
      uint32_t it = 0;
      for (int rt = rfirst; rt < tiles_r; rt += rstep) {
        for (int k = 0; k < nkb; ++k, ++it) {
          const int s = it % kRbStages, ph = (it / kRbStages) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), kABytes);
          tma_load_2d(sA + s * kABytes, &mapA, full_bar(s), k * kBK, rt * kBM);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(BF16 ? 1u : 0u, 0u, B_MN ? 1u : 0u, BN);
      mbar_wait(bfull_bar, 0);
      tc_fence_after_sync();
      uint32_t it = 0, lt = 0;
      for (int rt = rfirst; rt < tiles_r; rt += rstep, ++lt) {
        const int acc = lt & 1;
        mbar_wait(tempty_bar(acc), ((lt >> 1) & 1) ^ 1);           // the epilogue has drained this accumulator
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int k = 0; k < nkb; ++k, ++it) {
          const int s = it % kRbStages, ph = (it / kRbStages) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after_sync();
          const uint32_t a_addr = sA + s * kABytes, b_addr = sB + k * kBPanel;
#pragma unroll
          for (int kk = 0; kk < kBK / 16; ++kk) {
            // A K-major: 32 B inside the swizzle span.  B MN-major (FWD): 16 k-rows = 2048 B inside a [64 k x 64 n] panel,
            // panels 8 KB apart; B K-major (DGRAD): rows = output columns, 128-row groups 16 KB apart handled by SBO = 1024.
            const uint64_t adesc = umma_smem_desc(a_addr + kk * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? umma_smem_desc(b_addr + kk * 2048, kBK * 128, 1024) : umma_smem_desc(b_addr + kk * 32, 16, 1024);
            umma_bf16(d_tmem, adesc, bdesc, idesc, (k > 0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else {
    const int q = warp & 3;
    uint32_t lt = 0;
    for (int rt = rfirst; rt < tiles_r; rt += rstep, ++lt) {
      const int acc = lt & 1, r0 = rt * kBM;
      mbar_wait(tfull_bar(acc), (lt >> 1) & 1); tc_fence_after_sync();
      const int r = r0 + q * 32 + lane;
#pragma unroll 1
      for (int cc = 0; cc < BN; cc += 32) {
        const bool live = r < R && c0 + cc < C;     // global operands of the epilogue first: their latency hides under the TMEM load
        float4 bpre[8];
        uint32_t xpre[16];
        if constexpr (MODE == DIB_GEMM_FWD) {
          if (live) {
#pragma unroll
            for (int j = 0; j < 8; ++j) bpre[j] = *reinterpret_cast<const float4*>(a.bias + c0 + cc + 4 * j);
          }
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) {
          if (live && a.X) {
            uint32_t xa[8], xb[8];
            dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc, xa);
            dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc + 16, xb);
#pragma unroll
            for (int j = 0; j < 8; ++j) { xpre[j] = xa[j]; xpre[8 + j] = xb[j]; }
          }
        }
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v);
        tmem_ld_wait();
        if (r < R && c0 + cc < C) {          // C is a multiple of 64: a 32-column chunk is entirely inside or outside
          const int c = c0 + cc;
          uint16_t* dst = a.out16 + (long long)r * a.ldc + c;
          uint32_t ow[16];
          const uint16_t* xs = (MODE == DIB_GEMM_DGRAD && a.X) ? a.X + (long long)r * a.ldx + c : nullptr;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float f[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] = __uint_as_float(v[j + k]);
            if constexpr (MODE == DIB_GEMM_FWD) {
              const float4 b0 = bpre[j >> 2], b1 = bpre[(j >> 2) + 1];
              const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
              for (int k = 0; k < 8; ++k) f[k] = dib_act16(a.act, f[k] + bb[k], a.alpha);
            } else if (xs) {
              const uint32_t xw[4] = {xpre[j >> 1], xpre[(j >> 1) + 1], xpre[(j >> 1) + 2], xpre[(j >> 1) + 3]};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float h0, h1;
                unpack_h2<BF16>(xw[k], h0, h1);
                f[2 * k] *= dib_act_grad(a.act, h0, a.alpha);
                f[2 * k + 1] *= dib_act_grad(a.act, h1, a.alpha);
              }
            }
            *reinterpret_cast<uint4*>(dst + j) = make_uint4(pack_h2<BF16>(f[0], f[1]), pack_h2<BF16>(f[2], f[3]), pack_h2<BF16>(f[4], f[5]), pack_h2<BF16>(f[6], f[7]));
            if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
              for (int k = 0; k < 8; ++k) v[j + k] = __float_as_uint(f[k]);     // keep the gated fp32 values for the column sums
            }
          }
        } else if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;                                  // rows / columns outside the matrix add nothing
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) {
          if (a.dbias) {
            // bias gradient of the layer below = column sums of the gradient just produced (31-shuffle transpose-reduce)
            float w[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __uint_as_float(v[j]);
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
#pragma unroll
              for (int i = 0; i < o; ++i) {
                const bool up = (lane & o) != 0;
                const float send = up ? w[i] : w[i + o], keep = up ? w[i + o] : w[i];
                w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
              }
            }
            colsum_s[q][cc + lane] = w[0];
          }
        }
      }
      if constexpr (MODE == DIB_GEMM_DGRAD) {
        if (a.dbias) {
          asm volatile("bar.sync 1, 128;" ::: "memory");
          const int et = (warp - 2) * 32 + lane;
          for (int cidx = et; cidx < BN; cidx += 128)
            if (c0 + cidx < C)
              a.dbias[(long long)rt * C + c0 + cidx] = (colsum_s[0][cidx] + colsum_s[1][cidx]) + (colsum_s[2][cidx] + colsum_s[3][cidx]);
          asm volatile("bar.sync 1, 128;" ::: "memory");
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) { tc_fence_after_sync(); tmem_dealloc(tmem_base, rb_tmem_cols<BN>()); }
}

// 32 values per lane over the warp's 32 rows -> lane L holds the column-L total (31 shuffles, fixed order)
__device__ __forceinline__ float warp_colsum32(float (&w)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const bool up = (lane & o) != 0;
      const float send = up ? w[i] : w[i + o], keep = up ? w[i + o] : w[i];
      w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return w[0];
}

// ====================================================================================================
// CTA-pair variant (tcgen05 cta_group::2): the streamed GEMMs above move 64 FLOP per byte of L2->SM traffic with their
// 128 x 128 tiles and run AT the L2 fabric's rate (fwd_l0: 268 MB in 32 us = 8.4 TB/s, 540 TFLOP/s).  Here two CTAs on the
// two SMs of a TPC share one 256 x 256 output tile: each loads its own 128 rows of A and HALF of the B tile (128 of the 256
// columns), one thread of the even CTA issues M = 256 MMAs that read both shared memories, and each CTA's TMEM receives its
// 128 rows of the fp32 accumulator -> 128 FLOP per byte, half the traffic.  One CTA per SM, 6-stage ring of 32 KB per CTA,
// accumulator double-buffered (2 x 256 TMEM columns), eight epilogue warps (two column halves).
// Warp roles: 0 TMA producer (both CTAs) | 1 TMEM owner (both), MMA issuer (even CTA) | 2..9 epilogue.
// ====================================================================================================
constexpr int k2BN = 256, k2Stages = 6;
constexpr int k2StageBytes = kABytes + kBBytes;
constexpr int k2BarOff = k2Stages * k2StageBytes;
constexpr int k2SmemTotal = k2BarOff + 256 + 1024;

template <int MODE, bool BF16>
__global__ void __launch_bounds__(320, 1)
dib_int16_gemm2_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const Int16Args a) {
  constexpr bool A_MN = (MODE == DIB_GEMM_WGRAD), B_MN = (MODE != DIB_GEMM_DGRAD);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar_base = sb + k2BarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (k2Stages + s); };
  auto tfull_bar = [&](int acc) { return bar_base + 8u * (2 * k2Stages + acc); };
  auto tempty_bar = [&](int acc) { return bar_base + 8u * (2 * k2Stages + 2 + acc); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * k2Stages + 4);
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + k2BarOff + 8 * (2 * k2Stages + 4));

  __shared__ float colsum_s[2][4][128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int R = (MODE == DIB_GEMM_WGRAD) ? a.R : a.M, C = a.C;
  const int tiles_rp = DIB_CEIL_DIV(R, 2 * kBM), tiles_c = DIB_CEIL_DIV(C, k2BN);
  const int nsp = (MODE == DIB_GEMM_WGRAD) ? a.nsplit : 1;
  const int ntile = tiles_rp * tiles_c * nsp;
  const int cl = blockIdx.x >> 1, ncl = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapB);
    for (int s = 0; s < k2Stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int acc = 0; acc < 2; ++acc) { mbar_init(tfull_bar(acc), 1); mbar_init(tempty_bar(acc), 16); }
    fence_barrier_init();
  }
  if (warp == 1) { tmem2_alloc(tmem_slot, 2 * k2BN); tmem2_relinquish(); }
  tc_fence_before_sync();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_g;

  auto decode = [&](int tile, int& r0, int& c0, int& split, int& t_begin, int& nk) {
    const int per = tiles_rp * tiles_c;
    split = tile / per;
    const int rem = tile - split * per;
    r0 = (rem / tiles_c) * 2 * kBM + (int)rank * kBM; c0 = (rem % tiles_c) * k2BN;
    int t_end;
    if (MODE == DIB_GEMM_WGRAD) { t_begin = split * a.rows_per_split; t_end = min(a.M, t_begin + a.rows_per_split); }
    else { t_begin = 0; t_end = a.T; }
    nk = t_end > t_begin ? DIB_CEIL_DIV(t_end - t_begin, kBK) : 0;
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      const uint32_t fl0 = mapa_shared(full_bar(0), 0);          // the even CTA's barriers count both CTAs' bytes
      for (int tile = cl; tile < ntile; tile += ncl) {
        int r0, c0, split, t_begin, nk;
        decode(tile, r0, c0, split, t_begin, nk);
        const int cb = c0 + (int)rank * kBN;                     // this CTA's half of the B tile
        for (int k = 0; k < nk; ++k) {
          mbar_wait(empty_bar(s), ph ^ 1);
          if (rank == 0) mbar_expect_tx(full_bar(s), 2 * k2StageBytes);
          const uint32_t fl = fl0 + 8u * s;
          const uint32_t a_dst = sb + s * k2StageBytes, b_dst = a_dst + kABytes;
          const int t0 = t_begin + k * kBK;
          if constexpr (A_MN) tma2_load_3d(a_dst, &mapA, fl, 0, t0, r0 / 64);
          else                tma2_load_2d(a_dst, &mapA, fl, t0, r0);
          if constexpr (B_MN) tma2_load_3d(b_dst, &mapB, fl, 0, t0, cb / 64);
          else                tma2_load_2d(b_dst, &mapB, fl, t0, cb);
          if (++s == k2Stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {                       // the whole warp runs the issue loop (uniform registers), one elected lane issues
      constexpr uint32_t idesc = umma_idesc(BF16 ? 1u : 0u, A_MN ? 1u : 0u, B_MN ? 1u : 0u, k2BN, 2 * kBM);
      // descriptors: only the start-address field moves (stage, 16-deep k step) -- see umma_desc_lo
      const uint32_t a_lo0 = umma_desc_lo(sb, A_MN ? kBK * 128 : 16), b_lo0 = umma_desc_lo(sb + kABytes, B_MN ? kBK * 128 : 16);
      const uint32_t d_hi = umma_desc_hi(1024);
      constexpr uint32_t a_step = (A_MN ? 2048 : 32) >> 4, b_step = (B_MN ? 2048 : 32) >> 4, st_step = k2StageBytes >> 4;
      uint32_t s = 0, ph = 0, lt = 0;
      for (int tile = cl; tile < ntile; tile += ncl) {
        int r0, c0, split, t_begin, nk;
        decode(tile, r0, c0, split, t_begin, nk);
        if (nk == 0) continue;
        const int acc = lt & 1;
        mbar_wait(tempty_bar(acc), ((lt >> 1) & 1) ^ 1);           // both CTAs' epilogues have drained this accumulator
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * k2BN;
        for (int k = 0; k < nk; ++k) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after_sync();
          const uint32_t a_lo = a_lo0 + s * st_step, b_lo = b_lo0 + s * st_step;
#pragma unroll
          for (int kk = 0; kk < kBK / 16; ++kk)
            umma2_f16_w(d_tmem, umma_desc_join(a_lo + kk * a_step, d_hi), umma_desc_join(b_lo + kk * b_step, d_hi), idesc, (k > 0 || kk > 0) ? 1u : 0u);
          umma2_commit_w(empty_bar(s), 3);
          if (++s == k2Stages) { s = 0; ph ^= 1; }
        }
        umma2_commit_w(tfull_bar(acc), 3);
        ++lt;
      }
    }
  } else {
    const int wg = (warp - 2) >> 2, wq = (warp - 2) & 3, q = warp & 3;
    const int wcol = wg * 128;
    uint32_t lt = 0;
    for (int tile = cl; tile < ntile; tile += ncl) {
      int r0, c0, split, t_begin, nk;
      decode(tile, r0, c0, split, t_begin, nk);
      const int acc = lt & 1;
      if (nk > 0) { mbar_wait(tfull_bar(acc), (lt >> 1) & 1); tc_fence_after_sync(); }
      const int r = r0 + q * 32 + lane;
#pragma unroll 1
      for (int cc = wcol; cc < wcol + 128; cc += 32) {
        const bool live = r < R && c0 + cc < C;
        float4 bpre[8];
        uint32_t xpre[16];
        if constexpr (MODE == DIB_GEMM_FWD) {
          if (live) {
#pragma unroll
            for (int j = 0; j < 8; ++j) bpre[j] = *reinterpret_cast<const float4*>(a.bias + c0 + cc + 4 * j);
          }
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) {
          if (live && a.X) {
            uint32_t xa[8], xb[8];
            dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc, xa);
            dib_ld_global_v8(a.X + (long long)r * a.ldx + c0 + cc + 16, xb);
#pragma unroll
            for (int j = 0; j < 8; ++j) { xpre[j] = xa[j]; xpre[8 + j] = xb[j]; }
          }
        }
        uint32_t v[32];
        if (nk > 0) { tmem_ld_32x32b_x32(tmem_base + acc * k2BN + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v); tmem_ld_wait(); }
        else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        if (live && !(a.dbg & 1)) {
          const int c = c0 + cc;
          if constexpr (MODE == DIB_GEMM_WGRAD) {
            float* dst = a.out32 + (long long)split * a.split_stride + (long long)r * a.ldc + c;
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              dib_st_global_v8(dst + j, __float_as_uint(__uint_as_float(v[j]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 1]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 2]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 3]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 4]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 5]) * a.out_scale),
                               __float_as_uint(__uint_as_float(v[j + 6]) * a.out_scale), __float_as_uint(__uint_as_float(v[j + 7]) * a.out_scale));
          } else {
            uint16_t* dst = a.out16 + (long long)r * a.ldc + c;
            uint32_t ow[16];
            const bool gate = (MODE == DIB_GEMM_DGRAD) && a.X != nullptr;
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              float f[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) f[k] = __uint_as_float(v[j + k]);
              if constexpr (MODE == DIB_GEMM_FWD) {
                const float4 b0 = bpre[j >> 2], b1 = bpre[(j >> 2) + 1];
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int k = 0; k < 8; ++k) f[k] = dib_act16(a.act, f[k] + bb[k], a.alpha);
              } else if (gate) {
                const uint32_t xw[4] = {xpre[j >> 1], xpre[(j >> 1) + 1], xpre[(j >> 1) + 2], xpre[(j >> 1) + 3]};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  float h0, h1;
                  unpack_h2<BF16>(xw[k], h0, h1);
                  f[2 * k] *= dib_act_grad(a.act, h0, a.alpha);
                  f[2 * k + 1] *= dib_act_grad(a.act, h1, a.alpha);
                }
              }
              ow[(j >> 1)] = pack_h2<BF16>(f[0], f[1]); ow[(j >> 1) + 1] = pack_h2<BF16>(f[2], f[3]);
              ow[(j >> 1) + 2] = pack_h2<BF16>(f[4], f[5]); ow[(j >> 1) + 3] = pack_h2<BF16>(f[6], f[7]);
              if (j & 8) dib_st_global_v8(dst + j - 8, ow[(j >> 1) - 4], ow[(j >> 1) - 3], ow[(j >> 1) - 2], ow[(j >> 1) - 1], ow[(j >> 1)], ow[(j >> 1) + 1], ow[(j >> 1) + 2], ow[(j >> 1) + 3]);
              if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
                for (int k = 0; k < 8; ++k) v[j + k] = __float_as_uint(f[k]);
              }
            }
          }
        } else if constexpr (MODE == DIB_GEMM_DGRAD) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        if constexpr (MODE == DIB_GEMM_DGRAD) {
          if (a.dbias) {
            float w[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __uint_as_float(v[j]);
            colsum_s[wg][wq][cc - wcol + lane] = warp_colsum32(w, lane);
          }
        }
      }
      if constexpr (MODE == DIB_GEMM_DGRAD) {
        if (a.dbias) {
          if (wg == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
          const int et = wq * 32 + lane;
          if (r0 < R && c0 + wcol + et < C)
            a.dbias[(long long)(r0 / kBM) * C + c0 + wcol + et] = (colsum_s[wg][0][et] + colsum_s[wg][1][et]) + (colsum_s[wg][2][et] + colsum_s[wg][3][et]);
          if (wg == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
        }
      }
      if (nk > 0) {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_shared(tempty_bar(acc), 0));
        ++lt;
      }
    }
  }
  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == 1) { tc_fence_after_sync(); tmem2_dealloc(tmem_base, 2 * k2BN); }
}

// ----------------------------------------------------------------------------------------------------
// output head: one warp per row; lanes own 8 hidden units each (K = 256) or loop (K = multiple of 256)
// ----------------------------------------------------------------------------------------------------
constexpr int kHeadMaxOut = 16, kHeadWarps = 8;

template <int KPT, int OUT, int ROWS, bool BF16>   // hidden units per lane (K / 32); bound of the output width; rows in flight per warp
__global__ void __launch_bounds__(kHeadWarps * 32)
dib_int16_head_kernel(const uint16_t* __restrict__ g, int ldg, int K, const float* __restrict__ Wc, const float* __restrict__ bc,
                      int out_dim, int out_act, int hid_act, float alpha, int loss, const float* __restrict__ y, long long n,
                      float inv_batch, float gscale, uint16_t* __restrict__ dg, int lddg, float* __restrict__ user_pred,
                      float* __restrict__ wpart, int wpart_stride, float* __restrict__ loss_part, float* __restrict__ acc_part) {
  __shared__ float red[kHeadWarps][KPT * 32];
  __shared__ float sred[kHeadWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kHeadWarps + warp, nw = gridDim.x * kHeadWarps;
  float w[KPT][OUT], dw[KPT][OUT], db[OUT], bias[OUT], dbh[KPT];
#pragma unroll
  for (int i = 0; i < KPT; ++i) dbh[i] = 0.f;
#pragma unroll
  for (int o = 0; o < OUT; ++o) {
    db[o] = 0.f;
    bias[o] = o < out_dim ? bc[o] : 0.f;
#pragma unroll
    for (int i = 0; i < KPT; ++i) {
      w[i][o] = o < out_dim ? Wc[(long long)(lane * KPT + i) * out_dim + o] : 0.f;
      dw[i][o] = 0.f;
    }
  }
  float lsum = 0.f, asum = 0.f;
  const bool train = dg != nullptr;

  for (long long row0 = (long long)gw * ROWS; row0 < n; row0 += (long long)nw * ROWS) {
    uint4 hv[ROWS][KPT / 8];
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {                 // issue all loads of the row group first (memory-level parallelism)
      const long long row = row0 + rr < n ? row0 + rr : n - 1;
#pragma unroll
      for (int i = 0; i < KPT; i += 8) hv[rr][i / 8] = *reinterpret_cast<const uint4*>(g + row * ldg + lane * KPT + i);
    }
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const long long row = row0 + rr;
      if (row >= n) break;
      float h[KPT];
#pragma unroll
      for (int i = 0; i < KPT; i += 8) {
        const uint4 v = hv[rr][i / 8];
        unpack_h2<BF16>(v.x, h[i], h[i + 1]); unpack_h2<BF16>(v.y, h[i + 2], h[i + 3]);
        unpack_h2<BF16>(v.z, h[i + 4], h[i + 5]); unpack_h2<BF16>(v.w, h[i + 6], h[i + 7]);
      }
      float z[OUT], dz[OUT];
#pragma unroll
      for (int o = 0; o < OUT; ++o) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < KPT; ++i) s = fmaf(h[i], w[i][o], s);
        z[o] = dib_act(out_act, dib_warp_sum(s) + bias[o], alpha);
        dz[o] = 0.f;
      }
      // ---- compiled loss / metric / d loss / d z  (identical on all lanes)
      if (y) {
        float l = 0.f, acc = 0.f;
        const float inv_out = 1.f / (float)out_dim;
        if (loss == DIB_LOSS_SPARSE_CE_LOGITS) {
          const int label = (int)y[row];
          float m = z[0], zl = 0.f, se = 0.f; int am = 0;
#pragma unroll
          for (int o = 1; o < OUT; ++o) if (o < out_dim && z[o] > m) { m = z[o]; am = o; }
#pragma unroll
          for (int o = 0; o < OUT; ++o) if (o < out_dim) { se += expf(z[o] - m); if (o == label) zl = z[o]; }
          l = m + logf(se) - zl;
          acc = am == label ? 1.f : 0.f;
#pragma unroll
          for (int o = 0; o < OUT; ++o) if (o < out_dim) dz[o] = expf(z[o] - m) / se - (o == label ? 1.f : 0.f);
        } else {
#pragma unroll
          for (int o = 0; o < OUT; ++o) if (o < out_dim) {
            const float t = y[row * out_dim + o];
            if (loss == DIB_LOSS_BCE_LOGITS) { l += fmaxf(z[o], 0.f) - z[o] * t + log1pf(expf(-fabsf(z[o]))); dz[o] = (1.f / (1.f + expf(-z[o])) - t) * inv_out; }
            else if (loss == DIB_LOSS_BCE_PROBS) {
              const float ep = 1e-7f, pc = fminf(fmaxf(z[o], ep), 1.f - ep);
              l -= t * logf(pc + ep) + (1.f - t) * logf(1.f - pc + ep);
              dz[o] = (z[o] > ep && z[o] < 1.f - ep) ? (-t / (pc + ep) + (1.f - t) / (1.f - pc + ep)) * inv_out : 0.f;
            } else { const float d = z[o] - t; l += d * d; dz[o] = 2.f * d * inv_out; }
            acc += ((z[o] > 0.5f ? 1.f : 0.f) == t) ? 1.f : 0.f;
          }
          l *= inv_out; acc *= inv_out;
        }
        lsum += l; asum += acc;
      }
      if (user_pred) {
#pragma unroll
        for (int o = 0; o < OUT; ++o) if (o < out_dim && lane == o) user_pred[row * out_dim + o] = z[o];
      }
      if (train) {
#pragma unroll
        for (int o = 0; o < OUT; ++o) { dz[o] *= inv_batch * dib_act_grad(out_act, z[o], alpha); db[o] += dz[o]; }
        float d[KPT];
#pragma unroll
        for (int i = 0; i < KPT; ++i) {
          float s = 0.f;
#pragma unroll
          for (int o = 0; o < OUT; ++o) { s = fmaf(dz[o], w[i][o], s); dw[i][o] = fmaf(h[i], dz[o], dw[i][o]); }
          d[i] = s * gscale * dib_act_grad(hid_act, h[i], alpha);
          dbh[i] += d[i];
        }
        uint16_t* dst = dg + row * lddg + lane * KPT;
#pragma unroll
        for (int i = 0; i < KPT; i += 8)
          *reinterpret_cast<uint4*>(dst + i) = make_uint4(pack_h2<BF16>(d[i], d[i + 1]), pack_h2<BF16>(d[i + 2], d[i + 3]),
                                                          pack_h2<BF16>(d[i + 4], d[i + 5]), pack_h2<BF16>(d[i + 6], d[i + 7]));
      }
    }
  }
  // ---- per-block partials (fixed order over the block's warps): output-layer weight/bias gradients, loss, accuracy
  if (train) {
#pragma unroll
    for (int o = 0; o < OUT; ++o) {
      if (o < out_dim) {
#pragma unroll
        for (int i = 0; i < KPT; ++i) red[warp][lane * KPT + i] = dw[i][o];
      }
      __syncthreads();
      if (warp == 0 && o < out_dim) {
#pragma unroll
        for (int i = 0; i < KPT; ++i) {
          float s = 0.f;
          for (int ww = 0; ww < kHeadWarps; ++ww) s += red[ww][lane * KPT + i];
          wpart[(long long)blockIdx.x * wpart_stride + (long long)(lane * KPT + i) * out_dim + o] = s;
        }
      }
      __syncthreads();
    }
    // bias gradient of the last hidden layer (column sums of dg, still multiplied by gscale) -> wpart[K*out+out + k]
#pragma unroll
    for (int i = 0; i < KPT; ++i) red[warp][lane * KPT + i] = dbh[i];
    __syncthreads();
    if (warp == 0) {
#pragma unroll
      for (int i = 0; i < KPT; ++i) {
        float s = 0.f;
        for (int ww = 0; ww < kHeadWarps; ++ww) s += red[ww][lane * KPT + i];
        wpart[(long long)blockIdx.x * wpart_stride + (long long)K * out_dim + out_dim + lane * KPT + i] = s;
      }
    }
    __syncthreads();
    if (lane == 0) {
#pragma unroll
      for (int o = 0; o < OUT; ++o) red[warp][o] = db[o];
    }
    __syncthreads();
    if (threadIdx.x < out_dim) {
      float s = 0.f;
      for (int ww = 0; ww < kHeadWarps; ++ww) s += red[ww][threadIdx.x];
      wpart[(long long)blockIdx.x * wpart_stride + (long long)K * out_dim + threadIdx.x] = s;
    }
    __syncthreads();
  }
  if (lane == 0) sred[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int ww = 0; ww < kHeadWarps; ++ww) s += sred[ww]; loss_part[blockIdx.x] = s; }
  __syncthreads();
  if (lane == 0) sred[warp] = asum;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int ww = 0; ww < kHeadWarps; ++ww) s += sred[ww]; acc_part[blockIdx.x] = s; }
}


// ----------------------------------------------------------------------------------------------------
// output head, single-output specialisation (C0, nb-radial: out = 1).  Same mapping as above (a warp per row, 8 hidden
// units per lane) but 8 rows per pass: the eight row dot products are reduced with ONE transposing butterfly (9 shuffles
// instead of 40), after which lane L holds the logit of row L & 7 and the loss / metric / d loss / d z arithmetic runs once
// per pass, lane-parallel, instead of once per row on every lane (ncu: the generic kernel was issue-bound at 45 %).
// ----------------------------------------------------------------------------------------------------
template <bool BF16>
__global__ void __launch_bounds__(kHeadWarps * 32)
dib_int16_head1_kernel(const uint16_t* __restrict__ g, int ldg, int K, const float* __restrict__ Wc, const float* __restrict__ bc,
                       int out_act, int hid_act, float alpha, int loss, const float* __restrict__ y, long long n,
                       float inv_batch, float gscale, uint16_t* __restrict__ dg, int lddg, float* __restrict__ user_pred,
                       float* __restrict__ wpart, int wpart_stride, float* __restrict__ loss_part, float* __restrict__ acc_part) {
  constexpr int KPT = 8, ROWS = 8;
  __shared__ float red[kHeadWarps][KPT * 32];
  __shared__ float sred[kHeadWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kHeadWarps + warp, nw = gridDim.x * kHeadWarps;
  float w[KPT], dw[KPT], dbh[KPT];
#pragma unroll
  for (int i = 0; i < KPT; ++i) { w[i] = Wc[lane * KPT + i]; dw[i] = 0.f; dbh[i] = 0.f; }
  const float bias = bc[0];
  float db = 0.f, lsum = 0.f, asum = 0.f;
  const bool train = dg != nullptr;
  const int myr = lane & (ROWS - 1);

  for (long long row0 = (long long)gw * ROWS; row0 < n; row0 += (long long)nw * ROWS) {
    float h[ROWS][KPT], s[ROWS];
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const long long row = row0 + rr < n ? row0 + rr : n - 1;
      const uint4 v = *reinterpret_cast<const uint4*>(g + row * ldg + lane * KPT);
      unpack_h2<BF16>(v.x, h[rr][0], h[rr][1]); unpack_h2<BF16>(v.y, h[rr][2], h[rr][3]);
      unpack_h2<BF16>(v.z, h[rr][4], h[rr][5]); unpack_h2<BF16>(v.w, h[rr][6], h[rr][7]);
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < KPT; ++i) a = fmaf(h[rr][i], w[i], a);
      s[rr] = a;
    }
    // transposing butterfly: afterwards lane L holds the warp total of s[L & 7]
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) {
#pragma unroll
      for (int i = 0; i < o; ++i) {
        const bool up = (lane & o) != 0;
        const float send = up ? s[i] : s[i + o], keep = up ? s[i + o] : s[i];
        s[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
    }
    float z = s[0];
    z += __shfl_xor_sync(0xffffffffu, z, 8);
    z += __shfl_xor_sync(0xffffffffu, z, 16);
    // ---- lane L: compiled loss / metric / d loss / d z of row row0 + (L & 7)
    const long long mrow = row0 + myr;
    const bool live = mrow < n;
    z = dib_act(out_act, z + bias, alpha);
    float dz = 0.f;
    if (live && y) {
      const float t = y[mrow];
      float l;
      if (loss == DIB_LOSS_BCE_LOGITS) { l = fmaxf(z, 0.f) - z * t + log1pf(expf(-fabsf(z))); dz = 1.f / (1.f + expf(-z)) - t; }
      else if (loss == DIB_LOSS_BCE_PROBS) {
        const float ep = 1e-7f, pc = fminf(fmaxf(z, ep), 1.f - ep);
        l = -(t * logf(pc + ep) + (1.f - t) * logf(1.f - pc + ep));
        dz = (z > ep && z < 1.f - ep) ? -t / (pc + ep) + (1.f - t) / (1.f - pc + ep) : 0.f;
      } else if (loss == DIB_LOSS_SPARSE_CE_LOGITS) { l = 0.f; dz = 0.f; }        // one class: the softmax is constant
      else { const float d = z - t; l = d * d; dz = 2.f * d; }
      const float acc = loss == DIB_LOSS_SPARSE_CE_LOGITS ? ((int)t == 0 ? 1.f : 0.f) : (((z > 0.5f ? 1.f : 0.f) == t) ? 1.f : 0.f);
      if (lane < ROWS) { lsum += l; asum += acc; }
    }
    if (user_pred && live && lane < ROWS) user_pred[mrow] = z;
    if (train) {
      dz = live ? dz * inv_batch * dib_act_grad(out_act, z, alpha) : 0.f;
      if (lane < ROWS) db += dz;
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        const float dzr = __shfl_sync(0xffffffffu, dz, rr);
        if (row0 + rr >= n) break;
        const float ds = dzr * gscale;
        float d[KPT];
#pragma unroll
        for (int i = 0; i < KPT; ++i) {
          dw[i] = fmaf(h[rr][i], dzr, dw[i]);
          d[i] = ds * w[i] * dib_act_grad(hid_act, h[rr][i], alpha);
          dbh[i] += d[i];
        }
        *reinterpret_cast<uint4*>(dg + (row0 + rr) * lddg + lane * KPT) =
            make_uint4(pack_h2<BF16>(d[0], d[1]), pack_h2<BF16>(d[2], d[3]), pack_h2<BF16>(d[4], d[5]), pack_h2<BF16>(d[6], d[7]));
      }
    }
  }
  // ---- per-block partials, fixed order over the block's warps (layout as the generic kernel: [dWc | dbc | colsum dg])
  if (train) {
#pragma unroll
    for (int i = 0; i < KPT; ++i) red[warp][lane * KPT + i] = dw[i];
    __syncthreads();
    if (warp == 0) {
#pragma unroll
      for (int i = 0; i < KPT; ++i) {
        float a = 0.f;
        for (int ww = 0; ww < kHeadWarps; ++ww) a += red[ww][lane * KPT + i];
        wpart[(long long)blockIdx.x * wpart_stride + lane * KPT + i] = a;
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < KPT; ++i) red[warp][lane * KPT + i] = dbh[i];
    __syncthreads();
    if (warp == 0) {
#pragma unroll
      for (int i = 0; i < KPT; ++i) {
        float a = 0.f;
        for (int ww = 0; ww < kHeadWarps; ++ww) a += red[ww][lane * KPT + i];
        wpart[(long long)blockIdx.x * wpart_stride + (long long)K + 1 + lane * KPT + i] = a;
      }
    }
    __syncthreads();
    db = dib_warp_sum(db);
    if (lane == 0) sred[warp] = db;
    __syncthreads();
    if (threadIdx.x == 0) { float a = 0.f; for (int ww = 0; ww < kHeadWarps; ++ww) a += sred[ww]; wpart[(long long)blockIdx.x * wpart_stride + K] = a; }
    __syncthreads();
  }
  lsum = dib_warp_sum(lsum);
  if (lane == 0) sred[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) { float a = 0.f; for (int ww = 0; ww < kHeadWarps; ++ww) a += sred[ww]; loss_part[blockIdx.x] = a; }
  __syncthreads();
  asum = dib_warp_sum(asum);
  if (lane == 0) sred[warp] = asum;
  __syncthreads();
  if (threadIdx.x == 0) { float a = 0.f; for (int ww = 0; ww < kHeadWarps; ++ww) a += sred[ww]; acc_part[blockIdx.x] = a; }
}

// ====================================================================================================
// Fused tail of the integration network for single-output models (C0, nb-radial): the last two hidden layers
// (256 wide each) and the output head in ONE persistent kernel -- models.py:81-84,122 + the compiled loss.
//   per 128-row tile:  L0  D0 = A W0   (A, W0 k-blocks streamed through a 3-stage TMA ring; N = 256, fp32 in TMEM cols 0..255)
//                      e0  g1 = act(D0 + b0) -> 16-bit -> swizzled shared tile (= L1's A operand) and -> HBM (the backward needs it)
//                      L1  D1 = g1 W1  (W1 k-blocks through the same ring; TMEM cols 256..511), started per 64-column chunk of g1
//                      e1  g2 = act(D1 + b1) kept PACKED IN REGISTERS (64 per thread), logit = g2 . w + b, compiled loss / metric,
//                          d loss / d logit, dg2 = dz w act'(g2) -> HBM, output-layer weight / bias gradients and the bias gradient
//                          of the last hidden layer as per-CTA partials.
// g2 never reaches HBM, the head's re-read of it (and its launch) disappears, and L0 of tile i+1 runs under e1 of tile i.
// Warp roles: 0 TMA producer | 1 MMA issuer (+ TMEM owner) | 2..5 epilogue columns 0..127 | 6..9 epilogue columns 128..255.
// ====================================================================================================
constexpr int kF2N = 256, kF2Stages = 3;
constexpr int kF2AB = kBM * 128, kF2BB = kF2N * 128, kF2Stage = kF2AB + kF2BB;      // 16 KB + 32 KB
constexpr int kF2G1Off = kF2Stages * kF2Stage;
constexpr int kF2BarOff = kF2G1Off + kBM * kF2N * 2;
constexpr int kF2Smem = kF2BarOff + 256 + 1024;

struct Fwd2Args {
  const float *b0, *b1, *wout, *bout;
  uint16_t* g1; int ldg1;             // out: first fused layer's activation [M x 256]
  uint16_t* dg2; int lddg;            // out (training) or null: gradient w.r.t. the second fused layer's pre-activation, x gscale
  const float* y; float* user_pred;
  float* wpart; int wpart_stride; float *loss_part, *acc_part;
  int M, nk0, act, out_act, loss;
  float alpha, inv_batch, gscale;
};

__device__ __forceinline__ void st_shared_v4u(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ACT is a template parameter: with the activation switch inside the fully unrolled register-resident passes the kernel grew to
// 14.5 K SASS instructions (232 KB, jump tables per element) and ran instruction-fetch bound (ncu: no_instructions 37 % of samples).
template <bool BF16, int ACT>
__global__ void __launch_bounds__(320, 1)
dib_int16_fwd2_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW0,
                      const __grid_constant__ CUtensorMap mapW1, const Fwd2Args a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar_base = sb + kF2BarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kF2Stages + s); };
  const uint32_t d0_full = bar_base + 8u * (2 * kF2Stages), d1_full = d0_full + 8u, d1_empty = d0_full + 16u;
  auto g1_ready = [&](int k) { return d0_full + 24u + 8u * k; };
  const uint32_t tmem_slot = d0_full + 24u + 32u;
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + kF2BarOff + 8 * (2 * kF2Stages) + 56);

  __shared__ __align__(16) float s_b0[kF2N], s_b1[kF2N], s_w[kF2N];
  __shared__ float s_z[2][2][kBM];
  __shared__ float s_col[2][2][4][128];
  __shared__ float s_red[3][4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntile = DIB_CEIL_DIV(a.M, kBM);

  for (int i = threadIdx.x; i < kF2N; i += blockDim.x) { s_b0[i] = a.b0[i]; s_b1[i] = a.b1[i]; s_w[i] = a.wout[i]; }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA); tma_prefetch_desc(&mapW0); tma_prefetch_desc(&mapW1);
    for (int s = 0; s < kF2Stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(d0_full, 1); mbar_init(d1_full, 1); mbar_init(d1_empty, 8);
    for (int k = 0; k < 4; ++k) mbar_init(g1_ready(k), 4);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot_g;
  const uint32_t g1s = sb + kF2G1Off;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
        for (int k = 0; k < a.nk0; ++k) {
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), kF2Stage);
          const uint32_t dst = sb + s * kF2Stage;
          tma_load_2d(dst, &mapA, full_bar(s), k * kBK, tile * kBM);
          tma_load_3d(dst + kF2AB, &mapW0, full_bar(s), 0, k * kBK, 0);
          if (++s == kF2Stages) { s = 0; ph ^= 1; }
        }
        for (int k = 0; k < kF2N / kBK; ++k) {
          mbar_wait(empty_bar(s), ph ^ 1);
          mbar_expect_tx(full_bar(s), kF2BB);
          tma_load_3d(sb + s * kF2Stage + kF2AB, &mapW1, full_bar(s), 0, k * kBK, 0);
          if (++s == kF2Stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {                                       // the whole warp runs the issue loop (uniform registers), one elected lane issues
      constexpr uint32_t idesc = umma_idesc(BF16 ? 1u : 0u, 0u, 1u, kF2N);
      // descriptors: only the start-address field moves (stage, 16-deep k step) -- see umma_desc_lo
      const uint32_t a_lo0 = umma_desc_lo(sb, 16), b_lo0 = umma_desc_lo(sb + kF2AB, kBK * 128), g_lo0 = umma_desc_lo(g1s, 16);
      const uint32_t d_hi = umma_desc_hi(1024);
      constexpr uint32_t st_step = kF2Stage >> 4;
      uint32_t s = 0, ph = 0, lt = 0;
      for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x, ++lt) {
        // L0 -> D0.  D0 was drained by e0 of the previous tile: L1 of that tile (already issued) waited for all g1 chunks.
        for (int k = 0; k < a.nk0; ++k) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after_sync();
          const uint32_t a_lo = a_lo0 + s * st_step, b_lo = b_lo0 + s * st_step;
#pragma unroll
          for (int kk = 0; kk < kBK / 16; ++kk)
            umma_f16_w(tmem_base, umma_desc_join(a_lo + kk * 2, d_hi), umma_desc_join(b_lo + kk * 128, d_hi), idesc, (k > 0 || kk > 0) ? 1u : 0u);
          umma_commit_w(empty_bar(s));
          if (++s == kF2Stages) { s = 0; ph ^= 1; }
        }
        umma_commit_w(d0_full);
        // L1 -> D1, k-block by k-block as e0 finishes the 64-column chunks of g1
        mbar_wait(d1_empty, (lt & 1) ^ 1);
        tc_fence_after_sync();
#pragma unroll
        for (int k = 0; k < kF2N / kBK; ++k) {
          mbar_wait(g1_ready(k), lt & 1);
          mbar_wait(full_bar(s), ph);
          tc_fence_after_sync();
          const uint32_t a_lo = g_lo0 + k * (kF2AB >> 4), b_lo = b_lo0 + s * st_step;
#pragma unroll
          for (int kk = 0; kk < kBK / 16; ++kk)
            umma_f16_w(tmem_base + kF2N, umma_desc_join(a_lo + kk * 2, d_hi), umma_desc_join(b_lo + kk * 128, d_hi), idesc, (k > 0 || kk > 0) ? 1u : 0u);
          umma_commit_w(empty_bar(s));
          if (++s == kF2Stages) { s = 0; ph ^= 1; }
        }
        umma_commit_w(d1_full);
      }
    }
  } else {
    const int wg = (warp - 2) >> 2, wq = (warp - 2) & 3, q = warp & 3;       // TMEM lane quarter = warp id % 4
    const int colbase = wg * 128, rt = q * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const bool train = a.dg2 != nullptr;
    const float bout = a.bout[0];
    float acc_dw = 0.f, acc_dbh = 0.f, lsum = 0.f, asum = 0.f, dbo = 0.f;     // column accumulators: column colbase + wq * 32 + lane
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x, ++lt) {
      const long long row = (long long)tile * kBM + rt;
      const bool live = row < a.M;
      // ---------------- e0: g1 = act(D0 + b0)
      mbar_wait(d0_full, lt & 1);
      tc_fence_after_sync();
#pragma unroll 1
      for (int j = 0; j < 4; ++j) {
        const int cc = colbase + 32 * j;
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + lane_off + (uint32_t)cc, v);
        tmem_ld_wait();
        uint32_t q0 = 0, q1 = 0, q2 = 0, q3 = 0;
#pragma unroll
        for (int g = 0; g < 32; g += 8) {
          const float4 ba = *reinterpret_cast<const float4*>(&s_b0[cc + g]), bb = *reinterpret_cast<const float4*>(&s_b0[cc + g + 4]);
          const float bv[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
          float f[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] = dib_act16(ACT, __uint_as_float(v[g + k]) + bv[k], a.alpha);
          const uint32_t p0 = pack_h2<BF16>(f[0], f[1]), p1 = pack_h2<BF16>(f[2], f[3]), p2 = pack_h2<BF16>(f[4], f[5]), p3 = pack_h2<BF16>(f[6], f[7]);
          const int c = cc + g;
          st_shared_v4u(g1s + (c >> 6) * kF2AB + rt * 128 + ((((c & 63) >> 3) ^ (rt & 7)) << 4), p0, p1, p2, p3);
          if (g & 8) { if (live) dib_st_global_v8(a.g1 + row * a.ldg1 + c - 8, q0, q1, q2, q3, p0, p1, p2, p3); }
          else { q0 = p0; q1 = p1; q2 = p2; q3 = p3; }
        }
        if (j & 1) {                       // a 64-column chunk of g1 (one k-block of L1) is complete for this warp's rows
          fence_proxy_async_smem();
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(g1_ready(wg * 2 + (j >> 1)));
        }
      }
      // ---------------- e1, pass 1: g2 = act(D1 + b1) packed into registers, partial logit
      mbar_wait(d1_full, lt & 1);
      tc_fence_after_sync();
      uint32_t g2p[64];
      float zp = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int cc = colbase + 32 * j;
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + lane_off + (uint32_t)(kF2N + cc), v);
        tmem_ld_wait();
#pragma unroll
        for (int g = 0; g < 32; g += 4) {
          const float4 bv = *reinterpret_cast<const float4*>(&s_b1[cc + g]), wv = *reinterpret_cast<const float4*>(&s_w[cc + g]);
          const uint32_t pa = pack_h2<BF16>(dib_act16(ACT, __uint_as_float(v[g]) + bv.x, a.alpha), dib_act16(ACT, __uint_as_float(v[g + 1]) + bv.y, a.alpha));
          const uint32_t pb = pack_h2<BF16>(dib_act16(ACT, __uint_as_float(v[g + 2]) + bv.z, a.alpha), dib_act16(ACT, __uint_as_float(v[g + 3]) + bv.w, a.alpha));
          g2p[j * 16 + (g >> 1)] = pa; g2p[j * 16 + (g >> 1) + 1] = pb;
          float h0, h1, h2, h3;
          unpack_h2<BF16>(pa, h0, h1); unpack_h2<BF16>(pb, h2, h3);
          zp = fmaf(h0, wv.x, zp); zp = fmaf(h1, wv.y, zp); zp = fmaf(h2, wv.z, zp); zp = fmaf(h3, wv.w, zp);
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(d1_empty);
      // ---------------- logit, compiled loss / metric, d loss / d logit (both column halves compute it; half 0 accumulates)
      s_z[lt & 1][wg][rt] = zp;
      asm volatile("bar.sync 3, 256;" ::: "memory");
      float z = dib_act(a.out_act, (s_z[lt & 1][0][rt] + s_z[lt & 1][1][rt]) + bout, a.alpha);
      float dz = 0.f;
      if (live && a.y) {
        const float t = a.y[row];
        float l;
        if (a.loss == DIB_LOSS_BCE_LOGITS) { l = fmaxf(z, 0.f) - z * t + log1pf(expf(-fabsf(z))); dz = 1.f / (1.f + expf(-z)) - t; }
        else if (a.loss == DIB_LOSS_BCE_PROBS) {
          const float ep = 1e-7f, pc = fminf(fmaxf(z, ep), 1.f - ep);
          l = -(t * logf(pc + ep) + (1.f - t) * logf(1.f - pc + ep));
          dz = (z > ep && z < 1.f - ep) ? -t / (pc + ep) + (1.f - t) / (1.f - pc + ep) : 0.f;
        } else if (a.loss == DIB_LOSS_SPARSE_CE_LOGITS) { l = 0.f; dz = 0.f; }        // one class: the softmax is constant
        else { const float d = z - t; l = d * d; dz = 2.f * d; }
        const float acc = a.loss == DIB_LOSS_SPARSE_CE_LOGITS ? ((int)t == 0 ? 1.f : 0.f) : (((z > 0.5f ? 1.f : 0.f) == t) ? 1.f : 0.f);
        if (wg == 0) { lsum += l; asum += acc; }
      }
      if (a.user_pred && live && wg == 0) a.user_pred[row] = z;
      if (train) {
        const float dzs = live ? dz * a.inv_batch * dib_act_grad(a.out_act, z, a.alpha) : 0.f;
        const float ds = dzs * a.gscale;
        if (wg == 0) dbo += dzs;
        // ---------------- e1, pass 2: dg2 = ds w act'(g2) -> HBM; column sums of g2 dz (output-layer dW) and of dg2 (bias gradient)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int cc = colbase + 32 * j;
          float wa[32], wb[32];
          uint32_t dq[4] = {0u, 0u, 0u, 0u};
#pragma unroll
          for (int g = 0; g < 32; g += 8) {
            const float4 w0 = *reinterpret_cast<const float4*>(&s_w[cc + g]), w1 = *reinterpret_cast<const float4*>(&s_w[cc + g + 4]);
            const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            float d[8];
#pragma unroll
            for (int k = 0; k < 8; k += 2) {
              float h0, h1;
              unpack_h2<BF16>(g2p[j * 16 + ((g + k) >> 1)], h0, h1);
              wa[g + k] = h0 * dzs; wa[g + k + 1] = h1 * dzs;
              d[k] = ds * wv[k] * dib_act_grad(ACT, h0, a.alpha);
              d[k + 1] = ds * wv[k + 1] * dib_act_grad(ACT, h1, a.alpha);
              wb[g + k] = d[k]; wb[g + k + 1] = d[k + 1];
            }
            const uint32_t e0 = pack_h2<BF16>(d[0], d[1]), e1 = pack_h2<BF16>(d[2], d[3]), e2 = pack_h2<BF16>(d[4], d[5]), e3 = pack_h2<BF16>(d[6], d[7]);
            if (g & 8) { if (live) dib_st_global_v8(a.dg2 + row * a.lddg + cc + g - 8, dq[0], dq[1], dq[2], dq[3], e0, e1, e2, e3); }
            else { dq[0] = e0; dq[1] = e1; dq[2] = e2; dq[3] = e3; }
          }
          const float ca = warp_colsum32(wa, lane), cb = warp_colsum32(wb, lane);
          s_col[wg][0][wq][32 * j + lane] = ca;
          s_col[wg][1][wq][32 * j + lane] = cb;
        }
        // the four warps of this column half cover the tile's 128 rows: fixed-order combine into the thread-owned column
        if (wg == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
        const int t = wq * 32 + lane;
        acc_dw += (s_col[wg][0][0][t] + s_col[wg][0][1][t]) + (s_col[wg][0][2][t] + s_col[wg][0][3][t]);
        acc_dbh += (s_col[wg][1][0][t] + s_col[wg][1][1][t]) + (s_col[wg][1][2][t] + s_col[wg][1][3][t]);
        if (wg == 0) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory");
      }
    }
    // ---------------- per-CTA partials, layout of the head kernels: [dWc (K) | dbc (1) | column sums of dg2 (K)], loss, accuracy
    const int t = colbase + wq * 32 + lane;
    if (train) {
      a.wpart[(long long)blockIdx.x * a.wpart_stride + t] = acc_dw;
      a.wpart[(long long)blockIdx.x * a.wpart_stride + kF2N + 1 + t] = acc_dbh;
    }
    if (wg == 0) {
      lsum = dib_warp_sum(lsum); asum = dib_warp_sum(asum); dbo = dib_warp_sum(dbo);
      if (lane == 0) { s_red[0][wq] = lsum; s_red[1][wq] = asum; s_red[2][wq] = dbo; }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (wq == 0 && lane == 0) {
        a.loss_part[blockIdx.x] = (s_red[0][0] + s_red[0][1]) + (s_red[0][2] + s_red[0][3]);
        a.acc_part[blockIdx.x] = (s_red[1][0] + s_red[1][1]) + (s_red[1][2] + s_red[1][3]);
        if (train) a.wpart[(long long)blockIdx.x * a.wpart_stride + kF2N] = (s_red[2][0] + s_red[2][1]) + (s_red[2][2] + s_red[2][3]);
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) { tc_fence_after_sync(); tmem_dealloc(tmem_base, 512); }
}

template <bool BF16>
__global__ void dib_f32_to_16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    if constexpr (BF16) { const __nv_bfloat16 b = __float2bfloat16_rn(src[i]); dst[i] = *reinterpret_cast<const uint16_t*>(&b); }
    else { const __half b = __float2half_rn(src[i]); dst[i] = *reinterpret_cast<const uint16_t*>(&b); }
  }
}

// K-major: [rows x ld] fp16, box 64 cols x brows
bool map_k(CUtensorMap* m, const void* base, long long cols, long long rows, long long ld, int brows) {
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)brows}, es[2] = {1, 1};
  return tensor_map_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// MN-major: [krows x ld] fp16 whose contiguous dim is M/N -> (64, krow, panel), box 64 x 64 x npanels => smem [panel][krow][128 B]
bool map_mn(CUtensorMap* m, const void* base, long long cols, long long krows, long long ld, int npanels) {
  cuuint64_t dims[3] = {64, (cuuint64_t)krows, (cuuint64_t)(cols / 64)};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, 128};
  cuuint32_t box[3] = {64, (cuuint32_t)kBK, (cuuint32_t)npanels}, es[3] = {1, 1, 1};
  return tensor_map_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, es,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int g_num_sms16 = 0;
template <int MODE, bool BF16>
cudaError_t launch16(const CUtensorMap& mA, const CUtensorMap& mB, const Int16Args& a, dim3 tiles, cudaStream_t st) {
  if (!g_num_sms16) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_num_sms16, cudaDevAttrMultiProcessorCount, dev); }
  const long long nt = (long long)tiles.x * tiles.y * tiles.z;
  if (nt <= 0) return cudaSuccess;
  dim3 grid((unsigned)(nt < 2ll * g_num_sms16 ? nt : 2ll * g_num_sms16));
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(dib_int16_gemm_kernel<MODE, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  Int16Args none{};
  dib_int16_gemm_kernel<MODE, BF16><<<grid, 192, kSmemTotal, st>>>(mA, mB, a, mA, mB, none);
  dib_note_launch();
  return cudaGetLastError();
}

// two weight-gradient problems (same batch, same split stride) in one launch
template <bool BF16>
cudaError_t launch16_wgrad2(const CUtensorMap& mA, const CUtensorMap& mB, const Int16Args& a, const CUtensorMap& mA2, const CUtensorMap& mB2,
                            const Int16Args& a2, cudaStream_t st) {
  if (!g_num_sms16) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_num_sms16, cudaDevAttrMultiProcessorCount, dev); }
  const long long nt = (long long)DIB_CEIL_DIV(a.R, kBM) * DIB_CEIL_DIV(a.C, kBN) * a.nsplit +
                       (long long)DIB_CEIL_DIV(a2.R, kBM) * DIB_CEIL_DIV(a2.C, kBN) * a2.nsplit;
  if (nt <= 0) return cudaSuccess;
  dim3 grid((unsigned)(nt < 2ll * g_num_sms16 ? nt : 2ll * g_num_sms16));
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(dib_int16_gemm_kernel<DIB_GEMM_WGRAD, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  dib_int16_gemm_kernel<DIB_GEMM_WGRAD, BF16><<<grid, 192, kSmemTotal, st>>>(mA, mB, a, mA2, mB2, a2);
  dib_note_launch();
  return cudaGetLastError();
}

// resident-B launch: grid = a multiple of the column-tile count, at most one CTA per SM
template <int MODE, bool BF16, int BN>
cudaError_t launch_rb(const CUtensorMap& mA, const CUtensorMap& mB, const Int16Args& a, int nkb, cudaStream_t st) {
  if (!g_num_sms16) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_num_sms16, cudaDevAttrMultiProcessorCount, dev); }
  const int tiles_r = DIB_CEIL_DIV(a.M, kBM), tiles_c = DIB_CEIL_DIV(a.C, BN);
  long long grid = (long long)tiles_r * tiles_c;
  const long long cap = (long long)(g_num_sms16 / tiles_c) * tiles_c;
  if (grid > cap) grid = cap;
  if (grid <= 0) return cudaSuccess;
  const int smem = nkb * BN * 128 + kRbStages * kABytes + 128 + 1024;
  static int attr_smem = 0;
  if (attr_smem < smem) {
    cudaError_t e = cudaFuncSetAttribute(dib_int16_rb_kernel<MODE, BF16, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    attr_smem = smem;
  }
  dib_int16_rb_kernel<MODE, BF16, BN><<<(unsigned)grid, 192, smem, st>>>(mA, mB, a, nkb);
  dib_note_launch();
  return cudaGetLastError();
}

// CTA-pair launch: clusters of two CTAs (one per SM of a TPC), at most one cluster per SM pair
template <int MODE, bool BF16>
cudaError_t launch2(const CUtensorMap& mA, const CUtensorMap& mB, const Int16Args& a, cudaStream_t st) {
  if (!g_num_sms16) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_num_sms16, cudaDevAttrMultiProcessorCount, dev); }
  const int R = (MODE == DIB_GEMM_WGRAD) ? a.R : a.M;
  const long long nt = (long long)DIB_CEIL_DIV(R, 2 * kBM) * DIB_CEIL_DIV(a.C, k2BN) * ((MODE == DIB_GEMM_WGRAD) ? a.nsplit : 1);
  if (nt <= 0) return cudaSuccess;
  const long long ncl = nt < g_num_sms16 / 2 ? nt : g_num_sms16 / 2;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(dib_int16_gemm2_kernel<MODE, BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2SmemTotal);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(2 * ncl)); cfg.blockDim = dim3(320); cfg.dynamicSmemBytes = k2SmemTotal; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, dib_int16_gemm2_kernel<MODE, BF16>, mA, mB, a);
  dib_note_launch();
  return e != cudaSuccess ? e : cudaGetLastError();
}

// BN for the resident-B kernel (0 = not eligible): the weight slice [T x BN] 16-bit plus the A ring must fit in shared memory
int rb_pick_bn(int T, int C) {
  if (!dib_int16_rb_enabled() || T % kBK != 0 || C % 64 != 0) return 0;
  const int nkb = T / kBK, budget = 227 * 1024 - (kRbStages * kABytes + 128 + 1024) - 4 * 256 * 4 - 1024;
  if (C % 256 == 0 && nkb * 256 * 128 <= budget) return 256;
  if (nkb * 128 * 128 <= budget) return 128;
  return 0;
}

}  // namespace

static int g_int16_head1 = 1;           // single-output head: 8-rows-per-pass kernel (1, default) or the generic one (0)
int dib_int16_head1_enabled() { return g_int16_head1; }
void dib_int16_head1_set(int on) { g_int16_head1 = on ? 1 : 0; }

int g_int16_dbg = 0;
void dib_int16_dbg_set(int v) { g_int16_dbg = v; }
static int g_int16_2sm = -1;             // CTA-pair (cta_group::2) GEMMs for output widths that are multiples of 256
int dib_int16_2sm_enabled() {
  if (g_int16_2sm < 0) { const char* e = getenv("DIB_INT16_2SM"); g_int16_2sm = (e && e[0] == '1') ? 1 : 0; }
  return g_int16_2sm;
}
void dib_int16_2sm_set(int on) { g_int16_2sm = on ? 1 : 0; }

static int g_int16_rb = -1;
int dib_int16_rb_enabled() {
  // measured on B200 at C0 (profiles/r02_int16_resident_b_ab.json): slower than the streamed kernels (fwd 48 vs 37 / 32 us,
  // dgrad_l1 99 vs 63 us) -- one CTA per SM halves the epilogue warps per SM and the epilogue, not the L2 re-reads of the
  // weights, is what paces these GEMMs.  Kept selectable (DIB_INT16_RB=1, dib_debug_set_variant(1, 1)); default off.
  if (g_int16_rb < 0) { const char* e = getenv("DIB_INT16_RB"); g_int16_rb = (e && e[0] == '1') ? 1 : 0; }
  return g_int16_rb;
}
void dib_int16_rb_set(int on) { g_int16_rb = on ? 1 : 0; }

namespace {
struct ConvSegs { const float* src[8]; uint16_t* dst[8]; long long first[9]; int nseg; };
template <bool BF16>
__global__ void dib_f32_to_16_segs_kernel(const ConvSegs A) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.first[A.nseg]) return;
  int k = 0;
#pragma unroll
  for (int q = 1; q < 8; ++q) if (q < A.nseg && i >= A.first[q]) k = q;
  const float v = A.src[k][i - A.first[k]];
  uint16_t o;
  if constexpr (BF16) { const __nv_bfloat16 b = __float2bfloat16_rn(v); o = *reinterpret_cast<const uint16_t*>(&b); }
  else { const __half b = __float2half_rn(v); o = *reinterpret_cast<const uint16_t*>(&b); }
  A.dst[k][i - A.first[k]] = o;
}
}  // namespace

// several fp32 -> 16-bit conversions (the integration network's weight matrices) in one launch
cudaError_t dib_int16_convert_many(const float* const* src, void* const* dst16, const long long* n, int count, int bf16, cudaStream_t st) {
  for (int base = 0; base < count; base += 8) {
    ConvSegs A{};
    long long tot = 0; int m = 0;
    for (int k = base; k < count && m < 8; ++k) {
      if (n[k] <= 0) continue;
      A.src[m] = src[k]; A.dst[m] = static_cast<uint16_t*>(dst16[k]); A.first[m] = tot; tot += n[k]; ++m;
    }
    A.first[m] = tot; A.nseg = m;
    for (int q = m + 1; q < 9; ++q) A.first[q] = tot;
    if (m == 0) continue;
    if (bf16) dib_f32_to_16_segs_kernel<true><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(A);
    else dib_f32_to_16_segs_kernel<false><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(A);
    dib_note_launch();
  }
  return cudaGetLastError();
}

cudaError_t dib_int16_convert(const float* src, void* dst16, long long n, int bf16, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  if (bf16) dib_f32_to_16_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, static_cast<uint16_t*>(dst16), n);
  else dib_f32_to_16_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, static_cast<uint16_t*>(dst16), n);
  dib_note_launch();
  return cudaGetLastError();
}

// g_out[M x N] = act(g_in[M x K] W16[K x N] + bias)
cudaError_t dib_int16_fwd(const void* g_in, int ld_in, const void* w16, const float* bias, void* g_out, int ld_out, int M,
                          int K, int N, int act, float alpha, int bf16, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  CUtensorMap mA, mB;
  if (!map_k(&mA, g_in, K, M, ld_in, kBM) || !map_mn(&mB, w16, N, K, N, kBN / 64))
    return cudaErrorInvalidValue;
  Int16Args a{};
  a.dbg = g_int16_dbg;
  a.out16 = static_cast<uint16_t*>(g_out); a.ldc = ld_out; a.bias = bias; a.M = M; a.T = K; a.C = N; a.act = act; a.alpha = alpha;
  a.out_scale = 1.f; a.nsplit = 1;
  if (const int bn = rb_pick_bn(K, N)) {          // weights resident in shared memory, activations streamed
    if (!map_mn(&mB, w16, N, K, N, bn / 64)) return cudaErrorInvalidValue;
    if (bn == 256) return bf16 ? launch_rb<DIB_GEMM_FWD, true, 256>(mA, mB, a, K / kBK, st) : launch_rb<DIB_GEMM_FWD, false, 256>(mA, mB, a, K / kBK, st);
    return bf16 ? launch_rb<DIB_GEMM_FWD, true, 128>(mA, mB, a, K / kBK, st) : launch_rb<DIB_GEMM_FWD, false, 128>(mA, mB, a, K / kBK, st);
  }
  if (dib_int16_2sm_enabled() && N % k2BN == 0)
    return bf16 ? launch2<DIB_GEMM_FWD, true>(mA, mB, a, st) : launch2<DIB_GEMM_FWD, false>(mA, mB, a, st);
  const dim3 tiles(DIB_CEIL_DIV(M, kBM), DIB_CEIL_DIV(N, kBN), 1);
  return bf16 ? launch16<DIB_GEMM_FWD, true>(mA, mB, a, tiles, st) : launch16<DIB_GEMM_FWD, false>(mA, mB, a, tiles, st);
}

// dz_in[M x K] = (dz[M x N] W16[K x N]^T) * act'(g_in[M x K])      (g_in may be null: no activation, e.g. d_emb)
cudaError_t dib_int16_dgrad(const void* dz, int ld_dz, const void* w16, const void* g_in, int ld_g, void* dz_in, int ld_out,
                            int M, int K, int N, int act, float alpha, float* colsum_part, int bf16, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  CUtensorMap mA, mB;
  if (!map_k(&mA, dz, N, M, ld_dz, kBM) || !map_k(&mB, w16, N, K, N, kBN))
    return cudaErrorInvalidValue;
  Int16Args a{};
  a.dbg = g_int16_dbg;
  a.out16 = static_cast<uint16_t*>(dz_in); a.ldc = ld_out; a.X = static_cast<const uint16_t*>(g_in); a.ldx = ld_g;
  a.M = M; a.T = N; a.C = K; a.act = act; a.alpha = alpha; a.out_scale = 1.f; a.nsplit = 1; a.dbias = colsum_part;
  if (const int bn = rb_pick_bn(N, K)) {          // W^T slice resident, dz streamed
    if (!map_k(&mB, w16, N, K, N, bn)) return cudaErrorInvalidValue;
    if (bn == 256) return bf16 ? launch_rb<DIB_GEMM_DGRAD, true, 256>(mA, mB, a, N / kBK, st) : launch_rb<DIB_GEMM_DGRAD, false, 256>(mA, mB, a, N / kBK, st);
    return bf16 ? launch_rb<DIB_GEMM_DGRAD, true, 128>(mA, mB, a, N / kBK, st) : launch_rb<DIB_GEMM_DGRAD, false, 128>(mA, mB, a, N / kBK, st);
  }
  if (dib_int16_2sm_enabled() && K % k2BN == 0)
    return bf16 ? launch2<DIB_GEMM_DGRAD, true>(mA, mB, a, st) : launch2<DIB_GEMM_DGRAD, false>(mA, mB, a, st);
  const dim3 tiles(DIB_CEIL_DIV(M, kBM), DIB_CEIL_DIV(K, kBN), 1);
  return bf16 ? launch16<DIB_GEMM_DGRAD, true>(mA, mB, a, tiles, st) : launch16<DIB_GEMM_DGRAD, false>(mA, mB, a, tiles, st);
}

// dW[K x N] (fp32 split partials, * out_scale) = g_in[M x K]^T dz[M x N];  db = colsum dz
cudaError_t dib_int16_wgrad(const void* g_in, int ld_g, const void* dz, int ld_dz, float* dW_part, float* db_part, int M, int K,
                            int N, int nsplit, int rows_per_split, long long split_stride, float out_scale, int bf16, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  CUtensorMap mA, mB;
  if (!map_mn(&mA, g_in, K, M, ld_g, kBM / 64) || !map_mn(&mB, dz, N, M, ld_dz, kBN / 64))
    return cudaErrorInvalidValue;
  Int16Args a{};
  a.dbg = g_int16_dbg;
  a.out32 = dW_part; a.ldc = N; a.dbias = nullptr; a.M = M; a.T = 0; a.C = N; a.R = K; a.out_scale = out_scale;
  a.nsplit = nsplit; a.rows_per_split = rows_per_split; a.split_stride = split_stride;
  (void)db_part;   // bias gradients come from the kernel that PRODUCES dz (dgrad epilogue / output head), not from here
  if (dib_int16_2sm_enabled() && N % k2BN == 0)
    return bf16 ? launch2<DIB_GEMM_WGRAD, true>(mA, mB, a, st) : launch2<DIB_GEMM_WGRAD, false>(mA, mB, a, st);
  const dim3 tiles(DIB_CEIL_DIV(N, kBN), DIB_CEIL_DIV(K, kBM), nsplit);
  return bf16 ? launch16<DIB_GEMM_WGRAD, true>(mA, mB, a, tiles, st) : launch16<DIB_GEMM_WGRAD, false>(mA, mB, a, tiles, st);
}

static int g_int16_fwd2 = -1;            // fused [hidden, hidden, head] kernel for single-output models (1, default) or the separate kernels (0)
int dib_int16_fwd2_enabled() {
  if (g_int16_fwd2 < 0) { const char* e = getenv("DIB_INT16_FWD2"); g_int16_fwd2 = (e && e[0] == '0') ? 0 : 1; }
  return g_int16_fwd2;
}
void dib_int16_fwd2_set(int on) { g_int16_fwd2 = on ? 1 : 0; }
int dib_int16_fwd2_ok(int K0, int N1, int N2, int out_dim) {
  return dib_int16_fwd2_enabled() && K0 % kBK == 0 && K0 >= kBK && N1 == kF2N && N2 == kF2N && out_dim == 1;
}

// g1 = act(g_in W0 + b0) -> HBM;  g2 = act(g1 W1 + b1) (on chip);  logit = g2 . wout + bout;  compiled loss / metric;
// training (dg2 != null): dg2, per-CTA partials of the output layer's gradients and of the last hidden layer's bias gradient.
// *nblocks = CTAs launched = rows of wpart / loss_part / acc_part written.
cudaError_t dib_int16_fwd2_head(const void* g_in, int ld_in, int K0, const void* w16_0, const float* b0, const void* w16_1, const float* b1,
                                void* g1, const float* wout, const float* bout, int act, int out_act, float alpha, int loss, const float* y,
                                int M, float inv_batch, float gscale, void* dg2, float* user_pred, float* wpart, int wpart_stride,
                                float* loss_part, float* acc_part, int* nblocks, int bf16, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  if (!g_num_sms16) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_num_sms16, cudaDevAttrMultiProcessorCount, dev); }
  CUtensorMap mA, mW0, mW1;
  if (!map_k(&mA, g_in, K0, M, ld_in, kBM) || !map_mn(&mW0, w16_0, kF2N, K0, kF2N, kF2N / 64) || !map_mn(&mW1, w16_1, kF2N, kF2N, kF2N, kF2N / 64))
    return cudaErrorInvalidValue;
  Fwd2Args a{};
  a.b0 = b0; a.b1 = b1; a.wout = wout; a.bout = bout; a.g1 = static_cast<uint16_t*>(g1); a.ldg1 = kF2N;
  a.dg2 = static_cast<uint16_t*>(dg2); a.lddg = kF2N; a.y = y; a.user_pred = user_pred; a.wpart = wpart; a.wpart_stride = wpart_stride;
  a.loss_part = loss_part; a.acc_part = acc_part; a.M = M; a.nk0 = K0 / kBK; a.act = act; a.out_act = out_act; a.loss = loss;
  a.alpha = alpha; a.inv_batch = inv_batch; a.gscale = gscale;
  const int tiles = DIB_CEIL_DIV(M, kBM);
  const int grid = tiles < g_num_sms16 ? tiles : g_num_sms16;
  *nblocks = grid;
  if (grid <= 0) return cudaSuccess;
  cudaError_t e = cudaErrorInvalidValue;
#define DIB_F2_LAUNCH(BF, ACT)                                                                                                       \
  do {                                                                                                                               \
    static bool attr = false;                                                                                                        \
    e = attr ? cudaSuccess : cudaFuncSetAttribute(dib_int16_fwd2_kernel<BF, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, kF2Smem); \
    if (e != cudaSuccess) return e;                                                                                                  \
    attr = true;                                                                                                                     \
    dib_int16_fwd2_kernel<BF, ACT><<<grid, 320, kF2Smem, st>>>(mA, mW0, mW1, a);                                                      \
  } while (0)
#define DIB_F2_ACT(ACT) do { if (bf16) DIB_F2_LAUNCH(true, ACT); else DIB_F2_LAUNCH(false, ACT); } while (0)
  switch (act) {
    case DIB_ACT_LINEAR: DIB_F2_ACT(DIB_ACT_LINEAR); break;
    case DIB_ACT_RELU: DIB_F2_ACT(DIB_ACT_RELU); break;
    case DIB_ACT_TANH: DIB_F2_ACT(DIB_ACT_TANH); break;
    case DIB_ACT_LEAKY_RELU: DIB_F2_ACT(DIB_ACT_LEAKY_RELU); break;
    case DIB_ACT_SIGMOID: DIB_F2_ACT(DIB_ACT_SIGMOID); break;
    case DIB_ACT_ELU: DIB_F2_ACT(DIB_ACT_ELU); break;
    default: return cudaErrorInvalidValue;
  }
#undef DIB_F2_ACT
#undef DIB_F2_LAUNCH
  dib_note_launch();
  return cudaGetLastError();
}

// the weight gradients of TWO layers in one launch (same batch M, same partial stride): dW_j = g_in_j^T dz_j over batch slices
cudaError_t dib_int16_wgrad_pair(const void* g_in0, int K0, const void* dz0, int N0, float* dW_part0, int nsplit0, int rps0,
                                 const void* g_in1, int K1, const void* dz1, int N1, float* dW_part1, int nsplit1, int rps1,
                                 int M, long long split_stride, float out_scale, int bf16, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  CUtensorMap mA, mB, mA2, mB2;
  if (!map_mn(&mA, g_in0, K0, M, K0, kBM / 64) || !map_mn(&mB, dz0, N0, M, N0, kBN / 64) ||
      !map_mn(&mA2, g_in1, K1, M, K1, kBM / 64) || !map_mn(&mB2, dz1, N1, M, N1, kBN / 64))
    return cudaErrorInvalidValue;
  Int16Args a{}, b{};
  a.dbg = b.dbg = g_int16_dbg;
  a.out32 = dW_part0; a.ldc = N0; a.M = M; a.C = N0; a.R = K0; a.out_scale = out_scale; a.nsplit = nsplit0; a.rows_per_split = rps0; a.split_stride = split_stride;
  b.out32 = dW_part1; b.ldc = N1; b.M = M; b.C = N1; b.R = K1; b.out_scale = out_scale; b.nsplit = nsplit1; b.rows_per_split = rps1; b.split_stride = split_stride;
  return bf16 ? launch16_wgrad2<true>(mA, mB, a, mA2, mB2, b, st) : launch16_wgrad2<false>(mA, mB, a, mA2, mB2, b, st);
}

int dib_int16_head_blocks(int num_sms) { return num_sms * 2; }

cudaError_t dib_int16_head(const void* g, int ldg, int K, const float* Wc, const float* bc, int out_dim, int out_act, int hid_act,
                           float alpha, int loss, const float* y, long long n, float inv_batch, float gscale, void* dg, int lddg,
                           float* user_pred, float* wpart, int wpart_stride, float* loss_part, float* acc_part, int nblocks,
                           int bf16, cudaStream_t st) {
  if (out_dim > kHeadMaxOut || out_dim < 1 || K != 256) return cudaErrorInvalidValue;
#define DIB_HEAD_T(OUT, BF)                                                                                             \
  dib_int16_head_kernel<8, OUT, (OUT <= 2 ? 4 : 1), BF><<<nblocks, kHeadWarps * 32, 0, st>>>(static_cast<const uint16_t*>(g), ldg, K, Wc, bc, out_dim,  \
      out_act, hid_act, alpha, loss, y, n, inv_batch, gscale, static_cast<uint16_t*>(dg), lddg, user_pred, wpart, wpart_stride, \
      loss_part, acc_part)
#define DIB_HEAD(OUT) do { if (bf16) DIB_HEAD_T(OUT, true); else DIB_HEAD_T(OUT, false); } while (0)
  if (out_dim == 1 && dib_int16_head1_enabled()) {
    if (bf16) dib_int16_head1_kernel<true><<<nblocks, kHeadWarps * 32, 0, st>>>(static_cast<const uint16_t*>(g), ldg, K, Wc, bc, out_act,
        hid_act, alpha, loss, y, n, inv_batch, gscale, static_cast<uint16_t*>(dg), lddg, user_pred, wpart, wpart_stride, loss_part, acc_part);
    else dib_int16_head1_kernel<false><<<nblocks, kHeadWarps * 32, 0, st>>>(static_cast<const uint16_t*>(g), ldg, K, Wc, bc, out_act,
        hid_act, alpha, loss, y, n, inv_batch, gscale, static_cast<uint16_t*>(dg), lddg, user_pred, wpart, wpart_stride, loss_part, acc_part);
  } else if (out_dim == 1) DIB_HEAD(1);
  else if (out_dim == 2) DIB_HEAD(2);
  else if (out_dim <= 4) DIB_HEAD(4);
  else if (out_dim <= 8) DIB_HEAD(8);
  else DIB_HEAD(16);
#undef DIB_HEAD
#undef DIB_HEAD_T
  dib_note_launch();
  return cudaGetLastError();
}
