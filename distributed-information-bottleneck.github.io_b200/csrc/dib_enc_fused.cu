// dib_enc_fused.cu -- the fused per-feature encoder kernels of the tensor-core mode (sm_100a).
//
// One persistent CTA per SM works on ONE feature at a time: the feature's encoder weights (positional-encoding
// layer incl. its bias row, 128x128 hidden layer, 128x64 (mu|logvar) layer) are TMA-staged into shared memory
// once and reused for every 128-sample tile of that feature.  Per tile the whole chain of models.py:101-112
//     x column -> positional encoding -> Dense(128,act) -> Dense(128,act) -> Dense(2E) -> split (mu, logvar)
//     -> u = mu + exp(logvar/2) eps -> KL partial sums -> emb[:, f*E:(f+1)*E]
// runs on chip: the three contractions are tcgen05.mma instructions (16-bit operands with an 11-bit significand
// = TF32's, fp32 accumulation in TMEM), the activations travel TMEM -> registers -> shared memory (as the next
// MMA's swizzled A operand) and never touch HBM.  Only x (4 B/sample/feature) is read and emb is written.
//
// Operand layouts (16-bit): every activation/weight tile is [rows][64-element panels of 128 B] with the 16-byte
// chunk index XORed with (row % 8) -- the SWIZZLE_128B pattern, which for 16-bit types is simultaneously a valid
// K-major operand (rows = M/N, panel = K) and a valid MN-major operand (rows = K, panel = M/N).  That dual view is
// what lets the backward kernel use one copy of h1/h2/dz/W for dgrad (reduction over features) and wgrad
// (reduction over samples).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

// (DIB_MBAR_SPIN: non-blocking mbarrier.test_wait probes instead of try_wait in the hand-shake chains -- measured 0.253 vs 0.244 ms
//  for the backward kernel, 0.136 vs 0.133 ms for the forward: the spinning warps take issue slots from the working ones; not defined)
#include "dib_common.cuh"
#include "dib_kernels.h"
#include "dib_sm100.cuh"

namespace {

using namespace sm100;

constexpr int TM = 128;            // samples per tile (UMMA M)
constexpr int HID = 128;           // hidden width of both encoder layers
constexpr int EO = 64;             // 2 * embedding dim
constexpr int K0 = 16;             // padded fan-in of the first layer: [pe (d*nfreq) | 1 (bias) | 0...]
constexpr int kEpiWarps = 8;
constexpr int kThreads = 32 * (1 + kEpiWarps);
constexpr int kPanel = TM * 128;   // bytes of one 64-column panel of a 128-row tile (16 KB)

// packed 16-bit weights in global memory, per feature (elements): W0p[16][128] | W1[128][128] | W2[128][64]
// followed by the bias carriers Bb1[16][128] | Bb2[16][64] whose only non-zero row (index w_in, the position of the
// ones column in the first-layer operand) holds b1 / b2: one extra K=16 MMA step adds the bias for free.
constexpr int kW0Elems = K0 * HID, kW1Elems = HID * HID, kW2Elems = HID * EO, kB1Elems = K0 * HID, kB2Elems = K0 * EO;
constexpr int kPackElems = kW0Elems + kW1Elems + kW2Elems + kB1Elems + kB2Elems;

// shared memory map (bytes; operand tiles 1024-aligned)
constexpr int kOffW1 = 0;
constexpr int kOffW2 = kOffW1 + 2 * kPanel;        // 32 KB
constexpr int kOffW0 = kOffW2 + kPanel;            // 16 KB
constexpr int kOffBb1 = kOffW0 + 2 * K0 * 128;     // 4 KB : W0p = 2 panels x 16 rows x 128 B
constexpr int kOffBb2 = kOffBb1 + 2 * K0 * 128;    // 4 KB : Bb1 likewise
constexpr int kOffA0 = kOffBb2 + K0 * 128;         // 2 KB : Bb2 = 1 panel x 16 rows x 128 B
constexpr int kOffH1 = kOffA0 + 2 * TM * 16 + 2048;// 4 KB : A0 = [2 k-halves][128 rows][16 B] (no swizzle); +2 KB keeps 1024-alignment
constexpr int kOffFwdA0b = kOffH1 + 2 * kPanel;    // forward kernel: h2 overwrites h1 (its MMA has retired); second A0 buffer
constexpr int kOffFwdEnd1 = kOffFwdA0b + 2 * TM * 16;
constexpr int kOffH2 = kOffH1 + 2 * kPanel;
constexpr int kOffFwdEnd = kOffH2 + 2 * kPanel;
// backward-only tiles
constexpr int kOffDO = kOffFwdEnd;                 // [128 x 64]  one panel
constexpr int kOffDZ2 = kOffDO + kPanel;           // [128 x 128] (dz1 aliases H2 once wgrad2 has drained)
constexpr int kOffBwdA0b = kOffDZ2 + 2 * kPanel;    // second A0 buffer (the next tile's operand is staged while this one runs)
constexpr int kOffBwdH1b = kOffBwdA0b + 2 * TM * 16; // second h1 buffer: the next tile's first epilogue does not wait for this tile's dW1
constexpr int kOffBwdEnd = kOffBwdH1b + 2 * kPanel;
static_assert(kOffBwdH1b % 1024 == 0, "operand tiles must be 1024-byte aligned");

struct EncFusedParams {
  const float* x; int ldx;                 // [n, D]
  const int* x_off;                        // [F] first x column of each feature
  const int* fdim;                         // [F] d_i
  int nfreq;                               // 1 + number of sinusoid blocks (1 = no positional encoding)
  const float* params;                     // fp32 master parameters (biases b1, b2 are read from here)
  const long long* b1_off; const long long* b2_off;   // [F] offsets of b1, b2 in params
  const float* eps;                        // [n, F, E] or null -> Philox
  unsigned long long seed; unsigned int step; unsigned long long sample_offset;
  const unsigned int* step_dev;            // optional device addend of `step` (CUDA-Graph replay)
  float* emb; int ldemb; float* user_emb;  // outputs (forward); emb may be null when emb16 is given
  uint16_t* emb16; int ldemb16;            // 16-bit (fp16 / bf16) copy of emb for the 16-bit integration path (or null)
  uint16_t* a0g;                           // [2 F, n, 8] 16-bit copy of the [pe|1] first-layer operand rows (k-halves): written by the training
                                           // forward, TMA-loaded by the two-chain backward instead of recomputing the encoding
  uint16_t* eps16;                         // [n, F*32] 16-bit copy of the Philox noise: written by the training forward, read by the
                                           // two-chain backward instead of regenerating it (the gradient operands are 16-bit anyway)
  float* kl_part; int kl_stride;           // [F][kl_stride] per-(feature, slot) KL partial sums
  int F; long long n; int act; float alpha;
  int round_emb;
};

// two fp32 -> one 32-bit word of two 16-bit values (a in the low half), saturating instead of producing inf
template <bool BF16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  uint32_t r;
  if constexpr (BF16) asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// same with relu fused into the conversion (F2FP.RELU): max(x, 0) costs no instruction of its own
template <bool BF16>
__device__ __forceinline__ uint32_t pack2_relu(float a, float b) {
  uint32_t r;
  if constexpr (BF16) asm("cvt.rn.relu.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  else asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// address of the 16-byte chunk holding columns [8c, 8c+8) of row r in a [128 x 64k] swizzled tile
__device__ __forceinline__ uint32_t tile_chunk_addr(uint32_t tile, int r, int col) {
  const int panel = col >> 6, c = (col & 63) >> 3;
  return tile + panel * kPanel + r * 128 + ((c ^ (r & 7)) << 4);
}

// TMEM -> activation -> 16-bit -> swizzled shared tile, for 64 columns [col0, col0+64) of row r (bias is already in
// the accumulator).  col0 is a multiple of 64, i.e. exactly one 128-byte panel row per thread.
template <bool BF16, bool RELU, int NC = 64>
__device__ __forceinline__ void epilogue_to_tile(uint32_t taddr, uint32_t tile, int r, int col0, int act, float alpha) {
  constexpr int CH = 32;                      // columns per TMEM load
#pragma unroll
  for (int hh = 0; hh < NC / CH; ++hh) {
    uint32_t v[CH];
    tmem_ld_32x32b_x32(taddr + col0 + hh * CH, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < CH; j += 8) {
      if constexpr (RELU) {
        st_shared_v4(tile_chunk_addr(tile, r, col0 + hh * CH + j),
                     pack2_relu<BF16>(__uint_as_float(v[j]), __uint_as_float(v[j + 1])),
                     pack2_relu<BF16>(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])),
                     pack2_relu<BF16>(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5])),
                     pack2_relu<BF16>(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7])));
      } else {
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = dib_act16(act, __uint_as_float(v[j + k]), alpha);
        st_shared_v4(tile_chunk_addr(tile, r, col0 + hh * CH + j), pack2<BF16>(f[0], f[1]), pack2<BF16>(f[2], f[3]),
                     pack2<BF16>(f[4], f[5]), pack2<BF16>(f[6], f[7]));
      }
    }
  }
}

// first-layer operand row: [x_0..x_{d-1}, sin(2x).., sin(4x).., ..., 1, 0...] (models.py:22-23 + the ones column
// that carries every layer's bias through the bias-carrier matrices).  xv = the row's (prefetched) feature values.
// sin for the positional encoding: reduce to one period in units of turns, then the SFU (sin.approx of an argument in
// [-pi, pi] is good to ~1e-6 absolute; the reduction adds |arg| * 6e-8) -- no local-memory slow path like sinf's, and far
// below the 16-bit operand rounding (5e-4 relative) that follows.
__device__ __forceinline__ float dib_sin_pe(float a) {
  float t = a * 0.15915494309189535f;
  t -= rintf(t);
  return __sinf(6.283185307179586f * t);
}
constexpr int kMaxFeatDim = 3;     // d * nfreq + 1 <= 16 and nfreq >= 1
__device__ __forceinline__ void load_x(const float* xrow, int d, float (&xv)[kMaxFeatDim]) {
#pragma unroll
  for (int j = 0; j < kMaxFeatDim; ++j) xv[j] = (xrow && j < d) ? xrow[j] : 0.f;
}
template <bool BF16>
__device__ __forceinline__ void write_a0_row(uint32_t a0, int r, int khalf, bool valid, const float (&xv)[kMaxFeatDim], int d,
                                             int nfreq, uint16_t* gdst = nullptr) {
  float f[8];
  const int w_in = d * nfreq;
  int blk = (khalf * 8) / d, j = khalf * 8 - blk * d;      // one division per call; (blk, j) then advance with the column
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int col = khalf * 8 + k;
    float v = 0.f;
    if (col < w_in) {
      float xj = xv[0];
#pragma unroll
      for (int q = 1; q < kMaxFeatDim; ++q) if (j == q) xj = xv[q];
      v = blk == 0 ? xj : dib_sin_pe((float)(1 << blk) * xj);
    } else if (col == w_in) {
      v = valid ? 1.f : 0.f;          // rows past the batch end contribute nothing
    }
    f[k] = v;
    if (++j == d) { j = 0; ++blk; }
  }
  const uint32_t p0 = pack2<BF16>(f[0], f[1]), p1 = pack2<BF16>(f[2], f[3]), p2 = pack2<BF16>(f[4], f[5]), p3 = pack2<BF16>(f[6], f[7]);
  st_shared_v4(a0 + khalf * (TM * 16) + r * 16, p0, p1, p2, p3);
  if (gdst) *reinterpret_cast<uint4*>(gdst) = make_uint4(p0, p1, p2, p3);       // hand-off to this step's backward kernel
}

// eps for embedding dims [dim0, dim0 + 8) of one row (dim0 a multiple of 8; eps_row points at dim0): explicit tensor or
// Philox (same keying as dib_elementwise.cu: counter word = dim / 4).
// Generated in the idle windows while the tensor pipe runs layers 1/2, not on the critical path behind D2.
__device__ __forceinline__ void noise8(const float* eps_row, unsigned long long seed, unsigned int step,
                                       unsigned long long grow, int f, int dim0, bool valid, float (&nrm)[8]) {
  if (eps_row) {
    if (valid) {
      const float4 a = *reinterpret_cast<const float4*>(eps_row), b = *reinterpret_cast<const float4*>(eps_row + 4);
      nrm[0] = a.x; nrm[1] = a.y; nrm[2] = a.z; nrm[3] = a.w; nrm[4] = b.x; nrm[5] = b.y; nrm[6] = b.z; nrm[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) nrm[j] = 0.f;
    }
  } else {
    float lo[4], hi[4];
    dib_philox_normal4(seed, step, grow, (uint32_t)f, (uint32_t)(dim0 >> 2), lo);
    dib_philox_normal4(seed, step, grow, (uint32_t)f, (uint32_t)((dim0 >> 2) + 1), hi);
#pragma unroll
    for (int j = 0; j < 4; ++j) { nrm[j] = lo[j]; nrm[4 + j] = hi[j]; }
  }
}

struct WeightMaps { CUtensorMap w0, w1, w2, b1, b2, a0lo, a0hi; };   // a0lo / a0hi: the two k-halves of the [pe|1] hand-off (bwd2)

// one thread: stage a feature's packed weights (W0p, W1, W2, bias carriers) into shared memory
__device__ __forceinline__ void load_weights(uint32_t sb, const WeightMaps& m, uint32_t bar, int f) {
  mbar_expect_tx(bar, 2 * K0 * 128 + 2 * kPanel + kPanel + 2 * K0 * 128 + K0 * 128);
  tma_load_3d(sb + kOffW0, &m.w0, bar, 0, 0, f);
  tma_load_3d(sb + kOffW0 + K0 * 128, &m.w0, bar, 64, 0, f);
  tma_load_3d(sb + kOffW1, &m.w1, bar, 0, 0, f);
  tma_load_3d(sb + kOffW1 + kPanel, &m.w1, bar, 64, 0, f);
  tma_load_3d(sb + kOffW2, &m.w2, bar, 0, 0, f);
  tma_load_3d(sb + kOffBb1, &m.b1, bar, 0, 0, f);
  tma_load_3d(sb + kOffBb1 + K0 * 128, &m.b1, bar, 64, 0, f);
  tma_load_3d(sb + kOffBb2, &m.b2, bar, 0, 0, f);
}

// the three forward contractions of one tile, each preceded by its bias-carrier step (issued by one thread)
// W = true: called by a fully converged warp, one elected lane issues (operands stay in uniform registers, no waterfall loop)
template <bool BF16, bool W>
__device__ __forceinline__ void umma_issue(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (W) umma_f16_w(d_tmem, adesc, bdesc, idesc, accumulate);
  else umma_f16<BF16>(d_tmem, adesc, bdesc, idesc, accumulate);
}
template <bool BF16, bool W = false>
__device__ __forceinline__ void issue_layer0(uint32_t sb, uint32_t tD, uint32_t a0) {
  constexpr uint32_t id = umma_idesc(BF16 ? 1u : 0u, 0, 1, HID);
  umma_issue<BF16, W>(tD, umma_desc16(a0 >> 4, TM * 16, 128, kLayoutNone), umma_desc16((sb >> 4) + ((kOffW0) >> 4), K0 * 128, 1024), id, 0u);
}
template <bool BF16, bool W = false>
__device__ __forceinline__ void issue_layer1(uint32_t sb, uint32_t tD, uint32_t h1, uint32_t a0) {
  constexpr uint32_t id = umma_idesc(BF16 ? 1u : 0u, 0, 1, HID);
  umma_issue<BF16, W>(tD, umma_desc16(a0 >> 4, TM * 16, 128, kLayoutNone), umma_desc16((sb >> 4) + ((kOffBb1) >> 4), K0 * 128, 1024), id, 0u);
#pragma unroll
  for (int kk = 0; kk < HID / 16; ++kk)
    umma_issue<BF16, W>(tD, umma_desc16((h1 >> 4) + (((kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024),
                   umma_desc16((sb >> 4) + ((kOffW1 + kk * 2048) >> 4), kPanel, 1024), id, 1u);
}
template <bool BF16, bool W = false>
__device__ __forceinline__ void issue_layer2(uint32_t sb, uint32_t tD, uint32_t h2, uint32_t a0) {
  constexpr uint32_t id = umma_idesc(BF16 ? 1u : 0u, 0, 1, EO);
  umma_issue<BF16, W>(tD, umma_desc16(a0 >> 4, TM * 16, 128, kLayoutNone), umma_desc16((sb >> 4) + ((kOffBb2) >> 4), K0 * 128, 1024), id, 0u);
#pragma unroll
  for (int kk = 0; kk < HID / 16; ++kk)
    umma_issue<BF16, W>(tD, umma_desc16((h2 >> 4) + (((kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024),
                   umma_desc16((sb >> 4) + ((kOffW2 + kk * 2048) >> 4), kPanel, 1024), id, 1u);
}

#define DIB_EPI_SIGNAL(bar)            \
  do {                                 \
    fence_proxy_async_smem();          \
    tc_fence_before_sync();            \
    __syncwarp();                      \
    if (lane == 0) mbar_arrive(bar);   \
  } while (0)

// ====================================================================================================
// forward: x -> emb, KL partial sums.  96 KB of shared memory and 256 TMEM columns per CTA -> two CTAs per SM, so
// one CTA's epilogue overlaps the other's MMAs.
// ====================================================================================================
template <bool BF16, bool RELU>
__global__ void __launch_bounds__(kThreads, 2)
dib_enc_fused_fwd_kernel(const __grid_constant__ WeightMaps maps, const EncFusedParams P) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  constexpr int kOffBar = kOffFwdEnd1;
  float* red_s = reinterpret_cast<float*>(sg + kOffBar + 128);          // [kEpiWarps]
  const uint32_t bar = sb + kOffBar;
  const uint32_t bar_w = bar, bar_a0 = bar + 8, bar_d0 = bar + 16, bar_h1 = bar + 24, bar_d1 = bar + 32,
                 bar_h2 = bar + 40, bar_d2 = bar + 48, tmem_slot = bar + 56;
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + kOffBar + 56);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int G = gridDim.x, c = blockIdx.x, F = P.F;
  const int ntiles = (int)((P.n + TM - 1) / TM);
  const unsigned int nstep = P.step + (P.step_dev ? P.step_dev[0] : 0u);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&maps.w0); tma_prefetch_desc(&maps.w1); tma_prefetch_desc(&maps.w2);
    tma_prefetch_desc(&maps.b1); tma_prefetch_desc(&maps.b2);
    mbar_init(bar_w, 1);
    mbar_init(bar_a0, kEpiWarps); mbar_init(bar_h1, kEpiWarps); mbar_init(bar_h2, kEpiWarps);
    mbar_init(bar_d0, 1); mbar_init(bar_d1, 1); mbar_init(bar_d2, 1);
    fence_barrier_init();
  }
  if (warp == 0) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot_g;
  const uint32_t tR0 = tmem, tR1 = tmem + 128;          // D0 and D1 share R0; D2 -> R1
  const uint32_t hbuf = sb + kOffH1;                    // h1, then h2

  int f_first, f_step, nslots, slot;
  if (G >= F) { f_first = c % F; f_step = F * G; slot = c / F; nslots = (G - f_first + F - 1) / F; }
  else { f_first = c; f_step = G; slot = 0; nslots = 1; }
  uint32_t it = 0, fit = 0;

  for (int f = f_first; f < F; f += f_step, ++fit) {
    if (warp == 0) {
      // the whole warp walks the issue sequence (uniform control flow: descriptors and barrier addresses stay in uniform
      // registers); one elected lane executes each tcgen05 instruction
      if (lane == 0) load_weights(sb, maps, bar_w, f);
      __syncwarp();
      mbar_wait_backoff(bar_w, fit & 1);
      for (int t = slot; t < ntiles; t += nslots, ++it) {
        const uint32_t ph = it & 1;
        mbar_wait_backoff(bar_a0, ph); tc_fence_after_sync();
        const uint32_t a0 = sb + ((it & 1) ? kOffFwdA0b : kOffA0);
        issue_layer0<BF16, true>(sb, tR0, a0); umma_commit_w(bar_d0);
        mbar_wait_backoff(bar_h1, ph); tc_fence_after_sync();
        issue_layer1<BF16, true>(sb, tR0, hbuf, a0); umma_commit_w(bar_d1);
        mbar_wait_backoff(bar_h2, ph); tc_fence_after_sync();
        issue_layer2<BF16, true>(sb, tR1, hbuf, a0); umma_commit_w(bar_d2);
        if (t + nslots >= ntiles) mbar_wait_backoff(bar_d2, ph);   // drain before the next feature's weights land
      }
      __syncwarp();
    } else {
      const int ew = warp - 1, q = warp & 3, hsel = ew >> 2;      // TMEM lane quarter, column half
      const int et = ew * 32 + lane;
      const int r = q * 32 + lane;
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      const int d = P.fdim[f], xo = P.x_off[f];
      float kl_acc = 0.f;
      const int ar = et & (TM - 1), khalf = et >> 7;             // first-layer operand: row / k-half staged by this thread
      float xv[kMaxFeatDim];
      if (slot < ntiles) {                                       // operand of the first tile
        const long long grow = (long long)slot * TM + ar;
        load_x(grow < P.n ? P.x + grow * P.ldx + xo : nullptr, d, xv);
        write_a0_row<BF16>(sb + ((it & 1) ? kOffFwdA0b : kOffA0), ar, khalf, grow < P.n, xv, d, P.nfreq,
                           (P.a0g && grow < P.n) ? P.a0g + ((long long)(2 * f + khalf) * P.n + grow) * 8 : nullptr);
        DIB_EPI_SIGNAL(bar_a0);
      }
      for (int t = slot; t < ntiles; t += nslots, ++it) {
        const uint32_t ph = it & 1;
        const long long row0 = (long long)t * TM;
        const bool has_next = t + nslots < ntiles;
        const long long grow_n = (long long)(t + nslots) * TM + ar;
        if (has_next) load_x(grow_n < P.n ? P.x + grow_n * P.ldx + xo : nullptr, d, xv);   // prefetch the next tile's x
        const long long grow = row0 + r;
        const bool valid = grow < P.n;
        const float* ep = (P.eps && valid) ? P.eps + (grow * F + f) * 32 + hsel * 16 : P.eps;
        float nrmA[8], nrmB[8];
        mbar_wait(bar_d0, ph); tc_fence_after_sync();
        epilogue_to_tile<BF16, RELU>(tR0 + lane_addr, hbuf, r, hsel * 64, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h1);
        if (has_next) {      // stage the next tile's operand in the other A0 buffer: its layer-0 MMA then runs early
          write_a0_row<BF16>(sb + (((it + 1) & 1) ? kOffFwdA0b : kOffA0), ar, khalf, grow_n < P.n, xv, d, P.nfreq,
                             (P.a0g && grow_n < P.n) ? P.a0g + ((long long)(2 * f + khalf) * P.n + grow_n) * 8 : nullptr);
          DIB_EPI_SIGNAL(bar_a0);
        }
        noise8(ep, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, hsel * 16, valid, nrmA);   // while layer 1 runs
        mbar_wait(bar_d1, ph); tc_fence_after_sync();
        epilogue_to_tile<BF16, RELU>(tR0 + lane_addr, hbuf, r, hsel * 64, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h2);
        noise8(ep ? ep + 8 : nullptr, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, hsel * 16 + 8, valid, nrmB);   // while layer 2 runs
        if (P.eps16 && valid)        // hand the noise to the backward kernel of this step (16-bit, like its gradient operands): one 32-byte store
          dib_st_global_v8(P.eps16 + (grow * F + f) * 32 + hsel * 16,
                           pack2<BF16>(nrmA[0], nrmA[1]), pack2<BF16>(nrmA[2], nrmA[3]), pack2<BF16>(nrmA[4], nrmA[5]), pack2<BF16>(nrmA[6], nrmA[7]),
                           pack2<BF16>(nrmB[0], nrmB[1]), pack2<BF16>(nrmB[2], nrmB[3]), pack2<BF16>(nrmB[4], nrmB[5]), pack2<BF16>(nrmB[6], nrmB[7]));
        // ---- (mu, logvar) -> reparameterise, KL, emb   (16 embedding dims per thread)
        mbar_wait(bar_d2, ph); tc_fence_after_sync();
        {
          uint32_t vm[16], vl[16];
          tmem_ld_32x32b_x16(tR1 + lane_addr + hsel * 16, vm);
          tmem_ld_32x32b_x16(tR1 + lane_addr + 32 + hsel * 16, vl);
          tmem_ld_wait();
          tc_fence_before_sync();
          if (valid) {
            float* dst = P.emb ? P.emb + grow * P.ldemb + f * 32 + hsel * 16 : nullptr;
            uint16_t* dst16 = P.emb16 ? P.emb16 + grow * P.ldemb16 + f * 32 + hsel * 16 : nullptr;
            float* udst = P.user_emb ? P.user_emb + grow * ((long long)F * 32) + f * 32 + hsel * 16 : nullptr;
            uint32_t ew[8];
#pragma unroll
            for (int e0 = 0; e0 < 16; e0 += 4) {
              float u[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float mu = __uint_as_float(vm[e0 + j]), lv = __uint_as_float(vl[e0 + j]);
                const float s = __expf(0.5f * lv);      // ex2.approx: relative error 2^-21, far inside the 16-bit operand rounding
                u[j] = fmaf(s, e0 < 8 ? nrmA[e0 + j] : nrmB[e0 - 8 + j], mu);
                kl_acc += 0.5f * (mu * mu + s * s - lv - 1.f);
              }
              if (udst) *reinterpret_cast<float4*>(udst + e0) = make_float4(u[0], u[1], u[2], u[3]);
              ew[e0 >> 1] = pack2<BF16>(u[0], u[1]); ew[(e0 >> 1) + 1] = pack2<BF16>(u[2], u[3]);
              if (dst) {
                if (P.round_emb) {
#pragma unroll
                  for (int j = 0; j < 4; ++j) u[j] = dib_round_tf32(u[j]);
                }
                *reinterpret_cast<float4*>(dst + e0) = make_float4(u[0], u[1], u[2], u[3]);
              }
            }
            if (dst16) dib_st_global_v8(dst16, ew);      // this thread's 16 embedding dims: one full 32-byte sector
          }
        }
      }
      // ---- per-(feature, slot) KL partial: fixed-order reduction over the 256 epilogue threads
      kl_acc = dib_warp_sum(kl_acc);
      if (lane == 0) red_s[ew] = kl_acc;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
      if (et == 0) {
        float s = 0.f;
        for (int i = 0; i < kEpiWarps; ++i) s += red_s[i];
        P.kl_part[(long long)f * P.kl_stride + slot] = s;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) { tc_fence_after_sync(); tmem_dealloc(tmem, 256); }
}

// ====================================================================================================
// backward: recompute the forward chain on chip, then dgrad + wgrad of all three layers.
//   d(mu)     = S*du + (beta*S/B)*mu                       (du = d loss / d u from the integration network)
//   d(logvar) = S*du*eps*0.5*sigma + (beta*S/B)*0.5*(sigma^2-1)
//   dz2 = (d(mu|logvar) W2^T) * act'(h2);  dz1 = (dz2 W1^T) * act'(h1)
//   dW2 += h2^T d(mu|logvar);  dW1 += h1^T dz2;  [dW0;db0]^T += dz1^T [pe|1];  db1 = colsum dz2 (ones column of A0)
// S is a power-of-two loss scale that keeps the 16-bit gradient operands in range (fp16); the fp32 accumulators
// are multiplied by 1/S when they are flushed.  Weight-gradient accumulators live in TMEM for the whole feature.
// TMEM columns: [0,128) D0/D1 | [128,256) D2, G2, G1 | [256,384) dW1 | [384,448) dW2 | [448,464) dW0p^T | [464,480) db1
//               | [480,496) db2  (bias gradients = the ones column of [pe|1] used as the B operand: colsum for free)
// ====================================================================================================
struct EncFusedBwdParams {
  EncFusedParams f;
  const float* d_emb; int ldd;              // [n, ldd] gradient w.r.t. emb (already scaled by 1/B_global)
  const uint16_t* d_emb16; int ldd16;       // or: 16-bit gradient already multiplied by the loss scale S
  const float* beta_dev; float inv_batch; float gscale;
  float* part; long long split_stride;      // weight-gradient partials [slot][P]
  const long long* w0_off; const long long* b0_off; const long long* w1_off; const long long* w2_off;
};

__device__ __forceinline__ void ld_shared_v4(uint32_t addr, uint32_t (&v)[4]) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr));
}
template <bool BF16>
__device__ __forceinline__ void unpack2(uint32_t u, float& a, float& b) {
  if constexpr (BF16) { const float2 f = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u)); a = f.x; b = f.y; }
  else { const float2 f = __half22float2(*reinterpret_cast<__half2*>(&u)); a = f.x; b = f.y; }
}

// packed 16-bit pair p * (h > 0): relu' applied to two gradients at once (exact: multiplication by 1.0 / 0.0)
template <bool BF16>
__device__ __forceinline__ uint32_t relu_gate2(uint32_t p, uint32_t h) {
  if constexpr (BF16) {
    const __nv_bfloat162 z = __float2bfloat162_rn(0.f);
    __nv_bfloat162 g = __hmul2(*reinterpret_cast<__nv_bfloat162*>(&p), __hgt2(*reinterpret_cast<__nv_bfloat162*>(&h), z));
    return *reinterpret_cast<uint32_t*>(&g);
  } else {
    const __half2 z = __float2half2_rn(0.f);
    __half2 g = __hmul2(*reinterpret_cast<__half2*>(&p), __hgt2(*reinterpret_cast<__half2*>(&h), z));
    return *reinterpret_cast<uint32_t*>(&g);
  }
}

// TMEM gradient g (64 columns) * act'(h) -> 16-bit -> shared tile `dtile`; h is read back from the shared tile
// `htile` that the forward epilogue wrote (relu: as a packed comparison, other activations through act'(h))
template <bool BF16, bool RELU, int NC = 64>
__device__ __forceinline__ void dgrad_epilogue(uint32_t taddr, uint32_t htile, uint32_t dtile, int r, int col0, int act,
                                               float alpha) {
  constexpr int CH = 32;
#pragma unroll
  for (int hh = 0; hh < NC / CH; ++hh) {
    uint32_t v[CH];
    tmem_ld_32x32b_x32(taddr + col0 + hh * CH, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < CH; j += 8) {
      const uint32_t ch = tile_chunk_addr(0u, r, col0 + hh * CH + j);
      uint32_t hv[4], o[4];
      ld_shared_v4(htile + ch, hv);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if constexpr (RELU) {
          o[k] = relu_gate2<BF16>(pack2<BF16>(__uint_as_float(v[j + 2 * k]), __uint_as_float(v[j + 2 * k + 1])), hv[k]);
        } else {
          float h0, h1;
          unpack2<BF16>(hv[k], h0, h1);
          o[k] = pack2<BF16>(__uint_as_float(v[j + 2 * k]) * dib_act_grad(act, h0, alpha),
                             __uint_as_float(v[j + 2 * k + 1]) * dib_act_grad(act, h1, alpha));
        }
      }
      st_shared_v4(dtile + ch, o[0], o[1], o[2], o[3]);
    }
  }
}

// EW epilogue warps (8 or 16): 4 TMEM lane quarters x CS = EW/4 column slices.  16 warps halve the columns per thread
// (fewer live registers) and double the warps per scheduler that hide the TMEM / shared-memory / SFU latencies.
template <bool BF16, bool RELU, int EW>
__global__ void __launch_bounds__(32 * (1 + EW), 1)
dib_enc_fused_bwd_kernel(const __grid_constant__ WeightMaps maps, const EncFusedBwdParams Q) {
  const EncFusedParams& P = Q.f;
  constexpr int CS = EW / 4, NC = HID / CS, ND = 32 / CS, NW2 = EO / CS;   // column slices; columns / emb dims / dW2 columns per thread
  static_assert(EW == 8 || EW == 16, "8 or 16 epilogue warps");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  constexpr int kOffBar = kOffBwdEnd;
  const uint32_t bar = sb + kOffBar;
  const uint32_t bar_w = bar, bar_a0 = bar + 8, bar_d0 = bar + 16, bar_h1 = bar + 24, bar_d1 = bar + 32,
                 bar_h2 = bar + 40, bar_d2 = bar + 48, bar_do = bar + 56, bar_g2 = bar + 64, bar_dz2 = bar + 72,
                 bar_g1 = bar + 80, bar_dz1 = bar + 88, bar_wg = bar + 96, tmem_slot = bar + 104;
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + kOffBar + 104);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int G = gridDim.x, c = blockIdx.x, F = P.F;
  const int ntiles = (int)((P.n + TM - 1) / TM);
  const unsigned int nstep = P.step + (P.step_dev ? P.step_dev[0] : 0u);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&maps.w0); tma_prefetch_desc(&maps.w1); tma_prefetch_desc(&maps.w2);
    tma_prefetch_desc(&maps.b1); tma_prefetch_desc(&maps.b2);
    mbar_init(bar_w, 1);
    mbar_init(bar_a0, EW); mbar_init(bar_h1, EW); mbar_init(bar_h2, EW);
    mbar_init(bar_do, EW); mbar_init(bar_dz2, EW); mbar_init(bar_dz1, EW);
    mbar_init(bar_d0, 1); mbar_init(bar_d1, 1); mbar_init(bar_d2, 1); mbar_init(bar_g2, 1); mbar_init(bar_g1, 1);
    mbar_init(bar_wg, 1);
    fence_barrier_init();
  }
  if (warp == 0) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot_g;
  const uint32_t tR0 = tmem, tR1 = tmem + 128, tWG1 = tmem + 256, tWG2 = tmem + 384, tWG0 = tmem + 448, tWB1 = tmem + 464, tWB2 = tmem + 480;

  int f_first, f_step, nslots, slot;
  if (G >= F) { f_first = c % F; f_step = F * G; slot = c / F; nslots = (G - f_first + F - 1) / F; }
  else { f_first = c; f_step = G; slot = 0; nslots = 1; }

  constexpr uint32_t fmt = BF16 ? 1u : 0u;
  constexpr uint32_t id_kk_128 = umma_idesc(fmt, 0, 0, HID);
  constexpr uint32_t id_mm_128 = umma_idesc(fmt, 1, 1, HID), id_mm_64 = umma_idesc(fmt, 1, 1, EO),
                     id_mm_16 = umma_idesc(fmt, 1, 1, 16);
  uint32_t it = 0, fit = 0;
  const float S = Q.gscale, invS = 1.f / Q.gscale;

  for (int f = f_first; f < F; f += f_step, ++fit) {
    const bool any_tiles = slot < ntiles;
    if (warp == 0) {
      if (lane == 0) {
        load_weights(sb, maps, bar_w, f);
        mbar_wait_backoff(bar_w, fit & 1);
        bool first = true;
        if (any_tiles) {     // layer 0 of the feature's first tile; every later tile's layer 0 is issued one tile ahead (below)
          mbar_wait_backoff(bar_a0, it & 1); tc_fence_after_sync();
          issue_layer0<BF16>(sb, tR0, sb + ((it & 1) ? kOffBwdA0b : kOffA0)); umma_commit(bar_d0);
        }
        for (int t = slot; t < ntiles; t += nslots, ++it, first = false) {
          const uint32_t ph = it & 1;
          // ---- recompute forward
          const uint32_t a0 = sb + ((it & 1) ? kOffBwdA0b : kOffA0);
          const uint32_t h1buf = sb + ((it & 1) ? kOffBwdH1b : kOffH1);
          mbar_wait_backoff(bar_h1, ph); tc_fence_after_sync();
          issue_layer1<BF16>(sb, tR0, h1buf, a0); umma_commit(bar_d1);
          mbar_wait_backoff(bar_h2, ph); tc_fence_after_sync();
          issue_layer2<BF16>(sb, tR1, sb + kOffH2, a0); umma_commit(bar_d2);
          // ---- layer 2 backward: G2 = dO W2^T ; dW2 += h2^T dO
          mbar_wait_backoff(bar_do, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16<BF16>(tR1, umma_desc16((sb >> 4) + ((kOffDO + kk * 32) >> 4), 16, 1024),
                           umma_desc16((sb >> 4) + ((kOffW2 + kk * 32) >> 4), 16, 1024), id_kk_128, kk > 0 ? 1u : 0u);
          umma_commit(bar_g2);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tWG2, umma_desc16((sb >> 4) + ((kOffH2 + kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((sb >> 4) + ((kOffDO + kk * 2048) >> 4), kPanel, 1024), id_mm_64, (first && kk == 0) ? 0u : 1u);
          // db2 += dO^T [pe|1]: M = 128 is formed by dO (64 columns) and the panel that follows it in shared memory
          // (dz2, finite garbage at this point): TMEM lanes 64..127 of this accumulator are never read.
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tWB2, umma_desc16((sb >> 4) + ((kOffDO + kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16,
                           (first && kk == 0) ? 0u : 1u);
          // ---- layer 1 backward: G1 = dz2 W1^T ; dW1 += h1^T dz2 ; db1 += dz2^T [pe|1]
          mbar_wait_backoff(bar_dz2, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tR1, umma_desc16((sb >> 4) + ((kOffDZ2 + (kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024),
                           umma_desc16((sb >> 4) + ((kOffW1 + (kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024), id_kk_128,
                           kk > 0 ? 1u : 0u);
          umma_commit(bar_g1);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tWG1, umma_desc16((h1buf >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((sb >> 4) + ((kOffDZ2 + kk * 2048) >> 4), kPanel, 1024), id_mm_128, (first && kk == 0) ? 0u : 1u);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tWB1, umma_desc16((sb >> 4) + ((kOffDZ2 + kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16,
                           (first && kk == 0) ? 0u : 1u);
          // ---- the NEXT tile's layer 0 (its operand was staged long ago; R0 is free since this tile's h2 epilogue):
          // its first epilogue then follows this tile's last one without an MMA round trip in between
          if (t + nslots < ntiles) {
            mbar_wait_backoff(bar_a0, ph ^ 1); tc_fence_after_sync();
            issue_layer0<BF16>(sb, tR0, sb + (((it + 1) & 1) ? kOffBwdA0b : kOffA0)); umma_commit(bar_d0);
          }
          // ---- layer 0 backward: [dW0;db0]^T += dz1^T [pe|1]     (dz1 lives in the H2 buffer)
          mbar_wait_backoff(bar_dz1, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16<BF16>(tWG0, umma_desc16((sb >> 4) + ((kOffH2 + kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16,
                           (first && kk == 0) ? 0u : 1u);
          umma_commit(bar_wg);
          if (t + nslots >= ntiles) mbar_wait_backoff(bar_wg, ph);
        }
      } else {
        for (int t = slot; t < ntiles; t += nslots) ++it;
      }
      __syncwarp();
    } else {
      const int ew = warp - 1, q = warp & 3, csel = ew >> 2;
      const int et = ew * 32 + lane;
      const int r = q * 32 + lane;
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      const int d = P.fdim[f], xo = P.x_off[f];
      const float bs = Q.beta_dev[0] * Q.inv_batch * S;
      const int ar = et & (TM - 1), khalf = (et >> 7) & 1;             // first-layer operand: row / k-half staged by this thread
      const bool stager = et < 2 * TM;                           // 256 (row, k-half) slots of A0
      float xv[kMaxFeatDim];
      if (slot < ntiles) {                                       // operand of the first tile
        const long long grow0 = (long long)slot * TM + ar;
        if (stager) {
          load_x(grow0 < P.n ? P.x + grow0 * P.ldx + xo : nullptr, d, xv);
          write_a0_row<BF16>(sb + ((it & 1) ? kOffBwdA0b : kOffA0), ar, khalf, grow0 < P.n, xv, d, P.nfreq);
        }
        DIB_EPI_SIGNAL(bar_a0);
      }
      for (int t = slot; t < ntiles; t += nslots, ++it) {
        const uint32_t ph = it & 1;
        const long long row0 = (long long)t * TM;
        // prefetch this thread's slice of the upstream gradient (32 B of fp16) long before the (mu, logvar) stage
        uint4 dpre[ND / 8];
        {
          const long long g2 = row0 + r < P.n ? row0 + r : 0;
          if (Q.d_emb16) {
            const uint16_t* src = Q.d_emb16 + g2 * Q.ldd16 + f * 32 + csel * ND;
#pragma unroll
            for (int u = 0; u < ND / 8; ++u) dpre[u] = *reinterpret_cast<const uint4*>(src + u * 8);
          }
        }
        const bool has_next = t + nslots < ntiles;
        const long long grow_n = (long long)(t + nslots) * TM + ar;
        if (has_next && stager) load_x(grow_n < P.n ? P.x + grow_n * P.ldx + xo : nullptr, d, xv);   // prefetch the next tile's x
        const uint32_t h1buf = sb + ((it & 1) ? kOffBwdH1b : kOffH1);
        const long long grow = row0 + r;
        const bool valid = grow < P.n;
        const float* ep = (P.eps && valid) ? P.eps + (grow * F + f) * 32 + csel * ND : P.eps;
        float nrm[ND];
        mbar_wait(bar_d0, ph); tc_fence_after_sync();
        epilogue_to_tile<BF16, RELU, NC>(tR0 + lane_addr, h1buf, r, csel * NC, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h1);
        noise8(ep, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, csel * ND, valid,
               *reinterpret_cast<float(*)[8]>(&nrm[0]));                                                  // while layer 1 runs
        mbar_wait(bar_d1, ph); tc_fence_after_sync();
        // the previous tile's weight-gradient MMAs read H2 (dz1), DO, DZ2 and the other A0 buffer: retired from here on
        if (t != slot) { mbar_wait(bar_wg, ph ^ 1); tc_fence_after_sync(); }
        epilogue_to_tile<BF16, RELU, NC>(tR0 + lane_addr, sb + kOffH2, r, csel * NC, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h2);
        if (has_next) {      // stage the next tile's first-layer operand in the other A0 buffer
          if (stager) write_a0_row<BF16>(sb + (((it + 1) & 1) ? kOffBwdA0b : kOffA0), ar, khalf, grow_n < P.n, xv, d, P.nfreq);
          DIB_EPI_SIGNAL(bar_a0);
        }
        if constexpr (ND == 16)
          noise8(ep ? ep + 8 : nullptr, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, csel * ND + 8, valid,
                 *reinterpret_cast<float(*)[8]>(&nrm[ND - 8]));                                           // while layer 2 runs
        // ---- (mu, logvar) -> d(mu), d(logvar) -> DO tile   (8 embedding dims at a time to bound live registers)
        mbar_wait(bar_d2, ph); tc_fence_after_sync();
        {
          const float* du = Q.d_emb ? Q.d_emb + (valid ? grow : 0) * Q.ldd + f * 32 + csel * ND : nullptr;
          const bool du16 = Q.d_emb16 != nullptr;
          const uint32_t do_row = sb + kOffDO + r * 128;
          const int r7 = r & 7;
#pragma unroll
          for (int e8 = 0; e8 < ND; e8 += 8) {
            uint32_t vm[8], vl[8];
            tmem_ld_32x32b_x8(tR1 + lane_addr + csel * ND + e8, vm);
            tmem_ld_32x32b_x8(tR1 + lane_addr + 32 + csel * ND + e8, vl);
            tmem_ld_wait();
            float dm[8], dl[8];
#pragma unroll
            for (int e0 = 0; e0 < 8; e0 += 4) {
              float g[4];
              if (du16) {
                const uint4 gq = dpre[e8 >> 3];
                uint32_t w0 = e0 == 0 ? gq.x : gq.z, w1 = e0 == 0 ? gq.y : gq.w;
                unpack2<BF16>(w0, g[0], g[1]); unpack2<BF16>(w1, g[2], g[3]);
              } else {
                const float4 g4 = *reinterpret_cast<const float4*>(du + e8 + e0);
                g[0] = g4.x * S; g[1] = g4.y * S; g[2] = g4.z * S; g[3] = g4.w * S;
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float mu = __uint_as_float(vm[e0 + j]), lv = __uint_as_float(vl[e0 + j]);
                const float sg = expf(0.5f * lv);
                const float gs = g[j];
                const float nz = nrm[e8 + e0 + j];
                dm[e0 + j] = valid ? fmaf(bs, mu, gs) : 0.f;
                dl[e0 + j] = valid ? fmaf(gs * nz, 0.5f * sg, bs * 0.5f * (sg * sg - 1.f)) : 0.f;
              }
            }
            const int cm = (csel * ND + e8) >> 3, cl = (32 + csel * ND + e8) >> 3;       // 16-byte chunk indices
            st_shared_v4(do_row + ((cm ^ r7) << 4), pack2<BF16>(dm[0], dm[1]), pack2<BF16>(dm[2], dm[3]),
                         pack2<BF16>(dm[4], dm[5]), pack2<BF16>(dm[6], dm[7]));
            st_shared_v4(do_row + ((cl ^ r7) << 4), pack2<BF16>(dl[0], dl[1]), pack2<BF16>(dl[2], dl[3]),
                         pack2<BF16>(dl[4], dl[5]), pack2<BF16>(dl[6], dl[7]));
          }
        }
        DIB_EPI_SIGNAL(bar_do);
        // ---- dz2 = G2 * act'(h2)
        mbar_wait(bar_g2, ph); tc_fence_after_sync();
        dgrad_epilogue<BF16, RELU, NC>(tR1 + lane_addr, sb + kOffH2, sb + kOffDZ2, r, csel * NC, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_dz2);
        // ---- dz1 = G1 * act'(h1)  -> H2 buffer (free: the dW2 MMAs that read h2 retired before G1 completed)
        mbar_wait(bar_g1, ph); tc_fence_after_sync();
        dgrad_epilogue<BF16, RELU, NC>(tR1 + lane_addr, h1buf, sb + kOffH2, r, csel * NC, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_dz1);
      }
      // every weight-gradient MMA of this feature has retired before the accumulators are read back
      if (any_tiles) { mbar_wait(bar_wg, (it - 1) & 1); tc_fence_after_sync(); }
      // ================= flush this (feature, slot)'s weight-gradient partials (scaled back by 1/S)
      float* part = Q.part + (long long)slot * Q.split_stride;
      const int w_in = d * P.nfreq;
      {
        float* dst = part + Q.w1_off[f] + (long long)r * HID + csel * NC;          // dW1[h1=r][h2 cols csel*NC..]
#pragma unroll
        for (int hh = 0; hh < NC / 32; ++hh) {
          uint32_t v[32];
          if (any_tiles) { tmem_ld_32x32b_x32(tWG1 + lane_addr + csel * NC + hh * 32, v); tmem_ld_wait(); }
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(dst + hh * 32 + j) = any_tiles
                ? make_float4(__uint_as_float(v[j]) * invS, __uint_as_float(v[j + 1]) * invS,
                              __uint_as_float(v[j + 2]) * invS, __uint_as_float(v[j + 3]) * invS)
                : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float* dst2 = part + Q.w2_off[f] + (long long)r * EO + csel * NW2;          // dW2[h2=r][o cols csel*NW2..]
#pragma unroll
        for (int hh = 0; hh < NW2 / 16; ++hh) {
          uint32_t v[16];
          if (any_tiles) { tmem_ld_32x32b_x16(tWG2 + lane_addr + csel * NW2 + hh * 16, v); tmem_ld_wait(); }
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(dst2 + hh * 16 + j) = any_tiles
                ? make_float4(__uint_as_float(v[j]) * invS, __uint_as_float(v[j + 1]) * invS,
                              __uint_as_float(v[j + 2]) * invS, __uint_as_float(v[j + 3]) * invS)
                : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (csel == 0) {
          // dW0[k][h1=r] (k < w_in), db0[r] = column w_in of dW0p^T; db1[h2=r] = column w_in of dz2^T [pe|1]
          uint32_t v0[16], v1[16];
          if (any_tiles) { tmem_ld_32x32b_x16(tWG0 + lane_addr, v0); tmem_ld_32x32b_x16(tWB1 + lane_addr, v1); tmem_ld_wait(); }
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            const float val = any_tiles ? __uint_as_float(v0[k]) * invS : 0.f;
            if (k < w_in) part[Q.w0_off[f] + (long long)k * HID + r] = val;
            else if (k == w_in) part[Q.b0_off[f] + r] = val;
          }
          float b1v = 0.f;
#pragma unroll
          for (int k = 0; k < 16; ++k) if (k == w_in) b1v = any_tiles ? __uint_as_float(v1[k]) * invS : 0.f;
          part[P.b1_off[f] + r] = b1v;
          if (r < EO) {                                     // db2[o = r]: lanes 0..63 of the db2 accumulator
            uint32_t v2[16];
            if (any_tiles) { tmem_ld_32x32b_x16(tWB2 + lane_addr, v2); tmem_ld_wait(); }
            float b2v = 0.f;
#pragma unroll
            for (int k = 0; k < 16; ++k) if (k == w_in) b2v = any_tiles ? __uint_as_float(v2[k]) * invS : 0.f;
            part[P.b2_off[f] + r] = b2v;
          }
        }
      }
      tc_fence_before_sync();
      asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory");
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) { tc_fence_after_sync(); tmem_dealloc(tmem, 512); }
}

// ====================================================================================================
// backward, version 2: the per-tile chain of version 1 (five MMA <-> epilogue round trips, one tile in flight) is cut
// into two chains that run CONCURRENTLY on consecutive tiles, each with its own MMA-issuing thread, its own epilogue
// warps and its own TMEM region:
//   chain A (tile i)  : x -> [pe|1] -> D0 -> h1 -> D1 -> h2 -> D2 = (mu|logvar) -> d(mu|logvar) = dO      [8 warps]
//   chain B (tile i-1): G2 = dO W2^T -> dz2 = G2*act'(h2) -> G1 = dz2 W1^T -> dz1 = G1*act'(h1); all wgrad MMAs [4 warps]
// so the tile time is max(A, B) instead of A + B and two sets of warps keep the issue slots busy.  What makes two
// tiles fit: dz2 / dz1 are written IN PLACE over h2 / h1 (their last reader, the dW2 / dW1 MMA, has retired by then),
// so a tile needs h1 + h2 = 64 KB and two of them plus three 4 KB [pe|1] operands, one dO tile and the 58 KB of
// weights are 214 KB.
// TMEM: [0,128) chain A (D0, D1, D2) | [128,256) chain B (G2, G1) | [256,496) weight-gradient accumulators (as v1).
// Warps: 0 MMA issuer A (+ weight TMA) | 1 MMA issuer B | 2 TMEM owner | 3 idle | 4..11 chain-A epilogue | 12..15 chain B.
// ====================================================================================================
constexpr int kV2OffDO = kOffA0;                       // 58 KB: [128 x 64] one panel (db2 reads 16 KB past it: A0s + h1)
constexpr int kV2OffA0 = kV2OffDO + kPanel;            // THREE [pe|1] operands, 4 KB each (tile i + 1's is staged while tile i - 1 may
                                                       // still be in chain B: a third buffer keeps chain A from waiting on it)
constexpr int kV2OffH1 = kV2OffA0 + 3 * (2 * TM * 16); // 86 KB, 1024-aligned; h1[0], h1[1]
constexpr int kV2OffH2 = kV2OffH1 + 2 * (2 * kPanel);  // h2[0], h2[1]
constexpr int kV2OffBar = kV2OffH2 + 2 * (2 * kPanel); // 210 KB
static_assert(kV2OffH1 % 1024 == 0 && kV2OffDO % 1024 == 0, "operand tiles must be 1024-byte aligned");
constexpr int kV2CtrlEA = 4 + 8;               // control warpgroup + chain-A epilogue warps; chain B adds EBW (4 or 8) warps

// gradient * act'(h) IN PLACE: the 128-byte row chunk of h is read, the gated 16-bit gradient is written back to the
// same address (same thread), NC columns starting at col0.
template <bool BF16, bool RELU, int NC>
__device__ __forceinline__ void dgrad_inplace(uint32_t taddr, uint32_t tile, int r, int col0, int act, float alpha) {
  constexpr int CH = 32;
#pragma unroll
  for (int hh = 0; hh < NC / CH; ++hh) {
    uint32_t v[CH];
    tmem_ld_32x32b_x32(taddr + col0 + hh * CH, v);
    uint32_t hv[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) ld_shared_v4(tile_chunk_addr(tile, r, col0 + hh * CH + j * 8), hv[j]);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float g0 = __uint_as_float(v[j * 8 + 2 * k]), g1 = __uint_as_float(v[j * 8 + 2 * k + 1]);
        if constexpr (RELU) {
          o[k] = relu_gate2<BF16>(pack2<BF16>(g0, g1), hv[j][k]);
        } else {
          float h0, h1;
          unpack2<BF16>(hv[j][k], h0, h1);
          o[k] = pack2<BF16>(g0 * dib_act_grad(act, h0, alpha), g1 * dib_act_grad(act, h1, alpha));
        }
      }
      st_shared_v4(tile_chunk_addr(tile, r, col0 + hh * CH + j * 8), o[0], o[1], o[2], o[3]);
    }
  }
}

template <bool BF16, bool RELU, bool EPS16, int EBW>
__global__ void __launch_bounds__(32 * (kV2CtrlEA + EBW), 1)
dib_enc_fused_bwd2_kernel(const __grid_constant__ WeightMaps maps, const EncFusedBwdParams Q) {
  const EncFusedParams& P = Q.f;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar = sb + kV2OffBar;
  const uint32_t bar_w = bar, bar_a0 = bar + 8, bar_d0 = bar + 16, bar_h1 = bar + 24, bar_d1 = bar + 32,
                 bar_h2 = bar + 40, bar_d2 = bar + 48, bar_do = bar + 56, bar_dofree = bar + 64, bar_g2 = bar + 72,
                 bar_dz2 = bar + 80, bar_g1 = bar + 88, bar_dw1 = bar + 96, bar_dz1 = bar + 104, bar_wg0 = bar + 112 /* [2] */,
                 tmem_slot = bar + 128, bar_a0t = bar + 136;
  volatile uint32_t* tmem_slot_g = reinterpret_cast<volatile uint32_t*>(sg + kV2OffBar + 128);
  constexpr int kEA = 8, kEB = EBW;   // epilogue warps of chain A / chain B
  constexpr int kV2Threads = 32 * (kV2CtrlEA + EBW);
  static_assert(EBW == 4 || EBW == 8, "chain B: 4 warps (a full row per thread) or 8 (half a row)");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int G = gridDim.x, c = blockIdx.x, F = P.F;
  const int ntiles = (int)((P.n + TM - 1) / TM);
  const unsigned int nstep = P.step + (P.step_dev ? P.step_dev[0] : 0u);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&maps.w0); tma_prefetch_desc(&maps.w1); tma_prefetch_desc(&maps.w2);
    tma_prefetch_desc(&maps.b1); tma_prefetch_desc(&maps.b2);
    mbar_init(bar_w, 1);
    mbar_init(bar_a0, kEA); mbar_init(bar_h1, kEA); mbar_init(bar_h2, kEA); mbar_init(bar_do, kEA);
    mbar_init(bar_dz2, kEB); mbar_init(bar_dz1, kEB);
    mbar_init(bar_d0, 1); mbar_init(bar_d1, 1); mbar_init(bar_d2, 1); mbar_init(bar_dofree, 1); mbar_init(bar_g2, 1);
    mbar_init(bar_g1, 1); mbar_init(bar_dw1, 1); mbar_init(bar_wg0, 1); mbar_init(bar_wg0 + 8, 1);
    mbar_init(bar_a0t, 1);
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot_g;
  const uint32_t tR0 = tmem, tR1 = tmem + 128, tWG1 = tmem + 256, tWG2 = tmem + 384, tWG0 = tmem + 448, tWB1 = tmem + 464, tWB2 = tmem + 480;

  int f_first, f_step, nslots, slot;
  if (G >= F) { f_first = c % F; f_step = F * G; slot = c / F; nslots = (G - f_first + F - 1) / F; }
  else { f_first = c; f_step = G; slot = 0; nslots = 1; }

  constexpr uint32_t fmt = BF16 ? 1u : 0u;
  constexpr uint32_t id_kk_128 = umma_idesc(fmt, 0, 0, HID);
  constexpr uint32_t id_mm_128 = umma_idesc(fmt, 1, 1, HID), id_mm_64 = umma_idesc(fmt, 1, 1, EO),
                     id_mm_16 = umma_idesc(fmt, 1, 1, 16);
  uint32_t it = 0, fit = 0;          // running tile / feature counters of this CTA (barrier phases)
  const float S = Q.gscale, invS = 1.f / Q.gscale;
  auto a0_of = [&](uint32_t i) { return sb + kV2OffA0 + (i % 3u) * (2 * TM * 16); };
  auto h1_of = [&](uint32_t i) { return sb + kV2OffH1 + (i & 1) * (2 * kPanel); };
  auto h2_of = [&](uint32_t i) { return sb + kV2OffH2 + (i & 1) * (2 * kPanel); };
  const uint32_t sDO = sb + kV2OffDO;

  // Each role runs its own copy of the feature loop INSIDE its branch, behind a setmaxnreg that rebalances the register
  // file between the warpgroups (launched with 128 per thread; per scheduler: 1 control warp x 56 + 2 chain-A warps x 168
  // + 1 chain-B warp x 112 = 504 <= 512).  ptxas allocates each branch against its own budget only if the branches do not
  // merge before the kernel's trivial tail.
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");     // per scheduler: 56 + 2 x 168 + 112 (EBW 4) | 56 + 2 x 128 + 2 x 96 (EBW 8) <= 512
    for (int f = f_first; f < F; f += f_step, ++fit) {
      const int ntl = slot < ntiles ? (ntiles - slot + nslots - 1) / nslots : 0;   // tiles of this (feature, CTA)
      const bool any_tiles = ntl > 0; (void)any_tiles;
      if (warp == 0) {
      // ================= MMA issuer A: the forward recompute chain
      // (the whole warp walks the issue sequence -- uniform control flow keeps descriptors and barrier addresses in uniform
      //  registers -- and one elected lane executes each tcgen05 instruction; TMA loads stay on lane 0)
      {
        if (lane == 0) load_weights(sb, maps, bar_w, f);
        // hand-off mode: the [pe|1] operand of a tile arrives by TMA from the forward kernel's copy (two 2 KB k-halves)
        auto load_a0 = [&](uint32_t i, int k) {
          if (lane == 0) {
            const int row0 = (slot + k * nslots) * TM;
            mbar_expect_tx(bar_a0t, 2 * TM * 16);
            tma_load_3d(a0_of(i), &maps.a0lo, bar_a0t, 0, row0, 2 * f);
            tma_load_3d(a0_of(i) + TM * 16, &maps.a0lo, bar_a0t, 0, row0, 2 * f + 1);
          }
          __syncwarp();
        };
        if (EPS16 && ntl > 0) load_a0(it, 0);
        __syncwarp();
        mbar_wait_backoff(bar_w, fit & 1);
        for (int k = 0; k < ntl; ++k) {
          const uint32_t i = it + k, ph = i & 1;
          const uint32_t a0 = a0_of(i);
          if (EPS16) mbar_wait_backoff(bar_a0t, ph);
          mbar_wait_backoff(bar_a0, ph); tc_fence_after_sync();
          issue_layer0<BF16, true>(sb, tR0, a0); umma_commit_w(bar_d0);
          mbar_wait_backoff(bar_h1, ph); tc_fence_after_sync();
          // chain A has started tile i, so tile i - 2 has retired and operand buffer (i + 1) % 3 is free
          if (EPS16 && k + 1 < ntl) load_a0(i + 1, k + 1);
          issue_layer1<BF16, true>(sb, tR0, h1_of(i), a0); umma_commit_w(bar_d1);
          mbar_wait_backoff(bar_h2, ph); tc_fence_after_sync();
          issue_layer2<BF16, true>(sb, tR0, h2_of(i), a0); umma_commit_w(bar_d2);
        }
      }
      __syncwarp();
      } else if (warp == 1) {
      // ================= MMA issuer B: dgrad + every weight-gradient MMA
      {                                     // whole warp, elected lane issues (see issuer A)
        mbar_wait_backoff(bar_w, fit & 1);
        for (int k = 0; k < ntl; ++k) {
          const uint32_t i = it + k, ph = i & 1;
          const uint32_t a0 = a0_of(i), h1 = h1_of(i), h2 = h2_of(i);
          const bool first = k == 0;
          // ---- layer 2 backward: G2 = dO W2^T ; dW2 += h2^T dO ; db2 += dO^T [pe|1]
          mbar_wait_backoff(bar_do, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16_w(tR1, umma_desc16((sDO >> 4) + ((kk * 32) >> 4), 16, 1024), umma_desc16((sb >> 4) + ((kOffW2 + kk * 32) >> 4), 16, 1024),
                           id_kk_128, kk > 0 ? 1u : 0u);
          umma_commit_w(bar_g2);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tWG2, umma_desc16((h2 >> 4) + ((kk * 2048) >> 4), kPanel, 1024), umma_desc16((sDO >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           id_mm_64, (first && kk == 0) ? 0u : 1u);
          // M = 128 is formed by dO (64 columns) and the 16 KB that follow it in shared memory (the [pe|1] operands and
          // the start of h1[0]): TMEM lanes 64..127 of this accumulator are never read.
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tWB2, umma_desc16((sDO >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16, (first && kk == 0) ? 0u : 1u);
          umma_commit_w(bar_dofree);          // dO is free again; h2 may be overwritten by dz2
          // ---- layer 1 backward: G1 = dz2 W1^T ; dW1 += h1^T dz2 ; db1 += dz2^T [pe|1]      (dz2 lives in the h2 buffer)
          mbar_wait_backoff(bar_dz2, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tR1, umma_desc16((h2 >> 4) + (((kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024),
                           umma_desc16((sb >> 4) + ((kOffW1 + (kk >> 2) * kPanel + (kk & 3) * 32) >> 4), 16, 1024), id_kk_128, kk > 0 ? 1u : 0u);
          umma_commit_w(bar_g1);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tWG1, umma_desc16((h1 >> 4) + ((kk * 2048) >> 4), kPanel, 1024), umma_desc16((h2 >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           id_mm_128, (first && kk == 0) ? 0u : 1u);
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tWB1, umma_desc16((h2 >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16, (first && kk == 0) ? 0u : 1u);
          umma_commit_w(bar_dw1);             // h1 may be overwritten by dz1
          // ---- layer 0 backward: [dW0;db0]^T += dz1^T [pe|1]      (dz1 lives in the h1 buffer)
          mbar_wait_backoff(bar_dz1, ph); tc_fence_after_sync();
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_f16_w(tWG0, umma_desc16((h1 >> 4) + ((kk * 2048) >> 4), kPanel, 1024),
                           umma_desc16((a0 >> 4) + ((kk * 256) >> 4), 128, TM * 16, kLayoutNone), id_mm_16, (first && kk == 0) ? 0u : 1u);
          umma_commit_w(bar_wg0 + 8 * (i & 1));   // buffer set (i & 1) is free for tile i + 2
        }
      }
      __syncwarp();
      }
      it += (uint32_t)ntl;
      // accumulators flushed, every MMA retired: the next feature may reload the weights (all 16 warps meet here)
      asm volatile("bar.sync 0, %0;" ::"n"(kV2Threads) : "memory");
      tc_fence_after_sync();
    }
  } else if (warp < 4 + kEA) {
    if constexpr (EBW == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 128;");
    for (int f = f_first; f < F; f += f_step, ++fit) {
      const int ntl = slot < ntiles ? (ntiles - slot + nslots - 1) / nslots : 0;   // tiles of this (feature, CTA)
      const bool any_tiles = ntl > 0; (void)any_tiles;
      {
      // ================= chain A epilogue warps: 4 TMEM lane quarters x 2 column halves
      const int ew = warp - 4, q = warp & 3, csel = ew >> 2;
      const int et = ew * 32 + lane;
      const int r = q * 32 + lane;
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      const int d = P.fdim[f], xo = P.x_off[f];
      const float bs = Q.beta_dev[0] * Q.inv_batch * S;
      const int ar = et & (TM - 1), khalf = et >> 7;          // [pe|1] operand: (row, k-half) staged by this thread
      float xv[kMaxFeatDim];
      if (any_tiles) {                                        // operand of the feature's first tile (both buffer sets are drained)
        if constexpr (!EPS16) {                               // (hand-off mode: issuer A loads it by TMA; the signal only frees R0)
          const long long grow0 = (long long)slot * TM + ar;
          load_x(grow0 < P.n ? P.x + grow0 * P.ldx + xo : nullptr, d, xv);
          write_a0_row<BF16>(a0_of(it), ar, khalf, grow0 < P.n, xv, d, P.nfreq);
        }
        DIB_EPI_SIGNAL(bar_a0);
      }
      for (int k = 0; k < ntl; ++k) {
        const uint32_t i = it + k, ph = i & 1;
        const int t = slot + k * nslots;
        const long long row0 = (long long)t * TM;
        const long long grow = row0 + r;
        const bool valid = grow < P.n;
        const bool has_next = k + 1 < ntl;
        const long long grow_n = (long long)(t + nslots) * TM + ar;
        // prefetch this thread's 16 embedding dims of the upstream gradient and the next tile's x
        uint4 dpre[2];
        if (Q.d_emb16) {
          const uint16_t* src = Q.d_emb16 + (valid ? grow : 0) * Q.ldd16 + f * 32 + csel * 16;
          uint32_t dw[8];
          dib_ld_global_v8(src, dw);
          dpre[0] = make_uint4(dw[0], dw[1], dw[2], dw[3]); dpre[1] = make_uint4(dw[4], dw[5], dw[6], dw[7]);
        }
        if constexpr (!EPS16) { if (has_next) load_x(grow_n < P.n ? P.x + grow_n * P.ldx + xo : nullptr, d, xv); }
        const float* ep = (P.eps && valid) ? P.eps + (grow * F + f) * 32 + csel * 16 : P.eps;
        uint32_t nz16[8];            // this thread's 16 noise values, packed 16-bit (they multiply a 16-bit gradient)
        constexpr bool have_eps16 = EPS16;
        if constexpr (have_eps16) {            // written by this step's forward kernel: 32 B per thread instead of 4 Philox calls
          const uint16_t* e16 = P.eps16 + ((valid ? grow : 0) * F + f) * 32 + csel * 16;
          dib_ld_global_v8(e16, nz16);
        }
        // buffer set (i & 1) was last used by tile i - 2: all of its MMAs (chain B commits last) have retired
        if (i >= 2) { mbar_wait(bar_wg0 + 8 * (i & 1), ((i >> 1) - 1) & 1); }
        mbar_wait(bar_d0, ph); tc_fence_after_sync();
        epilogue_to_tile<BF16, RELU>(tR0 + lane_addr, h1_of(i), r, csel * 64, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h1);
        if constexpr (!have_eps16) {                                                                // while layer 1 runs
          float nrm[8];
          noise8(ep, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, csel * 16, valid, nrm);
#pragma unroll
          for (int j = 0; j < 4; ++j) nz16[j] = pack2<BF16>(nrm[2 * j], nrm[2 * j + 1]);
        }
        mbar_wait(bar_d1, ph); tc_fence_after_sync();
        epilogue_to_tile<BF16, RELU>(tR0 + lane_addr, h2_of(i), r, csel * 64, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_h2);
        if constexpr (!have_eps16) {                                                                // while layer 2 runs
          float nrm[8];
          noise8(ep ? ep + 8 : nullptr, P.seed, nstep, P.sample_offset + (unsigned long long)grow, f, csel * 16 + 8, valid, nrm);
#pragma unroll
          for (int j = 0; j < 4; ++j) nz16[4 + j] = pack2<BF16>(nrm[2 * j], nrm[2 * j + 1]);
        }
        if constexpr (!EPS16) {
          if (has_next)      // stage the next tile's [pe|1] operand: buffer (i + 1) % 3 was last read by tile i - 2 (retired, see above)
            write_a0_row<BF16>(a0_of(i + 1), ar, khalf, grow_n < P.n, xv, d, P.nfreq);
        }
        // ---- (mu, logvar) -> d(mu), d(logvar) -> dO tile, 8 embedding dims at a time.  The dO buffer is single: wait
        // until the previous tile's dO has been consumed.  After the LAST TMEM load chain A's region is free for the
        // next tile's layer 0, which then runs under the second half of this stage.
        mbar_wait(bar_d2, ph); tc_fence_after_sync();
        if (i >= 1) { mbar_wait(bar_dofree, (i - 1) & 1); }
        {
          const float* du = Q.d_emb ? Q.d_emb + (valid ? grow : 0) * Q.ldd + f * 32 + csel * 16 : nullptr;
          const bool du16 = Q.d_emb16 != nullptr;
          const uint32_t do_row = sDO + r * 128;
          const int r7 = r & 7;
          // rows past the batch end contribute nothing: their upstream gradient and KL weight are zeroed once, here, instead of
          // selecting per element.  With hs = sigma / 2 = exp2(lv * log2(e)/2 - 1):
          //   d(mu)     = bs * mu + g
          //   d(logvar) = g * eps * sigma/2 + bs/2 * (sigma^2 - 1) = (g * eps) * hs + ((2 bs * hs) * hs - bs/2)
          const float bsv = valid ? bs : 0.f, gS = valid ? S : 0.f, bs2 = 2.f * bsv, hb = 0.5f * bsv;
          if (!valid) { dpre[0] = make_uint4(0u, 0u, 0u, 0u); dpre[1] = make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
          for (int e8 = 0; e8 < 16; e8 += 8) {
            uint32_t vm[8], vl[8];
            tmem_ld_32x32b_x8(tR0 + lane_addr + csel * 16 + e8, vm);
            tmem_ld_32x32b_x8(tR0 + lane_addr + 32 + csel * 16 + e8, vl);
            tmem_ld_wait();
            if (e8 == 8) {
              if (has_next) { DIB_EPI_SIGNAL(bar_a0); }
              else { tc_fence_before_sync(); }
            }
            float dm[8], dl[8];
#pragma unroll
            for (int e0 = 0; e0 < 8; e0 += 4) {
              float g[4], nz[4];
              if (du16) {
                const uint4 gq = dpre[e8 >> 3];
                uint32_t w0 = e0 == 0 ? gq.x : gq.z, w1 = e0 == 0 ? gq.y : gq.w;
                unpack2<BF16>(w0, g[0], g[1]); unpack2<BF16>(w1, g[2], g[3]);
              } else {
                const float4 g4 = *reinterpret_cast<const float4*>(du + e8 + e0);
                g[0] = g4.x * gS; g[1] = g4.y * gS; g[2] = g4.z * gS; g[3] = g4.w * gS;
              }
              unpack2<BF16>(nz16[(e8 + e0) >> 1], nz[0], nz[1]); unpack2<BF16>(nz16[((e8 + e0) >> 1) + 1], nz[2], nz[3]);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float mu = __uint_as_float(vm[e0 + j]), lv = __uint_as_float(vl[e0 + j]);
                float hs;
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(hs) : "f"(fmaf(lv, 0.72134752044448170f, -1.f)));
                dm[e0 + j] = fmaf(bsv, mu, g[j]);
                dl[e0 + j] = fmaf(g[j] * nz[j], hs, fmaf(bs2 * hs, hs, -hb));
              }
            }
            const int cm = (csel * 16 + e8) >> 3, cl = (32 + csel * 16 + e8) >> 3;       // 16-byte chunk indices
            st_shared_v4(do_row + ((cm ^ r7) << 4), pack2<BF16>(dm[0], dm[1]), pack2<BF16>(dm[2], dm[3]),
                         pack2<BF16>(dm[4], dm[5]), pack2<BF16>(dm[6], dm[7]));
            st_shared_v4(do_row + ((cl ^ r7) << 4), pack2<BF16>(dl[0], dl[1]), pack2<BF16>(dl[2], dl[3]),
                         pack2<BF16>(dl[4], dl[5]), pack2<BF16>(dl[6], dl[7]));
          }
        }
        DIB_EPI_SIGNAL(bar_do);
      }
      // every MMA of this feature has retired (chain B's last commit) before the accumulators are read back
      if (any_tiles) { const uint32_t il = it + ntl - 1; mbar_wait(bar_wg0 + 8 * (il & 1), (il >> 1) & 1); tc_fence_after_sync(); }
      // ---- flush dW1[h1 = r][h2 cols csel*64 ..] (scaled back by 1/S)
      {
        float* part = Q.part + (long long)slot * Q.split_stride;
        float* dst = part + Q.w1_off[f] + (long long)r * HID + csel * 64;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t v[32];
          if (any_tiles) { tmem_ld_32x32b_x32(tWG1 + lane_addr + csel * 64 + hh * 32, v); tmem_ld_wait(); }
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(dst + hh * 32 + j) = any_tiles
                ? make_float4(__uint_as_float(v[j]) * invS, __uint_as_float(v[j + 1]) * invS,
                              __uint_as_float(v[j + 2]) * invS, __uint_as_float(v[j + 3]) * invS)
                : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      tc_fence_before_sync();
      }
      it += (uint32_t)ntl;
      // accumulators flushed, every MMA retired: the next feature may reload the weights (all 16 warps meet here)
      asm volatile("bar.sync 0, %0;" ::"n"(kV2Threads) : "memory");
      tc_fence_after_sync();
    }
  } else {
    if constexpr (EBW == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
    for (int f = f_first; f < F; f += f_step, ++fit) {
      const int ntl = slot < ntiles ? (ntiles - slot + nslots - 1) / nslots : 0;   // tiles of this (feature, CTA)
      const bool any_tiles = ntl > 0; (void)any_tiles;
      {
      // ================= chain B epilogue warps: one full row (128 columns) per thread, or half a row with 8 warps
      constexpr int NCB = HID * 4 / EBW;               // columns per thread
      const int q = warp & 3, cselb = (warp - 4 - kEA) >> 2;
      const int r = q * 32 + lane;
      const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
      const int d = P.fdim[f];
      for (int k = 0; k < ntl; ++k) {
        const uint32_t i = it + k, ph = i & 1;
        // ---- dz2 = G2 * act'(h2), in place over h2 (its last reader, the dW2 MMA, has retired: bar_dofree)
        mbar_wait(bar_g2, ph); mbar_wait(bar_dofree, ph); tc_fence_after_sync();
        dgrad_inplace<BF16, RELU, NCB>(tR1 + lane_addr, h2_of(i), r, cselb * NCB, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_dz2);
        // ---- dz1 = G1 * act'(h1), in place over h1 (dW1 has retired: bar_dw1)
        mbar_wait(bar_g1, ph); mbar_wait(bar_dw1, ph); tc_fence_after_sync();
        dgrad_inplace<BF16, RELU, NCB>(tR1 + lane_addr, h1_of(i), r, cselb * NCB, P.act, P.alpha);
        DIB_EPI_SIGNAL(bar_dz1);
      }
      if (any_tiles) { const uint32_t il = it + ntl - 1; mbar_wait(bar_wg0 + 8 * (il & 1), (il >> 1) & 1); tc_fence_after_sync(); }
      // ---- flush dW2, [dW0;db0], db1, db2 (cold path: the first four chain-B warps cover the 128 TMEM lanes)
      if (cselb == 0) {
      float* part = Q.part + (long long)slot * Q.split_stride;
      const int w_in = d * P.nfreq;
      float* dst2 = part + Q.w2_off[f] + (long long)r * EO;                        // dW2[h2 = r][0..64)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t v[32];
        if (any_tiles) { tmem_ld_32x32b_x32(tWG2 + lane_addr + hh * 32, v); tmem_ld_wait(); }
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst2 + hh * 32 + j) = any_tiles
              ? make_float4(__uint_as_float(v[j]) * invS, __uint_as_float(v[j + 1]) * invS,
                            __uint_as_float(v[j + 2]) * invS, __uint_as_float(v[j + 3]) * invS)
              : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      {
        // dW0[k][h1 = r] (k < w_in), db0[r] = column w_in of dW0p^T; db1[h2 = r] = column w_in of dz2^T [pe|1]
        uint32_t v0[16], v1[16];
        if (any_tiles) { tmem_ld_32x32b_x16(tWG0 + lane_addr, v0); tmem_ld_32x32b_x16(tWB1 + lane_addr, v1); tmem_ld_wait(); }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float val = any_tiles ? __uint_as_float(v0[k]) * invS : 0.f;
          if (k < w_in) part[Q.w0_off[f] + (long long)k * HID + r] = val;
          else if (k == w_in) part[Q.b0_off[f] + r] = val;
        }
        float b1v = 0.f;
#pragma unroll
        for (int k = 0; k < 16; ++k) if (k == w_in) b1v = any_tiles ? __uint_as_float(v1[k]) * invS : 0.f;
        part[P.b1_off[f] + r] = b1v;
        if (r < EO) {                                     // db2[o = r]: lanes 0..63 of the db2 accumulator
          uint32_t v2[16];
          if (any_tiles) { tmem_ld_32x32b_x16(tWB2 + lane_addr, v2); tmem_ld_wait(); }
          float b2v = 0.f;
#pragma unroll
          for (int k = 0; k < 16; ++k) if (k == w_in) b2v = any_tiles ? __uint_as_float(v2[k]) * invS : 0.f;
          part[P.b2_off[f] + r] = b2v;
        }
      }
      }
      tc_fence_before_sync();
          }
      it += (uint32_t)ntl;
      // accumulators flushed, every MMA retired: the next feature may reload the weights (all 16 warps meet here)
      asm volatile("bar.sync 0, %0;" ::"n"(kV2Threads) : "memory");
      tc_fence_after_sync();
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) { tc_fence_after_sync(); tmem_dealloc(tmem, 512); }
}

// ----------------------------------------------------------------------------------------------------
// fp32 master parameters -> packed 16-bit per-feature weights [W0p | W1 | W2 | Bb1 | Bb2]
// (bias of layer 0 folded into W0p row w_in; b1 / b2 in row w_in of the bias carriers)
// ----------------------------------------------------------------------------------------------------
template <bool BF16>
__global__ void dib_enc_pack_weights_kernel(const float* __restrict__ params, const long long* __restrict__ w0_off,
                                            const long long* __restrict__ b0_off, const long long* __restrict__ w1_off,
                                            const long long* __restrict__ b1_off, const long long* __restrict__ w2_off,
                                            const long long* __restrict__ b2_off, const int* __restrict__ fdim, int nfreq,
                                            float logvar_offset, uint16_t* __restrict__ out, float* __restrict__ zero, long long zero_n) {
  const int f = blockIdx.y;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  {   // the KL partial-sum table of the forward kernel that follows is cleared here (one launch instead of a memset node)
    const long long z = ((long long)f * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
    if (z < zero_n) zero[z] = 0.f;
  }
  if (i >= kPackElems) return;
  const int idx = i, w_in = fdim[f] * nfreq;
  float v;
  if (i < kW0Elems) {
    const int k = i / HID, n = i - k * HID;
    v = k < w_in ? params[w0_off[f] + (long long)k * HID + n] : (k == w_in ? params[b0_off[f] + n] : 0.f);
  } else if ((i -= kW0Elems) < kW1Elems) {
    v = params[w1_off[f] + i];
  } else if ((i -= kW1Elems) < kW2Elems) {
    v = params[w2_off[f] + i];
  } else if ((i -= kW2Elems) < kB1Elems) {
    const int k = i / HID, n = i - k * HID;
    v = k == w_in ? params[b1_off[f] + n] : 0.f;
  } else {
    i -= kB1Elems;
    const int k = i / EO, n = i - k * EO;
    v = k == w_in ? params[b2_off[f] + n] + (n >= EO / 2 ? logvar_offset : 0.f) : 0.f;
  }
  uint16_t h;
  if constexpr (BF16) { __nv_bfloat16 b = __float2bfloat16_rn(v); h = *reinterpret_cast<uint16_t*>(&b); }
  else { __half b = __float2half_rn(v); h = *reinterpret_cast<uint16_t*>(&b); }
  out[(long long)f * kPackElems + idx] = h;
}


// [rows x cols] 16-bit matrix per feature -> 3D map (col, row, feature), box 64 cols x rows x 1, SWIZZLE_128B
bool make_wmap(CUtensorMap* m, const uint16_t* base, int cols, int rows, int nfeat, bool bf16) {
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)nfeat};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)kPackElems * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return tensor_map_encode_fn()(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                      const_cast<uint16_t*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool make_all_maps(WeightMaps* m, const void* packed, int F, bool bf16) {
  const uint16_t* pk = static_cast<const uint16_t*>(packed);
  return make_wmap(&m->w0, pk, HID, K0, F, bf16) && make_wmap(&m->w1, pk + kW0Elems, HID, HID, F, bf16) &&
         make_wmap(&m->w2, pk + kW0Elems + kW1Elems, EO, HID, F, bf16) &&
         make_wmap(&m->b1, pk + kW0Elems + kW1Elems + kW2Elems, HID, K0, F, bf16) &&
         make_wmap(&m->b2, pk + kW0Elems + kW1Elems + kW2Elems + kB1Elems, EO, K0, F, bf16);
}

// [2 F (feature, k-half), n, 8] 16-bit hand-off buffer -- consecutive rows of one (feature, k-half) are consecutive 16-byte pieces,
// so the forward kernel's row-per-lane stores are fully coalesced -- as a 3D map (8 elements, row, plane), box 8 x 128 rows x 1:
// one box lands as the unswizzled [128 rows][16 B] half of the first-layer operand; rows past n are zero-filled (their ones column too)
bool make_a0_maps(WeightMaps* m, const void* a0g, long long n, int F, bool bf16) {
  cuuint64_t dims[3] = {8, (cuuint64_t)n, (cuuint64_t)(2 * F)};
  cuuint64_t strides[2] = {16, (cuuint64_t)n * 16};
  cuuint32_t box[3] = {8, (cuuint32_t)TM, 1};
  cuuint32_t es[3] = {1, 1, 1};
  const CUtensorMapDataType dt = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  if (tensor_map_encode_fn()(&m->a0lo, dt, 3, const_cast<void*>(a0g), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  m->a0hi = m->a0lo;
  return true;
}

void fill_params(EncFusedParams& P, const DibEncFusedDesc& d, const DibEncFusedIO& io) {
  P.x = io.x; P.ldx = io.ldx; P.x_off = d.x_off; P.fdim = d.fdim; P.nfreq = d.nfreq; P.params = io.params;
  P.b1_off = d.b1_off; P.b2_off = d.b2_off; P.eps = io.eps; P.seed = io.seed; P.step = io.step; P.step_dev = io.step_dev;
  P.sample_offset = io.sample_offset; P.emb = io.emb; P.ldemb = io.ldemb; P.user_emb = io.user_emb;
  P.kl_part = io.kl_part; P.kl_stride = io.kl_stride; P.F = d.F; P.n = io.n; P.act = d.act; P.alpha = d.alpha;
  P.round_emb = 1; P.emb16 = static_cast<uint16_t*>(io.emb16); P.ldemb16 = io.ldemb16; P.eps16 = static_cast<uint16_t*>(io.eps16); P.a0g = static_cast<uint16_t*>(io.a0g);
}

template <typename K, typename A>
cudaError_t launch_fused(K kern, int smem, int grid, const WeightMaps& m, const A& args, cudaStream_t st, int threads = kThreads) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, threads, smem, st>>>(m, args);
  dib_note_launch();
  return cudaGetLastError();
}

}  // namespace

// which backward kernel runs: 2 (default: two chains on consecutive tiles, 0.329 ms at C0) or 1 (the single-chain kernel of
// round 1, 0.438 ms); DIB_ENC_BWD=1|2 in the environment or dib_debug_set_variant(0, v)
static int g_enc_bwd_version = 0;
int dib_enc_bwd_version() {
  if (!g_enc_bwd_version) { const char* e = getenv("DIB_ENC_BWD"); g_enc_bwd_version = (e && e[0] == '1') ? 1 : 2; }
  return g_enc_bwd_version;
}
void dib_enc_bwd_set_version(int v) { g_enc_bwd_version = v == 1 ? 1 : 2; }

size_t dib_enc_fused_pack_bytes(int F) { return (size_t)F * kPackElems * 2; }
long long dib_enc_fused_pack_zero_capacity(int F) { return (long long)DIB_CEIL_DIV(kPackElems, 256) * 256 * F; }   // floats the pack kernel can also clear
int dib_enc_fused_fwd_ctas_per_sm() { return 2; }

cudaError_t dib_enc_fused_pack(const DibEncFusedDesc& d, const float* params, void* packed, float* zero, long long zero_n, cudaStream_t st) {
  dim3 grid(DIB_CEIL_DIV(kPackElems, 256), d.F);
  if (zero_n > (long long)grid.x * grid.y * 256) return cudaErrorInvalidValue;
  if (d.bf16)
    dib_enc_pack_weights_kernel<true><<<grid, 256, 0, st>>>(params, d.w0_off, d.b0_off, d.w1_off, d.b1_off, d.w2_off,
                                                           d.b2_off, d.fdim, d.nfreq, d.logvar_offset, static_cast<uint16_t*>(packed), zero, zero_n);
  else
    dib_enc_pack_weights_kernel<false><<<grid, 256, 0, st>>>(params, d.w0_off, d.b0_off, d.w1_off, d.b1_off, d.w2_off,
                                                            d.b2_off, d.fdim, d.nfreq, d.logvar_offset, static_cast<uint16_t*>(packed), zero, zero_n);
  dib_note_launch();
  return cudaGetLastError();
}

cudaError_t dib_enc_fused_forward(const DibEncFusedDesc& d, const DibEncFusedIO& io, cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  WeightMaps m;
  if (!make_all_maps(&m, io.packed, d.F, d.bf16)) return cudaErrorInvalidValue;
  EncFusedParams P;
  fill_params(P, d, io);
  constexpr int smem = kOffFwdEnd1 + 256 + 1024;
  const bool relu = d.act == DIB_ACT_RELU;
  if (d.bf16) return relu ? launch_fused(dib_enc_fused_fwd_kernel<true, true>, smem, d.grid, m, P, st)
                          : launch_fused(dib_enc_fused_fwd_kernel<true, false>, smem, d.grid, m, P, st);
  return relu ? launch_fused(dib_enc_fused_fwd_kernel<false, true>, smem, d.grid, m, P, st)
              : launch_fused(dib_enc_fused_fwd_kernel<false, false>, smem, d.grid, m, P, st);
}

cudaError_t dib_enc_fused_backward(const DibEncFusedDesc& d, const DibEncFusedIO& io, const DibEncFusedBwdIO& b,
                                   cudaStream_t st) {
  if (!tensor_map_encode_fn()) return cudaErrorNotSupported;
  WeightMaps m;
  if (!make_all_maps(&m, io.packed, d.F, d.bf16)) return cudaErrorInvalidValue;
  EncFusedBwdParams Q;
  fill_params(Q.f, d, io);
  Q.f.round_emb = 0;
  Q.d_emb16 = static_cast<const uint16_t*>(b.d_emb16); Q.ldd16 = b.ldd16;
  Q.d_emb = b.d_emb; Q.ldd = b.ldd; Q.beta_dev = b.beta_dev; Q.inv_batch = b.inv_batch; Q.gscale = b.gscale;
  Q.part = b.part; Q.split_stride = b.split_stride;
  Q.w0_off = d.w0_off; Q.b0_off = d.b0_off; Q.w1_off = d.w1_off; Q.w2_off = d.w2_off;
  const bool relu = d.act == DIB_ACT_RELU;
  if (dib_enc_bwd_version() >= 2) {          // two chains on consecutive tiles (default)
    constexpr int smem2 = kV2OffBar + 256 + 1024;
    // this step's forward left the noise and the [pe|1] operand rows in the workspace (16-bit hand-off buffers)
    const bool e16 = Q.f.eps16 != nullptr && Q.f.a0g != nullptr && Q.f.eps == nullptr;
    if (e16 && !make_a0_maps(&m, Q.f.a0g, io.n, d.F, d.bf16)) return cudaErrorInvalidValue;
    // EBW = 8 (eight chain-B warps, half a row per thread, 640 threads) was built and HUNG on the B200 (round 2, run 4): not
    // instantiated.  Measured with EBW = 4 at C0: 0.263 ms.
#define DIB_BWD2(BF, RL)                                                                                                            \
  (e16 ? launch_fused(dib_enc_fused_bwd2_kernel<BF, RL, true, 4>, smem2, d.grid, m, Q, st, 32 * (kV2CtrlEA + 4))                     \
       : launch_fused(dib_enc_fused_bwd2_kernel<BF, RL, false, 4>, smem2, d.grid, m, Q, st, 32 * (kV2CtrlEA + 4)))
    if (d.bf16) return relu ? DIB_BWD2(true, true) : DIB_BWD2(true, false);
    return relu ? DIB_BWD2(false, true) : DIB_BWD2(false, false);
#undef DIB_BWD2
  }
  constexpr int smem = kOffBwdEnd + 256 + 1024;
  if (d.bf16)    // bf16 operands end to end (7-bit mantissa gradients: the usual bf16-training trade, BASELINE config 4)
    return relu ? launch_fused(dib_enc_fused_bwd_kernel<true, true, 8>, smem, d.grid, m, Q, st, 32 * 9)
                : launch_fused(dib_enc_fused_bwd_kernel<true, false, 8>, smem, d.grid, m, Q, st, 32 * 9);
  // 8 epilogue warps.  The 16-warp instantiation (<.., 16>, 32 columns per thread) was measured slower on B200
  // (0.498 vs 0.467 ms at C0): 17 warps cap the kernel at 96 registers and the spills outweigh the extra latency hiding.
  return relu ? launch_fused(dib_enc_fused_bwd_kernel<false, true, 8>, smem, d.grid, m, Q, st, 32 * 9)
              : launch_fused(dib_enc_fused_bwd_kernel<false, false, 8>, smem, d.grid, m, Q, st, 32 * 9);
}
