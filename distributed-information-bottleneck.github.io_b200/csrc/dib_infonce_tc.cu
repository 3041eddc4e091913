// dib_infonce_tc.cu -- the streaming InfoNCE head on tcgen05 (sm_100a) for the similarities that have a Gram form:
//   l2sq   s_ij = -max(|a_i|^2 + |b_j|^2 - 2 G_ij, 0) / T
//   l2     s_ij = -sqrt(max(|a_i|^2 + |b_j|^2 - 2 G_ij, 0) + 1e-9) / T        (the reference's own expansion, utils.py:85-90)
//   cosine s_ij = G_ij(a_hat, b_hat) / T
// with G = A B^T.  Same loss and gradients as dib_infonce.cu, but the [n, n] similarity matrix never reaches HBM:
// scratch is O(n d) and the head runs at any batch a B200 holds (dib_infonce.cu stops at n = 32768, 4 GB of S).
//
// Operands.  A prep kernel writes every row of e1 and e2 (normalised for cosine) as bf16 hi + lo halves, x = hi + lo
// to ~2^-17 relative, into [4][n_pad][d_pad] (side, part); every product below is hi*hi + hi*lo + lo*hi on kind::f16
// with fp32 accumulation in TMEM.  A single 16-bit or TF32 Gram matrix has an error of ~2^-11 |a||b| per entry, far too
// much for exp(s) once |a|^2 / T is large.  The diagonal s_ii -- the positive pairs, where the Gram expansion cancels
// catastrophically once training pulls the pairs together -- is computed exactly in fp32 from the rows themselves and
// substituted for the Gram value, and its gradient term is added in fp32 as well.
//
// Sweeps.  A CTA owns 128 rows of one side (blockIdx.y: 0 = rows of e1, 1 = rows of e2, i.e. columns of S) and walks
// every 64-row tile of the other side: TMA loads the tile, one thread issues the Gram MMAs into TMEM, and each of the
// 128 threads reads back its own row of the tile (tcgen05.ld 32x32b: thread = TMEM lane = owned row).  So a row's
// reductions are sequential in one thread, in a fixed order, with no atomics: two identical calls are bit-identical.
//   pass 1 (dib_infonce_tc_lse_kernel):  log-sum-exp of the owned row / column with a running maximum (rescaled per
//          32-column chunk, so the largest term of each chunk contributes exp(0) and no sum can underflow).
//   pass 2 (dib_infonce_tc_grad_kernel): dS_ij = (exp(s_ij - r_i) + exp(s_ij - c_j) - 2 delta_ij) / n, a per-kind
//          weight w_ij goes to shared memory as a bf16 hi/lo K-major operand, and a second MMA accumulates
//          sum_j w_ij y_j in TMEM (the other side's tile serves as its MN-major B operand: for 16-bit types the
//          128B-swizzled [rows][64-element panel] layout is both).  Then per owned row
//            d x_i = scale_i (sum_{j!=i} w_ij y_j - corr_i x_i + w_ii (y_i - c_ii x_i))
//          l2sq: w = dS, corr = sum w, scale = 2/T | l2: w = dS/q (q = -sT), corr = sum w, scale = 1/T
//          cosine (x, y normalised): w = dS, corr = sum dS cos, c_ii = cos_ii, scale = 1/(T |x_i|).
//          l2 pairs closer than kNearPair (e.g. duplicate rows) are treated like the diagonal: s_ij and their term
//          w_ij (y_j - x_i) come from the fp32 rows, because 1/q would amplify the Gram and product errors.
// Each pass is one launch over both sides; together with the prep and loss kernels a head is 4 launches.
#include <cuda.h>
#include <cuda_bf16.h>

#include "dib_common.cuh"
#include "dib_kernels.h"
#include "dib_sm100.cuh"

namespace {

using namespace sm100;

enum { SIM_L2SQ = 0, SIM_L2 = 1, SIM_COS = 4 };
constexpr float kL2Eps = 1e-9f;      // utils.py:150
constexpr int kBM = 128;             // owned rows per CTA = UMMA M = threads
constexpr int kBN = 64;              // other-side rows per tile = Gram N = gradient-product K
constexpr int kThreads = 128;
constexpr int kPrepRows = 8;         // rows per prep block (one warp each)
// l2 pairs with |x - y|^2 below this share of |x|^2 + |y|^2 are recomputed from the fp32 rows: there the Gram expansion
// (error ~2^-16 (|x|^2 + |y|^2)) loses q = |x - y|, and the weight dS / q amplifies the cancellation in the product
constexpr float kNearPair = 1.f / 64.f;

__host__ __device__ constexpr int part_own(int dp) { return kBM * dp * 2; }    // bytes of one bf16 half of the owned tile
__host__ __device__ constexpr int part_oth(int dp) { return kBN * dp * 2; }
constexpr int kWPart = kBM * kBN * 2;                                            // one half of the weight tile
__host__ __device__ constexpr int bar_off(int dp) { return 2 * part_own(dp) + 2 * part_oth(dp) + 2 * kWPart; }
__host__ __device__ constexpr int smem_bytes(int dp) { return bar_off(dp) + 64 + 1024; }
__host__ __device__ constexpr uint32_t tmem_cols(int dp) { return kBN + dp <= 128 ? 128u : (kBN + dp <= 256 ? 256u : 512u); }

// one warp per row of [e1; e2] (padded to n_pad each): squared norm, bf16 hi/lo operand rows, exact diagonal s_ii
template <int KIND>
__global__ void __launch_bounds__(32 * kPrepRows)
dib_infonce_tc_prep_kernel(const float* __restrict__ e1, const float* __restrict__ e2, int n, int n_pad, int d, int dp,
                           float inv_t, __nv_bfloat16* __restrict__ P, float* __restrict__ nrm2, float* __restrict__ diag) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ra = blockIdx.x * kPrepRows + warp;
  if (ra >= 2 * n_pad) return;
  const int side = ra / n_pad, r = ra % n_pad;
  const float* e = (side ? e2 : e1) + (long long)r * d;
  const bool valid = r < n;
  float x2 = 0.f;
  if (valid)
    for (int k = lane; k < d; k += 32) x2 = fmaf(e[k], e[k], x2);
  x2 = dib_warp_sum(x2);
  const float sc = (KIND == SIM_COS && valid) ? 1.f / sqrtf(x2) : 1.f;
  __nv_bfloat16* hi = P + ((long long)(2 * side) * n_pad + r) * dp;
  __nv_bfloat16* lo = P + ((long long)(2 * side + 1) * n_pad + r) * dp;
  for (int k = lane; k < dp; k += 32) {
    const float v = (valid && k < d) ? e[k] * sc : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[k] = h;
    lo[k] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
  if (lane == 0) nrm2[ra] = x2;
  if (side == 0 && valid) {
    const float* b = e2 + (long long)r * d;
    float q = 0.f, nb = 0.f;
    for (int k = lane; k < d; k += 32) {
      if (KIND == SIM_COS) { q = fmaf(e[k], b[k], q); nb = fmaf(b[k], b[k], nb); }
      else { const float df = e[k] - b[k]; q = fmaf(df, df, q); }
    }
    q = dib_warp_sum(q);
    if (KIND == SIM_COS) nb = dib_warp_sum(nb);
    if (lane == 0) {
      const float s = KIND == SIM_L2SQ ? -q : (KIND == SIM_L2 ? -sqrtf(q + kL2Eps) : q / (sqrtf(x2) * sqrtf(nb)));
      diag[r] = s * inv_t;
    }
  }
}

__device__ __noinline__ float row_d2(const float* __restrict__ x, const float* __restrict__ y, int d) {
  float s = 0.f;
  for (int k = 0; k < d; ++k) { const float df = x[k] - y[k]; s = fmaf(df, df, s); }
  return s;
}
// out[k] += w (y[k] - x[k]): a near pair's gradient term in fp32, into the thread's own output row
__device__ __noinline__ void row_add_diff(float* __restrict__ out, float w, const float* __restrict__ y,
                                          const float* __restrict__ x, int d) {
  for (int k = 0; k < d; ++k) out[k] = fmaf(w, y[k] - x[k], out[k]);
}

// s_ij from the Gram entry g; q (l2 only) = sqrt(d2 + eps) = -s T.  `near` (l2 only): the pair is closer than kNearPair
// allows, and s / q were recomputed from the fp32 rows x, y.
template <int KIND>
__device__ __forceinline__ float gram_sim(float g, float nx2, float ny2, float inv_t, float& q, bool& near, const float* x,
                                          const float* y, int d) {
  if (KIND == SIM_COS) return g * inv_t;
  float d2 = fmaxf(nx2 + ny2 - 2.f * g, 0.f);
  if (KIND == SIM_L2SQ) return -d2 * inv_t;
  near = d2 < kNearPair * (nx2 + ny2);
  if (near) d2 = row_d2(x, y, d);
  q = sqrtf(d2 + kL2Eps);
  return -q * inv_t;
}

struct Sweep {
  uint32_t s_own, s_oth, s_w, bar_own, bar_oth, bar_g, bar_w, tslot;
  uint8_t* gen;   // generic pointer to s_own
};

__device__ __forceinline__ Sweep sweep_layout(uint8_t* smem_raw, int dp) {
  Sweep S;
  S.s_own = (smem_u32(smem_raw) + 1023u) & ~1023u;
  S.gen = smem_raw + (S.s_own - smem_u32(smem_raw));
  S.s_oth = S.s_own + 2 * part_own(dp);
  S.s_w = S.s_oth + 2 * part_oth(dp);
  const uint32_t b = S.s_own + bar_off(dp);
  S.bar_own = b; S.bar_oth = b + 8; S.bar_g = b + 16; S.bar_w = b + 24; S.tslot = b + 32;
  return S;
}

// the owned 128 rows (both halves, every 64-column panel) as [half][panel][row][128 B]
__device__ __forceinline__ void load_own(const Sweep& S, const CUtensorMap* map, int side, int n_pad, int r0, int dp) {
  mbar_expect_tx(S.bar_own, 2 * part_own(dp));
  for (int p = 0; p < 2; ++p)
    for (int c = 0; c < dp / 64; ++c)
      for (int h = 0; h < kBM / 64; ++h)
        tma_load_2d(S.s_own + p * part_own(dp) + c * kBM * 128 + h * 64 * 128, map, S.bar_own, c * 64,
                    (2 * side + p) * n_pad + r0 + h * 64);
}
__device__ __forceinline__ void load_other(const Sweep& S, const CUtensorMap* map, int oside, int n_pad, int j0, int dp) {
  mbar_expect_tx(S.bar_oth, 2 * part_oth(dp));
  for (int p = 0; p < 2; ++p)
    for (int c = 0; c < dp / 64; ++c)
      tma_load_2d(S.s_oth + p * part_oth(dp) + c * kBN * 128, map, S.bar_oth, c * 64, (2 * oside + p) * n_pad + j0);
}

// G[128 x 64] = X Y^T, split operands: hi*hi + hi*lo + lo*hi
__device__ __forceinline__ void issue_gram(const Sweep& S, uint32_t tG, int dp) {
  constexpr uint32_t idesc = umma_idesc(1u, 0u, 0u, kBN);
  for (int kk = 0; kk < dp / 16; ++kk) {
    const uint32_t ao = (kk >> 2) * kBM * 128 + (kk & 3) * 32, bo = (kk >> 2) * kBN * 128 + (kk & 3) * 32;
    const uint64_t ah = umma_smem_desc(S.s_own + ao, 16, 1024), al = umma_smem_desc(S.s_own + part_own(dp) + ao, 16, 1024);
    const uint64_t bh = umma_smem_desc(S.s_oth + bo, 16, 1024), bl = umma_smem_desc(S.s_oth + part_oth(dp) + bo, 16, 1024);
    umma_bf16(tG, ah, bh, idesc, kk > 0 ? 1u : 0u);
    umma_bf16(tG, ah, bl, idesc, 1u);
    umma_bf16(tG, al, bh, idesc, 1u);
  }
}

// Acc[128 x dp] += W[128 x 64] Y[64 x dp]: W K-major, the other tile read MN-major (rows = K, panels along N)
__device__ __forceinline__ void issue_wy(const Sweep& S, uint32_t tAcc, int dp, bool first) {
  const uint32_t idesc = umma_idesc(1u, 0u, 1u, (uint32_t)dp);
  for (int kk = 0; kk < kBN / 16; ++kk) {
    const uint64_t wh = umma_smem_desc(S.s_w + kk * 32, 16, 1024), wl = umma_smem_desc(S.s_w + kWPart + kk * 32, 16, 1024);
    const uint64_t yh = umma_smem_desc(S.s_oth + kk * 2048, kBN * 128, 1024),
                   yl = umma_smem_desc(S.s_oth + part_oth(dp) + kk * 2048, kBN * 128, 1024);
    umma_bf16(tAcc, wh, yh, idesc, (first && kk == 0) ? 0u : 1u);
    umma_bf16(tAcc, wl, yh, idesc, 1u);
    umma_bf16(tAcc, wh, yl, idesc, 1u);
  }
}

__device__ __forceinline__ uint32_t sweep_setup(const Sweep& S, const CUtensorMap* map, int dp) {
  const int tid = threadIdx.x;
  if (tid == 0) {
    tma_prefetch_desc(map);
    mbar_init(S.bar_own, 1); mbar_init(S.bar_oth, 1); mbar_init(S.bar_g, 1); mbar_init(S.bar_w, 1);
    fence_barrier_init();
  }
  if (tid < 32) { tmem_alloc(S.tslot, tmem_cols(dp)); tmem_relinquish(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  return *reinterpret_cast<volatile uint32_t*>(S.gen + bar_off(dp) + 32);
}

__device__ __forceinline__ void sweep_teardown(uint32_t tmem, int dp) {
  tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x < 32) { tc_fence_after_sync(); tmem_dealloc(tmem, tmem_cols(dp)); }
}

// tile t's Gram product, then wait for it (every thread); thread 0 also drives the loads
__device__ __forceinline__ void gram_step(const Sweep& S, const CUtensorMap* map, uint32_t tG, int t, int dp) {
  if (threadIdx.x == 0) {
    if (t == 0) mbar_wait(S.bar_own, 0);
    mbar_wait(S.bar_oth, t & 1);
    tc_fence_after_sync();
    issue_gram(S, tG, dp);
    umma_commit(S.bar_g);
  }
  __syncwarp();
  mbar_wait(S.bar_g, t & 1);
  tc_fence_after_sync();
}

// pass 1: lse[side * n_pad + i] = log sum_j exp s(own_i, other_j)
template <int KIND>
__global__ void __launch_bounds__(kThreads)
dib_infonce_tc_lse_kernel(const __grid_constant__ CUtensorMap map, int n, int n_pad, int d, int dp, float inv_t,
                          const float* __restrict__ e1, const float* __restrict__ e2, const float* __restrict__ nrm2,
                          const float* __restrict__ diag, float* __restrict__ lse) {
  extern __shared__ uint8_t smem_raw[];
  const Sweep S = sweep_layout(smem_raw, dp);
  const int side = blockIdx.y, oside = 1 - side, tid = threadIdx.x, r0 = blockIdx.x * kBM, i = r0 + tid;
  const uint32_t tmem = sweep_setup(S, &map, dp), lane_off = (uint32_t)((tid >> 5) * 32) << 16;
  const float nx2 = nrm2[side * n_pad + i], s_diag = i < n ? diag[i] : 0.f;
  const float* ny2 = nrm2 + oside * n_pad;
  const float* xe = (side ? e2 : e1) + (long long)i * d;
  const float* ye = side ? e1 : e2;
  const int ntiles = DIB_CEIL_DIV(n, kBN);
  if (tid == 0) { load_own(S, &map, side, n_pad, r0, dp); load_other(S, &map, oside, n_pad, 0, dp); }
  float run_m = -INFINITY, run_s = 0.f;
  for (int t = 0; t < ntiles; ++t) {
    const int j0 = t * kBN;
    gram_step(S, &map, tmem, t, dp);
    if (tid == 0 && t + 1 < ntiles) load_other(S, &map, oside, n_pad, j0 + kBN, dp);   // the Gram MMAs have read the tile
#pragma unroll 1
    for (int h = 0; h < kBN / 32; ++h) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(tmem + lane_off + h * 32, v);
      tmem_ld_wait();
      float s[32], cm = -INFINITY;
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) {
        const int j = j0 + h * 32 + jj;
        float q;
        bool near;
        s[jj] = j < n ? (j == i ? s_diag
                                : gram_sim<KIND>(__uint_as_float(v[jj]), nx2, ny2[j], inv_t, q, near, xe, ye + (long long)j * d, d))
                      : -INFINITY;
        cm = fmaxf(cm, s[jj]);
      }
      if (cm > run_m) { run_s *= __expf(run_m - cm); run_m = cm; }
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) run_s += __expf(s[jj] - run_m);
    }
    tc_fence_before_sync();
    __syncthreads();            // every row has read G before the next tile's MMAs overwrite it
    tc_fence_after_sync();
  }
  if (i < n) lse[side * n_pad + i] = run_m + logf(run_s);
  sweep_teardown(tmem, dp);
}

// pass 2: d loss / d (owned rows)
template <int KIND>
__global__ void __launch_bounds__(kThreads)
dib_infonce_tc_grad_kernel(const __grid_constant__ CUtensorMap map, int n, int n_pad, int d, int dp, float inv_t,
                           const float* __restrict__ e1, const float* __restrict__ e2, const float* __restrict__ nrm2,
                           const float* __restrict__ diag, const float* __restrict__ lse, float* __restrict__ d_e1,
                           float* __restrict__ d_e2) {
  const int side = blockIdx.y, oside = 1 - side;
  float* __restrict__ d_own = side ? d_e2 : d_e1;
  if (!d_own) return;
  extern __shared__ uint8_t smem_raw[];
  const Sweep S = sweep_layout(smem_raw, dp);
  uint8_t* w_gen = S.gen + (S.s_w - S.s_own);
  const int tid = threadIdx.x, r0 = blockIdx.x * kBM, i = r0 + tid;
  const bool valid_i = i < n;
  const uint32_t tmem = sweep_setup(S, &map, dp), lane_off = (uint32_t)((tid >> 5) * 32) << 16;
  const uint32_t tG = tmem, tAcc = tmem + kBN;
  const float nx2 = nrm2[side * n_pad + i], s_diag = valid_i ? diag[i] : 0.f;
  const float lse_own = valid_i ? lse[side * n_pad + i] : 0.f, inv_n = 1.f / (float)n, temp = 1.f / inv_t;
  const float* ny2 = nrm2 + oside * n_pad;
  const float* lse_oth = lse + oside * n_pad;
  const float* xe = (side ? e2 : e1) + (long long)i * d;
  const float* ye_all = side ? e1 : e2;
  float* out_i = d_own + (long long)i * d;
  const int ntiles = DIB_CEIL_DIV(n, kBN);
  if (KIND == SIM_L2 && valid_i)
    for (int k = 0; k < d; ++k) out_i[k] = 0.f;   // accumulates the near pairs' terms until the epilogue
  if (tid == 0) { load_own(S, &map, side, n_pad, r0, dp); load_other(S, &map, oside, n_pad, 0, dp); }
  float corr = 0.f, w_diag = 0.f, c_diag = 1.f;
  for (int t = 0; t < ntiles; ++t) {
    const int j0 = t * kBN;
    gram_step(S, &map, tG, t, dp);     // also: the previous tile's W Y product has retired (thread 0 waited for it)
#pragma unroll 1
    for (int h = 0; h < kBN / 32; ++h) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(tG + lane_off + h * 32, v);
      tmem_ld_wait();
      float w[32];
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) {
        const int j = j0 + h * 32 + jj;
        w[jj] = 0.f;
        if (valid_i && j < n) {
          const float g = __uint_as_float(v[jj]);
          const bool dg = j == i;
          float q = 1.f, s;
          bool near = false;
          if (dg) { s = s_diag; q = -s_diag * temp; }
          else s = gram_sim<KIND>(g, nx2, ny2[j], inv_t, q, near, xe, ye_all + (long long)j * d, d);
          const float ds = (__expf(s - lse_own) + __expf(s - lse_oth[j]) - (dg ? 2.f : 0.f)) * inv_n;
          const float wv = KIND == SIM_L2 ? ds / q : ds;
          if (dg) { w_diag = wv; c_diag = KIND == SIM_COS ? s_diag * temp : 1.f; }
          else if (KIND == SIM_L2 && near) row_add_diff(out_i, wv, ye_all + (long long)j * d, xe, d);
          else { w[jj] = wv; corr += KIND == SIM_COS ? ds * g : wv; }
        }
      }
      // row tid of the K-major weight operand: 16-byte chunk c of the 128-byte row at (c ^ row % 8)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float a = w[c * 8 + 2 * u], b = w[c * 8 + 2 * u + 1];
          const __nv_bfloat162 hp = __floats2bfloat162_rn(a, b);
          const __nv_bfloat162 lp = __floats2bfloat162_rn(a - __low2float(hp), b - __high2float(hp));
          hw[u] = *reinterpret_cast<const uint32_t*>(&hp);
          lw[u] = *reinterpret_cast<const uint32_t*>(&lp);
        }
        const int off = tid * 128 + (((h * 4 + c) ^ (tid & 7)) << 4);
        *reinterpret_cast<uint4*>(w_gen + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(w_gen + kWPart + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    if (tid == 0) {
      issue_wy(S, tAcc, dp, t == 0);
      umma_commit(S.bar_w);
      mbar_wait(S.bar_w, t & 1);       // W and the other tile are free again
      if (t + 1 < ntiles) load_other(S, &map, oside, n_pad, j0 + kBN, dp);
    }
  }
  tc_fence_before_sync();
  __syncthreads();                     // thread 0 has seen the last W Y product retire
  tc_fence_after_sync();
  const float* ye = ye_all + (long long)i * d;
  float inv_nx = 1.f, inv_ny = 1.f, scale = (KIND == SIM_L2SQ ? 2.f : 1.f) * inv_t;
  if (KIND == SIM_COS && valid_i) { inv_nx = 1.f / sqrtf(nx2); inv_ny = 1.f / sqrtf(ny2[i]); scale = inv_t * inv_nx; }
#pragma unroll 1
  for (int c0 = 0; c0 < dp; c0 += 32) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(tAcc + lane_off + c0, v);
    tmem_ld_wait();
    if (valid_i) {
#pragma unroll
      for (int jj = 0; jj < 32; ++jj) {
        const int k = c0 + jj;
        if (k < d) {
          const float x = xe[k] * inv_nx, y = ye[k] * inv_ny;
          const float near_terms = KIND == SIM_L2 ? out_i[k] : 0.f;
          out_i[k] = scale * (__uint_as_float(v[jj]) - corr * x + w_diag * (y - c_diag * x) + near_terms);
        }
      }
    }
  }
  sweep_teardown(tmem, dp);
}

// loss = (1/n) sum_i (r_i + c_i - 2 s_ii), fixed-order reduction in one block
__global__ void __launch_bounds__(256)
dib_infonce_tc_loss_kernel(const float* __restrict__ lse, const float* __restrict__ diag, int n, int n_pad,
                           float* __restrict__ out_loss) {
  __shared__ float red[8];
  float v = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) v += lse[i] + lse[n_pad + i] - 2.f * diag[i];
  v = dib_warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    out_loss[0] = t / (float)n;
  }
}


struct TcGeom {
  int n_pad, dp;
  size_t p_bytes;
};
TcGeom geom(int64_t n, int d) {
  TcGeom g;
  g.n_pad = (int)DIB_ROUND_UP(n, (int64_t)kBM);
  g.dp = DIB_ROUND_UP(d, 64);
  g.p_bytes = (size_t)4 * g.n_pad * g.dp * sizeof(__nv_bfloat16);
  return g;
}

template <int KIND>
cudaError_t launch_kind(const float* e1, const float* e2, int n, int d, float temperature, void* scratch, float* out_loss,
                        float* d_e1, float* d_e2, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(dib_infonce_tc_lse_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         smem_bytes(256));
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(dib_infonce_tc_grad_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(256));
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  const TcGeom g = geom(n, d);
  __nv_bfloat16* P = static_cast<__nv_bfloat16*>(scratch);
  float* nrm2 = reinterpret_cast<float*>(static_cast<uint8_t*>(scratch) + g.p_bytes);
  float* lse = nrm2 + 2 * (size_t)g.n_pad;
  float* diag = lse + 2 * (size_t)g.n_pad;
  const float inv_t = 1.f / temperature;
  CUtensorMap map;
  {
    // [4 * n_pad rows][dp] bf16 (side, half, row), box 64 columns (one 128-byte swizzle span) x 64 rows
    cuuint64_t dims[2] = {(cuuint64_t)g.dp, (cuuint64_t)4 * g.n_pad};
    cuuint64_t strides[1] = {(cuuint64_t)g.dp * 2};
    cuuint32_t box[2] = {64, 64}, es[2] = {1, 1};
    if (tensor_map_encode_fn()(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, P, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) !=
        CUDA_SUCCESS)
      return cudaErrorInvalidValue;
  }
  dib_infonce_tc_prep_kernel<KIND><<<DIB_CEIL_DIV(2 * g.n_pad, kPrepRows), 32 * kPrepRows, 0, st>>>(
      e1, e2, n, g.n_pad, d, g.dp, inv_t, P, nrm2, diag);
  const dim3 grid(g.n_pad / kBM, 2);
  dib_infonce_tc_lse_kernel<KIND><<<grid, kThreads, smem_bytes(g.dp), st>>>(map, n, g.n_pad, d, g.dp, inv_t, e1, e2, nrm2,
                                                                             diag, lse);
  dib_infonce_tc_loss_kernel<<<1, 256, 0, st>>>(lse, diag, n, g.n_pad, out_loss);
  dib_note_launch(3);
  if (d_e1 || d_e2) {
    dib_infonce_tc_grad_kernel<KIND><<<grid, kThreads, smem_bytes(g.dp), st>>>(map, n, g.n_pad, d, g.dp, inv_t, e1, e2,
                                                                                nrm2, diag, lse, d_e1, d_e2);
    dib_note_launch();
  }
  return cudaGetLastError();
}

}  // namespace

size_t dib_infonce_head_tc_scratch(int64_t n, int d) {
  const TcGeom g = geom(n, d);
  return g.p_bytes + sizeof(float) * 5 * (size_t)g.n_pad;
}

bool dib_infonce_head_tc_available() { return tensor_map_encode_fn() != nullptr; }

// scratch: [4][n_pad][d_pad] bf16 operands | 2 n_pad squared norms | 2 n_pad log-sum-exps | n_pad diagonal s_ii
cudaError_t dib_launch_infonce_head_tc(int kind, const float* e1, const float* e2, int64_t n, int d, float temperature,
                                       void* scratch, float* out_loss, float* d_e1, float* d_e2, cudaStream_t st) {
  switch (kind) {
    case SIM_L2SQ: return launch_kind<SIM_L2SQ>(e1, e2, (int)n, d, temperature, scratch, out_loss, d_e1, d_e2, st);
    case SIM_L2: return launch_kind<SIM_L2>(e1, e2, (int)n, d, temperature, scratch, out_loss, d_e1, d_e2, st);
    case SIM_COS: return launch_kind<SIM_COS>(e1, e2, (int)n, d, temperature, scratch, out_loss, d_e1, d_e2, st);
  }
  return cudaErrorInvalidValue;
}
