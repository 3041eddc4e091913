// dib_gemm_tc.cu -- grouped TF32 tensor-core GEMMs (tcgen05.mma, fp32 accumulators in TMEM, TMA-fed shared
// memory, mbarrier pipeline, warp-specialised) with the same fused epilogues and the same problem descriptors
// as the fp32 SIMT path (dib_gemm_simt.cu).  TF32 reads the existing fp32 activation / weight buffers directly:
// TMA brings fp32 tiles into 128B-swizzled shared memory and kind::tf32 consumes the 32-bit containers, so no
// conversion pass and no second copy of the data exist.
//
// Canonical form Out[R x C] = sum_t Aop[R x T] * Bop[T x C]; operand majors per mode
//   FWD    A = h[M x K]   K-major | B = W[K x N]        MN-major      (reduction over fan-in)
//   (K-major tiles: SWIZZLE_128B; MN-major fp32 tiles: SWIZZLE_128B with 32-byte atoms, see dib_sm100.cuh)
//   DGRAD  A = dz[M x N]  K-major | B = W[K x N] as [k][n] K-major    (reduction over fan-out)
//   WGRAD  A = h[m][k]   MN-major | B = dz[m][n]        MN-major      (reduction over a batch slice)
// CTA tile 128 x BN (BN = 64 | 128), K step 32 fp32 (= one 128-byte swizzle span) per pipeline stage.
// Warp roles: 0 TMA producer | 1 TMEM owner + MMA issuer | 2..5 epilogue (TMEM lane quarter = warp_id % 4).
#include <cuda.h>

#include <cstdio>
#include <cstring>

#include "dib_common.cuh"
#include "dib_kernels.h"
#include "dib_sm100.cuh"

namespace {

using namespace sm100;

constexpr int kBM = 128, kBK = 32, kStages = 3;
constexpr int kABytes = kBM * 128;   // 128 rows x 128 B  (K-major)  ==  4 panels x 32 k-rows x 128 B (MN-major)

template <int BN>
struct SmemLayout {
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBarOff = kStages * kStageBytes;          // full[S], empty[S], tmem_full, tmem_ptr
  static constexpr int kTotal = kBarOff + 128 + 1024;            // + alignment slack
};

template <int MODE, int BN>
__global__ void __launch_bounds__(192, 1)
dib_gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                   const DibGemmProblem* __restrict__ probs, const float* __restrict__ baseP, float* __restrict__ baseC,
                   float* baseX, int M, int nsplit, int rows_per_split, long long split_stride, float alpha,
                   int round_out) {
  using L = SmemLayout<BN>;
  constexpr bool A_MN = (MODE == DIB_GEMM_WGRAD), B_MN = (MODE != DIB_GEMM_DGRAD);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + L::kBarOff;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * kStages);
  const uint32_t tmem_ptr_smem = bar_base + 8u * (2 * kStages + 1);
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + L::kBarOff + 8 * (2 * kStages + 1));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int prob, split = 0, r0, c0;
  if constexpr (MODE == DIB_GEMM_WGRAD) {
    prob = blockIdx.z / nsplit; split = blockIdx.z % nsplit;
    c0 = blockIdx.x * BN; r0 = blockIdx.y * kBM;
  } else {
    prob = blockIdx.z; r0 = blockIdx.x * kBM; c0 = blockIdx.y * BN;
  }
  const DibGemmProblem p = probs[prob];
  const int R = (MODE == DIB_GEMM_WGRAD) ? p.R : M;
  const int C = p.C;
  int t_begin = 0, t_end = p.T;
  if constexpr (MODE == DIB_GEMM_WGRAD) {
    t_begin = split * rows_per_split;
    t_end = min(M, t_begin + rows_per_split);
  }
  if (r0 >= R || c0 >= C) return;                       // uniform per CTA
  const int ntiles = t_end > t_begin ? DIB_CEIL_DIV(t_end - t_begin, kBK) : 0;
  const bool do_db = (MODE == DIB_GEMM_WGRAD) && (blockIdx.y == 0) && (p.x_off >= 0);

  // ---------------------------------------------------------------- one-time setup
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), do_db ? 5 : 1);           // MMA commit (+ one arrival per epilogue warp for db)
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, BN);
    tmem_relinquish();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_gen;

  if (warp == 0) {
    // ============================================================== TMA producer
    if (lane == 0) {
      for (int it = 0; it < ntiles; ++it) {
        const int s = it % kStages, ph = (it / kStages) & 1;
        mbar_wait(empty_bar(s), ph ^ 1);
        mbar_expect_tx(full_bar(s), L::kStageBytes);
        const uint32_t a_dst = smem_base + s * L::kStageBytes, b_dst = a_dst + kABytes;
        const int t0 = t_begin + it * kBK;
        if constexpr (A_MN) tma_load_4d(a_dst, &mapA, full_bar(s), 0, t0, r0 / 32, prob);
        else                tma_load_3d(a_dst, &mapA, full_bar(s), t0, r0, prob);
        if constexpr (B_MN) tma_load_4d(b_dst, &mapB, full_bar(s), 0, t0, c0 / 32, prob);
        else                tma_load_3d(b_dst, &mapB, full_bar(s), t0, c0, prob);
      }
    }
  } else if (warp == 1) {
    // ============================================================== MMA issuer (single thread)
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(2u, A_MN ? 1u : 0u, B_MN ? 1u : 0u, BN);
      for (int it = 0; it < ntiles; ++it) {
        const int s = it % kStages, ph = (it / kStages) & 1;
        mbar_wait(full_bar(s), ph);
        tc_fence_after_sync();
        const uint32_t a_addr = smem_base + s * L::kStageBytes, b_addr = a_addr + kABytes;
#pragma unroll
        for (int kk = 0; kk < kBK / 8; ++kk) {          // UMMA K = 8 for tf32 (32 bytes)
          // K-major: advance 32 B inside the 128 B swizzle span; MN-major: advance 8 k-rows (1024 B)
          const uint64_t adesc = A_MN ? umma_smem_desc(a_addr + kk * 1024, kBK * 128, 512, kLayoutSw128Base32)
                                      : umma_smem_desc(a_addr + kk * 32, 16, 1024);
          const uint64_t bdesc = B_MN ? umma_smem_desc(b_addr + kk * 1024, kBK * 128, 512, kLayoutSw128Base32)
                                      : umma_smem_desc(b_addr + kk * 32, 16, 1024);
          umma_tf32(tmem_base, adesc, bdesc, idesc, (it > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(empty_bar(s));                       // frees the stage once these MMAs have read it
      }
      if (ntiles > 0) umma_commit(tmem_full_bar);        // accumulator complete
    }
  } else {
    // ============================================================== epilogue warps (2..5)
    const int q = warp & 3;                              // TMEM lane quarter this warp may access
    const int et = (warp - 2) * 32 + lane;               // 0..127
    if (do_db) {
      // bias gradient: column sums of the dz tiles while they sit in shared memory (MN-major panels)
      float bs = 0.f;
      for (int it = 0; it < ntiles; ++it) {
        const int s = it % kStages, ph = (it / kStages) & 1;
        mbar_wait(full_bar(s), ph);
        if (et < BN) {
          const uint8_t* bt = smem_gen + s * L::kStageBytes + kABytes + (et >> 5) * (kBK * 128);
          const int ch = (et & 31) >> 3, w = et & 7;      // 32-byte chunk inside the 128 B row, word inside the chunk
#pragma unroll 8
          for (int row = 0; row < kBK; ++row)
            bs += *reinterpret_cast<const float*>(bt + row * 128 + ((ch ^ (row & 3)) << 5) + (w << 2));
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar(s));
      }
      if (et < BN && c0 + et < C) (baseX + p.x_off + (long long)split * split_stride)[c0 + et] = bs;
    }
    if (ntiles > 0) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after_sync();
    }
    const int r = r0 + q * 32 + lane;
    float* __restrict__ Out = baseC + p.c_off + (MODE == DIB_GEMM_WGRAD ? (long long)split * split_stride : 0ll);
#pragma unroll 1
    for (int cc = 0; cc < BN; cc += 32) {
      uint32_t v[32];
      if (ntiles > 0) {
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0u;
      }
      if (r < R) {
        const int c = c0 + cc;
        float* dst = Out + (long long)r * p.ldc + c;
        if constexpr (MODE == DIB_GEMM_FWD) {
          const float* bias = baseP + p.x_off + c;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias + j);
            float4 o;
            o.x = dib_maybe_round(dib_act(p.act, __uint_as_float(v[j + 0]) + b4.x, alpha), round_out);
            o.y = dib_maybe_round(dib_act(p.act, __uint_as_float(v[j + 1]) + b4.y, alpha), round_out);
            o.z = dib_maybe_round(dib_act(p.act, __uint_as_float(v[j + 2]) + b4.z, alpha), round_out);
            o.w = dib_maybe_round(dib_act(p.act, __uint_as_float(v[j + 3]) + b4.w, alpha), round_out);
            *reinterpret_cast<float4*>(dst + j) = o;
          }
        } else if constexpr (MODE == DIB_GEMM_DGRAD) {
          const float* xs = baseX + p.x_off + (long long)r * p.ldx + c;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                   __uint_as_float(v[j + 3]));
            if (p.act != DIB_ACT_LINEAR) {
              const float4 x4 = *reinterpret_cast<const float4*>(xs + j);
              o.x *= dib_act_grad(p.act, x4.x, alpha); o.y *= dib_act_grad(p.act, x4.y, alpha);
              o.z *= dib_act_grad(p.act, x4.z, alpha); o.w *= dib_act_grad(p.act, x4.w, alpha);
            }
            o.x = dib_maybe_round(o.x, round_out); o.y = dib_maybe_round(o.y, round_out);
            o.z = dib_maybe_round(o.z, round_out); o.w = dib_maybe_round(o.w, round_out);
            *reinterpret_cast<float4*>(dst + j) = o;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                              __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
    }
  }
  // ---------------------------------------------------------------- teardown
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, BN);
  }
}

// ------------------------------------------------------------------------------------------------ host side

// K-major operand: matrix [rows x ld] fp32, feature stride fs floats -> 3D map (col, row, feature), box 32 x brows x 1
bool make_map_kmajor(CUtensorMap* m, const float* base, long long cols, long long rows, long long ld, long long fs,
                     int nfeat, int box_rows) {
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)nfeat};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(nfeat > 1 ? fs : ld * rows) * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return tensor_map_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// MN-major operand: matrix [krows x ld] fp32 whose contiguous dimension is M/N -> 4D map
// (32 floats, k-row, 32-float panel, feature), box 32 x 32 x npanels x 1  => shared memory [panel][k-row][128 B]
// Swizzle: 128B span with 32B atoms (the only MN-major layout tcgen05 accepts for 32-bit operands).
bool make_map_mnmajor(CUtensorMap* m, const float* base, long long cols, long long krows, long long ld, long long fs,
                      int nfeat, int npanels) {
  cuuint64_t dims[4] = {32, (cuuint64_t)krows, (cuuint64_t)(cols / 32), (cuuint64_t)nfeat};
  cuuint64_t strides[3] = {(cuuint64_t)ld * 4, 128, (cuuint64_t)(nfeat > 1 ? fs : ld * krows) * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)kBK, (cuuint32_t)npanels, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  return tensor_map_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int MODE, int BN>
cudaError_t launch_tc(const DibGemmLaunch& L, const CUtensorMap& mapA, const CUtensorMap& mapB, cudaStream_t st) {
  using SL = SmemLayout<BN>;
  static bool attr_set = false;
  auto kern = dib_gemm_tc_kernel<MODE, BN>;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SL::kTotal);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  dim3 grid;
  if (MODE == DIB_GEMM_WGRAD)
    grid = dim3(DIB_CEIL_DIV(L.maxC, BN), DIB_CEIL_DIV(L.maxR, kBM), L.nprob * L.nsplit);
  else
    grid = dim3(DIB_CEIL_DIV(L.M, kBM), DIB_CEIL_DIV(L.maxC, BN), L.nprob);
  if (grid.x == 0 || grid.y == 0 || grid.z == 0) return cudaSuccess;
  kern<<<grid, 192, SL::kTotal, st>>>(mapA, mapB, L.probs, L.baseBias ? L.baseBias : L.baseB, L.baseC, L.baseX, L.M,
                                      L.nsplit, L.rows_per_split, L.split_stride, L.alpha, L.round_out);
  dib_note_launch();
  return cudaGetLastError();
}

}  // namespace

// Can this group of problems (host copies) run on the tensor-core kernel?  See the operand-major table above.
bool dib_gemm_tc_eligible(int mode, const DibGemmProblem* hp, int nprob, const float* params_base_hint) {
  (void)params_base_hint;
  if (!tensor_map_encode_fn() || nprob < 1) return false;
  const DibGemmProblem& p0 = hp[0];
  const long long sa = nprob > 1 ? hp[1].a_off - hp[0].a_off : 0, sb = nprob > 1 ? hp[1].b_off - hp[0].b_off : 0;
  for (int i = 0; i < nprob; ++i) {
    const DibGemmProblem& p = hp[i];
    if (p.T != p0.T || p.C != p0.C || p.R != p0.R || p.lda != p0.lda || p.ldb != p0.ldb || p.ldc != p0.ldc) return false;
    if (p.a_off != p0.a_off + i * sa || p.b_off != p0.b_off + i * sb) return false;
    if ((p.a_off & 3) || (p.b_off & 3) || (p.c_off & 3) || (p.x_off & 3)) return false;
  }
  if ((sa & 3) || (sb & 3) || sa < 0 || sb < 0) return false;
  if (p0.C % 64) return false;
  if (p0.lda < 32 || p0.ldb < 32 || (p0.ldc & 3)) return false;
  switch (mode) {
    case DIB_GEMM_FWD:   return p0.T >= 32 && (p0.ldb % 32) == 0;               // W panels of 32 along N
    case DIB_GEMM_DGRAD: return p0.T >= 32 && (p0.ldb % 4) == 0 && (p0.ldx % 4) == 0;
    case DIB_GEMM_WGRAD: return (p0.lda % 32) == 0 && (p0.ldb % 32) == 0 && (p0.ldc % 4) == 0;
  }
  return false;
}

cudaError_t dib_launch_gemm_tc(int mode, const DibGemmLaunch& L, const DibGemmProblem* hp, cudaStream_t st) {
  const DibGemmProblem& p0 = hp[0];
  const int nf = L.nprob;
  const long long sa = nf > 1 ? hp[1].a_off - hp[0].a_off : 0, sb = nf > 1 ? hp[1].b_off - hp[0].b_off : 0;
  const int BN = (p0.C % 128 == 0) ? 128 : 64;
  CUtensorMap mapA, mapB;
  bool ok = true;
  const float* A = L.baseA + p0.a_off;
  const float* B = L.baseB + p0.b_off;
  switch (mode) {
    case DIB_GEMM_FWD:    // A: h [M x lda] K-major; B: W [T x C] MN-major
      ok = make_map_kmajor(&mapA, A, p0.lda, L.M, p0.lda, sa, nf, kBM) &&
           make_map_mnmajor(&mapB, B, p0.ldb, p0.T, p0.ldb, sb, nf, BN / 32);
      break;
    case DIB_GEMM_DGRAD:  // A: dz [M x lda] K-major; B: W [C rows x T] K-major
      ok = make_map_kmajor(&mapA, A, p0.lda, L.M, p0.lda, sa, nf, kBM) &&
           make_map_kmajor(&mapB, B, p0.ldb, p0.C, p0.ldb, sb, nf, BN);
      break;
    default:              // A: h [m x lda] MN-major; B: dz [m x ldb] MN-major
      ok = make_map_mnmajor(&mapA, A, p0.lda, L.M, p0.lda, sa, nf, kBM / 32) &&
           make_map_mnmajor(&mapB, B, p0.ldb, L.M, p0.ldb, sb, nf, BN / 32);
      break;
  }
  if (!ok) return cudaErrorInvalidValue;
#define DIB_TC_CASE(MODE)                                                           \
  case MODE:                                                                        \
    return BN == 128 ? launch_tc<MODE, 128>(L, mapA, mapB, st) : launch_tc<MODE, 64>(L, mapA, mapB, st);
  switch (mode) {
    DIB_TC_CASE(DIB_GEMM_FWD)
    DIB_TC_CASE(DIB_GEMM_DGRAD)
    DIB_TC_CASE(DIB_GEMM_WGRAD)
  }
#undef DIB_TC_CASE
  return cudaErrorInvalidValue;
}
