// dib_infonce_train.cu -- the small kernels of the InfoNCE train step (dib_infonce_train_step) that the grouped GEMMs,
// the heads and the elementwise kernels do not already provide:
//   * the output encoder's weight pack: its Keras-ordered variables (params[P, P+Q), arbitrary offsets) copied into a
//     shadow whose every variable starts on a 16-byte boundary (the GEMM kernels' TMA operands need that), kernels
//     rounded to the TF32 grid in the tensor-core modes -- one launch for all variables;
//   * the InfoNCE entry of the statistics vector: stats[F] = n * L from the head's device scalar L;
//   * the hand-off of d e2 from the head to the output encoder's backward GEMMs: rows re-strided to the workspace
//     leading dimension, pad columns zeroed, and TF32-rounded in the tensor-core modes -- the same convention as d e1,
//     which the loss kernel rounds on its way into the model's backward.
#include "dib_common.cuh"
#include "dib_kernels.h"

namespace {

__global__ void dib_oe_pack_kernel(const float* __restrict__ src, float* __restrict__ dst, DibOePackTable t) {
  const int v = blockIdx.y;
  const long long cnt = t.count[v];
  const float* s = src + t.src_off[v];
  float* d = dst + t.dst_off[v];
  const int rnd = t.round[v];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (long long)gridDim.x * blockDim.x)
    d[i] = dib_maybe_round(s[i], rnd);
}

__global__ void dib_infonce_stats_kernel(const float* __restrict__ loss, long long n, float* __restrict__ stats_loss) {
  if (threadIdx.x == 0) stats_loss[0] = (float)n * loss[0];
}

// dst[r, c] = round(src[r, c]) for c < cols, 0 for cols <= c < ldd.  src may equal dst (lds == ldd): every element is read
// and written by the same thread, so the pointers are deliberately not __restrict__.
__global__ void dib_grad_handoff_kernel(const float* src, int lds, float* dst, int ldd, int cols, long long n, int rnd) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * ldd) return;
  const long long r = idx / ldd;
  const int c = (int)(idx - r * ldd);
  dst[idx] = c < cols ? dib_maybe_round(src[r * lds + c], rnd) : 0.f;
}

}  // namespace

cudaError_t dib_launch_grad_handoff(const float* src, int lds, float* dst, int ldd, int cols, int64_t n, int round_out,
                                    cudaStream_t st) {
  const long long total = (long long)n * ldd;
  if (total <= 0) return cudaSuccess;
  dib_grad_handoff_kernel<<<(unsigned)DIB_CEIL_DIV(total, 256ll), 256, 0, st>>>(src, lds, dst, ldd, cols, n, round_out);
  dib_note_launch();
  return cudaGetLastError();
}

cudaError_t dib_launch_oe_pack(const float* src, float* dst, const DibOePackTable& t, cudaStream_t st) {
  if (t.nvar < 1) return cudaSuccess;
  long long mx = 1;
  for (int v = 0; v < t.nvar; ++v) mx = t.count[v] > mx ? t.count[v] : mx;
  const int bx = (int)(DIB_CEIL_DIV(mx, 256ll) < 64 ? DIB_CEIL_DIV(mx, 256ll) : 64);
  dib_oe_pack_kernel<<<dim3(bx, t.nvar), 256, 0, st>>>(src, dst, t);
  dib_note_launch();
  return cudaGetLastError();
}

cudaError_t dib_launch_infonce_stats(const float* loss_dev, int64_t n, float* stats_loss, cudaStream_t st) {
  dib_infonce_stats_kernel<<<1, 32, 0, st>>>(loss_dev, n, stats_loss);
  dib_note_launch();
  return cudaGetLastError();
}
