// dib_kernels.h -- internal launcher prototypes shared by the translation units of libdib_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct DibGemmProblem;

// number of kernels launched by this library in this process (bench.py reports it as gpu_launches)
void dib_note_launch(int n = 1);

struct DibGemmLaunch {
  const DibGemmProblem* probs;  // device array, nprob entries
  int nprob;
  const float* baseA;
  const float* baseB;
  float* baseC;
  float* baseX;
  int M;               // batch rows
  int maxC, maxR;      // largest C (and, for WGRAD, R) over the group -> grid size
  int nsplit;          // WGRAD batch splits
  int rows_per_split;
  long long split_stride;
  float alpha;
  int round_out = 0;              // round FWD / DGRAD outputs to the TF32 grid (tensor-core mode operands)
  const float* baseBias = nullptr; // FWD bias base when baseB points at the TF32-rounded weight shadow
};

cudaError_t dib_launch_gemm_simt(int mode, const DibGemmLaunch& L, cudaStream_t st);

// TF32 tcgen05 path (dib_gemm_tc.cu); `hp` = host copies of the group's problem descriptors
bool dib_gemm_tc_eligible(int mode, const DibGemmProblem* hp, int nprob, const float* params_base_hint);
cudaError_t dib_launch_gemm_tc(int mode, const DibGemmLaunch& L, const DibGemmProblem* hp, cudaStream_t st);

// ---- elementwise / reduction kernels (dib_elementwise.cu) -----------------------------------------------
// positional encoding (models.py:22-23) into the padded first-layer operand; tables are per pe column.
cudaError_t dib_launch_pe(const float* x, int ldx, int x_col_shift, const int* col_src, const int* col_freq,
                          int col_begin, int col_end, float* pe, int ldpe, int pe_col_shift, int64_t n,
                          int round_out, cudaStream_t st, const int* row_index = nullptr,
                          const int* col_feat = nullptr, int64_t n_src = 0);

struct DibReparamArgs {
  const float* enc_out;    // [F][feat_stride] rows of ldo floats: (mu[E] | logvar[E] | pad)
  long long feat_stride;
  int ldo;
  const float* eps;        // [n, F, E] or nullptr -> Philox
  uint64_t seed; uint32_t step; uint64_t sample_offset;
  const uint32_t* step_dev = nullptr;   // optional device addend of `step` (CUDA-Graph replay)
  int F, E;
  int64_t n;
  int round_out = 0;
};
// u = mu + exp(logvar/2) eps (models.py:108); per-(block,feature) partial sums of the KL (models.py:111-112).
cudaError_t dib_launch_reparam_fwd(const DibReparamArgs& a, float* emb, int ldemb, float* user_emb,
                                   float* kl_part, int nblk_stride, cudaStream_t st);
// d(mu,logvar) from d(u) and beta * dKL (models.py:118).
cudaError_t dib_launch_reparam_bwd(const DibReparamArgs& a, const float* d_emb, int ldemb, const float* beta_dev,
                                   float inv_batch, float* d_out, cudaStream_t st);

// compiled loss + metrics=['accuracy'] + d(loss)/d(pre-activation output).
cudaError_t dib_launch_loss(int loss, int out_act, float alpha, const float* pred, int ldp, const float* y, int out_dim,
                            int64_t n, float inv_batch, float* d_pred /*nullable*/, float* user_pred /*nullable*/,
                            float* loss_part, float* acc_part, int round_out, cudaStream_t st);

cudaError_t dib_launch_round_copy(const float* src, float* dst, int64_t count, cudaStream_t st);

cudaError_t dib_launch_finalize_stats(const float* kl_part, int nblk_stride, int nblk_kl, const float* loss_part,
                                      const float* acc_part, int nblk_loss, int F, int64_t n, int has_y,
                                      float* out_stats, cudaStream_t st);

cudaError_t dib_launch_reduce_partials(const float* part, long long split_stride, int nsplit, int64_t count,
                                       float* out, cudaStream_t st);

cudaError_t dib_launch_copy2d(const float* src, int lds, float* dst, int ldd, int cols, int64_t n, cudaStream_t st);

cudaError_t dib_launch_optimizer(int kind, float* params, const float* grads, float* s1, float* s2, int64_t count,
                                 const float* lr_dev, int32_t* step_dev, float h0, float h1, float h2, cudaStream_t st);
cudaError_t dib_launch_pe_plain(const float* x, int64_t n, int d, int nfreq, float* out, cudaStream_t st);

cudaError_t dib_launch_adam(float* params, const float* grads, float* m, float* v, int64_t count,
                            const float* lr_dev, int32_t* step_dev, float b1, float b2, float eps, cudaStream_t st);

// mode 0: Bhattacharyya distance, 1: KL(1||2); ml* rows are (mu[E] | logvar[E]) with leading dimension ld*, `groups`
// independent problems gstride* floats apart; outputs [groups, n, m].
cudaError_t dib_launch_pairwise_gauss(int mode, const float* ml1, int64_t ld1, int64_t gstride1, int64_t n,
                                      const float* ml2, int64_t ld2, int64_t gstride2, int64_t m, int E, int groups,
                                      float* out_dist, float* out_comp, cudaStream_t st);

// next row f3 (dib_infonce.cu): kind 0 l2sq | 1 l2 | 2 l1 | 3 linf | 4 cosine
cudaError_t dib_launch_similarity(int kind, const float* e1, int64_t n, const float* e2, int64_t m, int d, float temperature,
                                  float* out, cudaStream_t st);
cudaError_t dib_launch_infonce_head(int kind, const float* e1, const float* e2, int64_t n, int d, float temperature,
                                    float* scratch, float* out_loss, float* d_e1, float* d_e2, cudaStream_t st);
// streaming tcgen05 head (dib_infonce_tc.cu): kinds 0 l2sq | 1 l2 | 4 cosine, d <= 256, scratch O(n d)
size_t dib_infonce_head_tc_scratch(int64_t n, int d);
bool dib_infonce_head_tc_available();
cudaError_t dib_launch_infonce_head_tc(int kind, const float* e1, const float* e2, int64_t n, int d, float temperature,
                                       void* scratch, float* out_loss, float* d_e1, float* d_e2, cudaStream_t st);

// InfoNCE train step (dib_infonce_train.cu): the output encoder's weight pack into its 16-byte-aligned shadow (variable v:
// dst[dst_off[v] + i] = src[src_off[v] + i], TF32-rounded where round[v]), and stats[F] = n * L
constexpr int kDibMaxOeLayers = 16;
struct DibOePackTable {
  int nvar = 0;
  long long src_off[2 * (kDibMaxOeLayers + 1)], dst_off[2 * (kDibMaxOeLayers + 1)], count[2 * (kDibMaxOeLayers + 1)];
  int round[2 * (kDibMaxOeLayers + 1)];
};
cudaError_t dib_launch_oe_pack(const float* src, float* dst, const DibOePackTable& t, cudaStream_t st);
cudaError_t dib_launch_infonce_stats(const float* loss_dev, int64_t n, float* stats_loss, cudaStream_t st);
// d e2 [n, cols] (row stride lds) -> dst rows of ldd floats: TF32-rounded when round_out, pad columns zeroed; src may be dst
cudaError_t dib_launch_grad_handoff(const float* src, int lds, float* dst, int ldd, int cols, int64_t n, int round_out,
                                    cudaStream_t st);

cudaError_t dib_launch_metrics_update(const float* stats, const float* beta_dev, float* acc, int F, float kl_exponent,
                                      float kl_scale, cudaStream_t st);

// ---- custom-step variants (SURVEY 8f3) ----
// enc_out[f][row][E + e] += offset  (nb-particle cell 8: logvar offset), all features or only `feature` (>= 0)
cudaError_t dib_launch_add_logvar_offset(float* enc_out, long long feat_stride, int ldo, int F, int E, int64_t n, float offset,
                                         int feature, cudaStream_t st);
// nb-bool cell 4 SimpleEncoder forward: enc_out[f][row] = (x[row, x_off[f] + e] * mu_scaling_f | logvar_f), e < E
cudaError_t dib_launch_simple_enc_fwd(const float* x, int ldx, const int* x_off_dev, const float* params, float* enc_out,
                                      long long feat_stride, int ldo, int F, int E, int64_t n, int feature, int x_is_feature_only,
                                      const int* row_index, int64_t n_src, cudaStream_t st);
// its weight gradients: part[split][2f] = sum_rows sum_e d_mu * x, part[split][2f+1] = sum_rows sum_e d_logvar
cudaError_t dib_launch_simple_enc_wgrad(const float* x, int ldx, const int* x_off_dev, const float* d_out, long long feat_stride,
                                        int ldo, int F, int E, int64_t n, int nsplit, int rows_per_split, float* part,
                                        long long split_stride, cudaStream_t st);
// Keras Dropout on the encoder activations [F][feat_stride] rows of ld floats, `width` live columns (nb-radial cell 5):
//   backward == 0: dst = src * keep / (1 - rate)   (rate == 0: plain copy -- inference, where Dropout is the identity)
//   backward == 1: dst *= keep / (1 - rate)         (src ignored)
// keep from Philox (seed, step [+ *step_dev], sample_offset + row, feature, layer, column): oracle/philox.py :: dropout_keep
cudaError_t dib_launch_dropout(const float* src, float* dst, long long feat_stride, int ld, int width, int F, int64_t n, float rate,
                               uint64_t seed, uint32_t step, const uint32_t* step_dev, uint64_t sample_offset, int layer,
                               int feature, int backward, int round_out, cudaStream_t st);

// beta_eff = beta * scale * p * (sum_i stats[i] * inv_global_batch)^(p-1)   (d(beta*scale*KL^p)/dKL; p = 1: beta * scale)
cudaError_t dib_launch_beta_eff(const float* stats, int F, float inv_global_batch, const float* beta_dev, float exponent,
                                float scale, float* beta_eff_dev, cudaStream_t st);

// ---- fused per-feature encoder kernels (dib_enc_fused.cu): x -> emb / KL without touching HBM in between ----
struct DibEncFusedDesc {        // static per model; all pointers are DEVICE arrays of length F
  int F = 0, nfreq = 1, act = 0, bf16 = 0, grid = 0;
  float alpha = 0.2f;
  float logvar_offset = 0.f;      // folded into the logvar half of the b2 bias carrier when the weights are packed
  const int* x_off = nullptr; const int* fdim = nullptr;
  const long long* w0_off = nullptr; const long long* b0_off = nullptr; const long long* w1_off = nullptr;
  const long long* b1_off = nullptr; const long long* w2_off = nullptr; const long long* b2_off = nullptr;
};
struct DibEncFusedIO {
  const float* params; const void* packed;      // fp32 masters, packed 16-bit weights (dib_enc_fused_pack)
  const float* x; int ldx; int64_t n;
  const float* eps; uint64_t seed; uint32_t step; uint64_t sample_offset;
  const uint32_t* step_dev = nullptr;       // optional device addend of `step` (CUDA-Graph replay)
  float* emb; int ldemb; float* user_emb;
  float* kl_part; int kl_stride;
  void* emb16 = nullptr; int ldemb16 = 0;   // optional fp16 copy of emb (16-bit integration path)
  void* eps16 = nullptr;                    // optional [n, F*32] 16-bit noise hand-off: forward writes, two-chain backward reads
  void* a0g = nullptr;                      // optional [2 F, n, 8] 16-bit [pe|1] operand hand-off, k-halves as planes (same direction)
};
int dib_enc_bwd_version();
void dib_enc_bwd_set_version(int v);
size_t dib_enc_fused_pack_bytes(int F);
long long dib_enc_fused_pack_zero_capacity(int F);
int dib_enc_fused_fwd_ctas_per_sm();
cudaError_t dib_enc_fused_pack(const DibEncFusedDesc& d, const float* params, void* packed, float* zero, long long zero_n, cudaStream_t st);
cudaError_t dib_enc_fused_forward(const DibEncFusedDesc& d, const DibEncFusedIO& io, cudaStream_t st);

struct DibEncFusedBwdIO {
  const float* d_emb; int ldd;          // gradient w.r.t. emb (scaled by 1/B_global), or null when d_emb16 is given
  const void* d_emb16 = nullptr; int ldd16 = 0;   // fp16 gradient already multiplied by gscale
  const float* beta_dev; float inv_batch; float gscale;
  float* part; long long split_stride;  // [slot][P] weight-gradient partials
};
cudaError_t dib_enc_fused_backward(const DibEncFusedDesc& d, const DibEncFusedIO& io, const DibEncFusedBwdIO& b,
                                   cudaStream_t st);

// ---- 16-bit integration network path (dib_int16.cu) ----
cudaError_t dib_int16_convert(const float* src, void* dst16, long long n, int bf16, cudaStream_t st);
cudaError_t dib_int16_convert_many(const float* const* src, void* const* dst16, const long long* n, int count, int bf16, cudaStream_t st);
cudaError_t dib_int16_fwd(const void* g_in, int ld_in, const void* w16, const float* bias, void* g_out, int ld_out, int M,
                          int K, int N, int act, float alpha, int bf16, cudaStream_t st);
// colsum_part (nullable): [ceil(M/128)][K] per-row-tile column sums of dz_in = bias-gradient partials of the layer below
cudaError_t dib_int16_dgrad(const void* dz, int ld_dz, const void* w16, const void* g_in, int ld_g, void* dz_in, int ld_out,
                            int M, int K, int N, int act, float alpha, float* colsum_part, int bf16, cudaStream_t st);
// several column-sum reductions in ONE launch: dst[i] = scale * sum_{r < nrows} src[r * row_stride + i], i < count (fixed order)
struct DibReduceSeg { const float* src; long long row_stride; int nrows; long long count; float scale; float* dst; };
constexpr int kDibMaxReduceSegs = 8;
cudaError_t dib_launch_reduce_segments(const DibReduceSeg* segs, int nseg, cudaStream_t st);
cudaError_t dib_launch_reduce_tall(const float* part, long long row_stride, int nrows, int64_t count, float scale, float* out,
                                   cudaStream_t st);
cudaError_t dib_int16_wgrad(const void* g_in, int ld_g, const void* dz, int ld_dz, float* dW_part, float* db_part, int M, int K,
                            int N, int nsplit, int rows_per_split, long long split_stride, float out_scale, int bf16, cudaStream_t st);
cudaError_t dib_int16_wgrad_pair(const void* g_in0, int K0, const void* dz0, int N0, float* dW_part0, int nsplit0, int rps0,
                                 const void* g_in1, int K1, const void* dz1, int N1, float* dW_part1, int nsplit1, int rps1,
                                 int M, long long split_stride, float out_scale, int bf16, cudaStream_t st);
int dib_int16_head_blocks(int num_sms);
void dib_int16_dbg_set(int v);
int dib_int16_2sm_enabled();
void dib_int16_2sm_set(int on);
int dib_int16_fwd2_enabled();
void dib_int16_fwd2_set(int on);
int dib_int16_fwd2_ok(int K0, int N1, int N2, int out_dim);
cudaError_t dib_int16_fwd2_head(const void* g_in, int ld_in, int K0, const void* w16_0, const float* b0, const void* w16_1, const float* b1,
                                void* g1, const float* wout, const float* bout, int act, int out_act, float alpha, int loss, const float* y,
                                int M, float inv_batch, float gscale, void* dg2, float* user_pred, float* wpart, int wpart_stride,
                                float* loss_part, float* acc_part, int* nblocks, int bf16, cudaStream_t st);
int dib_int16_rb_enabled();
void dib_int16_rb_set(int on);
void dib_int16_head1_set(int on);
cudaError_t dib_int16_head(const void* g, int ldg, int K, const float* Wc, const float* bc, int out_dim, int out_act, int hid_act,
                           float alpha, int loss, const float* y, long long n, float inv_batch, float gscale, void* dg, int lddg,
                           float* user_pred, float* wpart, int wpart_stride, float* loss_part, float* acc_part, int nblocks,
                           int bf16, cudaStream_t st);

cudaError_t dib_launch_mi_sandwich(const float* mu_logvar, int64_t n, int E, const float* eps, uint64_t seed, uint32_t step,
                                   float* row_scratch, float* out2, cudaStream_t st);
// G = features x batches groups of n rows in one launch, float64 accumulation; group g uses the noise stream
// (seed << 8) + g / batches_per_feature at step g % batches_per_feature
cudaError_t dib_launch_mi_sandwich_batched(const float* mu_logvar, int groups, int64_t n, int E, const float* eps, uint64_t seed,
                                           int batches_per_feature, double* row_scratch, double* out, cudaStream_t st);
