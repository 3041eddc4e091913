// dib_api.cu -- the C ABI declared in include/dib_b200.h: model description, workspace plan, and the
// orchestration of one forward / train step as a fixed sequence of asynchronous launches on the caller's stream.
#include <atomic>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "dib_common.cuh"
#include "dib_kernels.h"

namespace {

thread_local std::string g_last_error;
std::atomic<unsigned long long> g_launches{0};

int fail(const std::string& msg) {
  g_last_error = msg;
  return 1;
}

#define DIB_CUDA_OK(expr)                                                                        \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail(std::string(#expr) + ": " + cudaGetErrorString(_e));                           \
  } while (0)

struct Buf {
  long long off = 0;          // float offset inside the workspace
  int ld = 0;                 // leading dimension (multiple of 4)
  long long feat_stride = 0;  // distance between consecutive features (0 for single matrices)
};

constexpr int kMaxSplits = 32;
constexpr int kRowsPerBlock = 256;

}  // namespace

struct dib_model {
  int F = 0, L = 0, Li = 0, E = 0, D = 0, out = 0;
  int act = 0, out_act = 0, loss = 0, precision = 0, use_pe = 0, nfreq = 1;
  float alpha = 0.2f;
  long long maxB = 0;
  std::vector<int> fdims, enc_arch, int_arch;
  std::vector<int> x_off, pe_off, w_in;  // per feature: x column, pe column, first-layer fan-in
  int ldpe = 0;
  // parameters
  long long P = 0, Pp = 0;
  std::vector<long long> var_off;
  std::vector<int> var_rows, var_cols;
  std::vector<std::vector<long long>> encW, encB;  // [f][j]
  std::vector<long long> intW, intB;               // [j]
  // workspace plan
  long long ws_floats = 0;
  Buf pe, enc_out, emb, pred, d_pred, d_emb, d_out;
  std::vector<Buf> enc_act, d_enc;  // index 1..L  (output of layer j-1)
  std::vector<Buf> enc_drop;        // index 1..L  (dropout_rate > 0: what layer j reads -- enc_act[j] after Keras Dropout)
  float drop = 0.f;
  std::vector<Buf> int_act, d_int;  // index 1..Li
  long long part_off = 0, kl_part_off = 0, loss_part_off = 0, acc_part_off = 0, wshadow_off = 0;
  int nblk_max = 0;
  // device tables
  DibGemmProblem* d_probs = nullptr;
  std::vector<DibGemmProblem> h_probs;
  int* d_col_src = nullptr;
  int* d_col_freq = nullptr;
  int* d_col_feat = nullptr;   // feature owning each first-layer operand column (row gather of dib_compression_matrices)
  std::vector<int> enc_fwd, enc_dgrad, enc_wgrad;  // start index into d_probs per layer j
  std::vector<int> int_fwd, int_dgrad, int_wgrad;
  std::vector<int> enc_maxK;                        // max over features of fan-in of layer j
  // fused per-feature encoder kernels (tensor-core mode; dib_enc_fused.cu)
  bool fused_ok = false, fused_bwd_ok = false, force_unfused = false, force_int32 = false;
  DibEncFusedDesc fdesc;
  void* d_fused_tables = nullptr;
  long long pack_off = 0;       // packed 16-bit encoder weights inside the workspace (float offset)
  int kl_stride = 0, num_sms = 148, part_rows = kMaxSplits;
  // 16-bit integration network path (dib_int16.cu); offsets are FLOAT offsets into the workspace
  bool int16_ok = false;
  long long emb16_off = 0, demb16_off = 0, headpart_off = 0, dbpart_off = 0, eps16_off = 0, a0g_off = 0;
  int head_stride = 0, dbpart_stride = 0;
  long long dbpart_layer = 0;       // floats per layer of the dgrad column-sum partials
  std::vector<long long> g16_off, dg16_off, w16_off;   // [1..Li], [1..Li], [0..Li-1]
  int head_blocks = 0, lossacc_cap = 0;
  int head_used = 0;                // rows of the head partials the last forward wrote (fused tail kernel: its CTA count)
  // custom-step variants (SURVEY 8f3)
  float lv_off = 0.f, kl_exp = 1.f, kl_scale = 1.f;
  const uint32_t* step_dev = nullptr;  // optional device-resident addend of the Philox step word (dib_set_noise_step_device)
  bool simple = false;                 // nb-bool SimpleEncoder: two (1,1) constants per feature
  int* d_xoff = nullptr;               // device copy of x_off (simple-encoder kernels)
  long long beta_eff_off = 0;          // one float in the workspace: d(beta*scale*KL^p)/dKL
  // output encoder of a DIB_LOSS_INFONCE handle (train.py:186-193; dib_attach_output_encoder).  Its Q parameters sit at
  // params[P, P+Q) in Keras order; the GEMMs read them from a shadow in the workspace with every variable 4-float aligned:
  // [W0 | W1 | ... | b0 | b1 | ...] (the kernels TF32-rounded in the tensor-core modes)
  bool oe = false;
  int oe_dy = 0, oe_L = 0, oe_ldpe = 0;
  std::vector<int> oe_arch;
  long long Q = 0, oe_wlen = 0, oe_shadow_len = 0, oe_part_stride = 0;
  std::vector<long long> oe_var_off;                // relative to P, Keras order
  std::vector<int> oe_var_rows, oe_var_cols;
  std::vector<long long> oeW, oeB;                  // per layer: shadow / partial-row offsets
  Buf oe_pe, oe_out, oe_dout;
  std::vector<Buf> oe_act, oe_d;                    // index 1..oe_L
  long long oe_shadow_off = 0, oe_part_off = 0, oe_cont_off = 0, nce_loss_off = 0;
  int* d_oe_col_src = nullptr;
  int* d_oe_col_freq = nullptr;
  std::vector<int> oe_fwd, oe_dgrad, oe_wgrad;
  DibOePackTable oe_pack;
  // optional per-launch-group timing with CUDA events on the caller's stream (dib_profile_*)
  bool profiling = false;
  struct ProfRec { std::string label; cudaEvent_t a, b; };
  std::vector<ProfRec> prof;
};

namespace {

// precision modes: FP32 = CUDA-core FMA; TF32 = kind::tf32 grouped GEMMs on fp32 storage; FP16 / BF16 = the fused
// 16-bit-operand kernels (dib_enc_fused.cu, dib_int16.cu) where the shapes allow, kind::tf32 GEMMs elsewhere
bool is_tc(const dib_model* h) { return h->precision != DIB_PREC_FP32; }
bool want16(const dib_model* h) { return h->precision == DIB_PREC_FP16 || h->precision == DIB_PREC_BF16; }

int enc_fan_in(const dib_model* h, int f, int j) { return j == 0 ? h->w_in[f] : h->enc_arch[j - 1]; }
int enc_fan_out(const dib_model* h, int j) { return j < h->L ? h->enc_arch[j] : 2 * h->E; }
int int_fan_in(const dib_model* h, int j) { return j == 0 ? h->F * h->E : h->int_arch[j - 1]; }
int int_fan_out(const dib_model* h, int j) { return j < h->Li ? h->int_arch[j] : h->out; }
int oe_fan_in(const dib_model* h, int j) { return j == 0 ? h->oe_dy * h->nfreq : h->oe_arch[j - 1]; }
int oe_fan_out(const dib_model* h, int j) { return j < h->oe_L ? h->oe_arch[j] : h->out; }

long long take(long long& cursor, long long floats) {
  const long long off = cursor;
  cursor += DIB_ROUND_UP(floats, 64);   // 256-byte granularity
  return off;
}

Buf make_buf(long long& cursor, long long rows, int width, int nfeat) {
  Buf b;
  b.ld = DIB_ROUND_UP(width, 4);
  b.feat_stride = DIB_ROUND_UP(rows * b.ld, 64);
  b.off = take(cursor, b.feat_stride * nfeat);
  return b;
}

void plan(dib_model* h) {
  long long c = 0;
  const long long B = h->maxB;
  h->pe = make_buf(c, B, h->ldpe, 1);
  h->pe.ld = h->ldpe;
  h->enc_act.assign(h->L + 1, Buf());
  h->d_enc.assign(h->L + 1, Buf());
  for (int j = 1; j <= h->L; ++j) h->enc_act[j] = make_buf(c, B, h->enc_arch[j - 1], h->F);
  h->enc_drop.assign(h->L + 1, Buf());
  for (int j = 1; j <= h->L && h->drop > 0.f; ++j) h->enc_drop[j] = make_buf(c, B, h->enc_arch[j - 1], h->F);
  h->enc_out = make_buf(c, B, 2 * h->E, h->F);
  h->emb = make_buf(c, B, h->F * h->E, 1);
  h->int_act.assign(h->Li + 1, Buf());
  h->d_int.assign(h->Li + 1, Buf());
  for (int j = 1; j <= h->Li; ++j) h->int_act[j] = make_buf(c, B, h->int_arch[j - 1], 1);
  h->pred = make_buf(c, B, h->out, 1);
  // backward
  h->d_pred = make_buf(c, B, h->out, 1);
  for (int j = 1; j <= h->Li; ++j) h->d_int[j] = make_buf(c, B, h->int_arch[j - 1], 1);
  h->d_emb = make_buf(c, B, h->F * h->E, 1);
  h->d_out = make_buf(c, B, 2 * h->E, h->F);
  for (int j = 1; j <= h->L; ++j) h->d_enc[j] = make_buf(c, B, h->enc_arch[j - 1], h->F);
  h->nblk_max = (int)DIB_CEIL_DIV(B, (long long)kRowsPerBlock);
  h->part_rows = DIB_CEIL_DIV(h->num_sms, h->F) > kMaxSplits ? DIB_CEIL_DIV(h->num_sms, h->F) : kMaxSplits;
  h->part_off = take(c, (long long)h->part_rows * h->Pp);
  h->kl_stride = h->nblk_max > 2 * h->num_sms + 8 ? h->nblk_max : 2 * h->num_sms + 8;   // >= fused-kernel CTA slots per feature
  h->kl_part_off = take(c, (long long)h->F * h->kl_stride);
  h->head_blocks = dib_int16_head_blocks(h->num_sms);
  h->lossacc_cap = h->nblk_max > h->head_blocks ? h->nblk_max : h->head_blocks;
  h->loss_part_off = take(c, h->lossacc_cap);
  h->acc_part_off = take(c, h->lossacc_cap);
  {
    const long long FE = (long long)h->F * h->E;
    h->emb16_off = take(c, (B * FE + 1) / 2);
    h->demb16_off = take(c, (B * FE + 1) / 2);
    h->eps16_off = take(c, (B * FE + 1) / 2);      // the step's noise, 16-bit, from the forward to the backward kernel
    h->a0g_off = take(c, B * h->F * 8);            // ... and its [pe|1] first-layer operand rows (16 x 16-bit per row and feature)
    h->g16_off.assign(h->Li + 1, 0); h->dg16_off.assign(h->Li + 1, 0); h->w16_off.assign(h->Li + 1, 0);
    for (int j = 1; j <= h->Li; ++j) {
      h->g16_off[j] = take(c, (B * h->int_arch[j - 1] + 1) / 2);
      h->dg16_off[j] = take(c, (B * h->int_arch[j - 1] + 1) / 2);
    }
    for (int j = 0; j < h->Li; ++j) h->w16_off[j] = take(c, ((long long)int_fan_in(h, j) * int_fan_out(h, j) + 1) / 2);
    const int Kh = h->Li ? h->int_arch[h->Li - 1] : 1;
    h->head_stride = Kh * h->out + h->out + Kh;          // [dWc | dbc | column sums of dg (bias grad of the last hidden layer)]
    h->headpart_off = take(c, (long long)h->head_blocks * h->head_stride);
    int wmax = 1;
    for (int j = 0; j < h->Li; ++j) if (h->int_arch[j] > wmax) wmax = h->int_arch[j];
    h->dbpart_stride = wmax;                             // dgrad-epilogue column sums: [row tile][width]
    h->dbpart_layer = DIB_ROUND_UP((long long)DIB_CEIL_DIV(B, 128ll) * wmax, 64);
    h->dbpart_off = take(c, h->dbpart_layer * (h->Li > 0 ? h->Li : 1));    // one region per layer: all reduced in one launch
  }
  h->beta_eff_off = take(c, 64);
  h->wshadow_off = take(c, h->Pp);      // TF32-rounded copy of the parameters (tensor-core mode B operands)
  h->pack_off = take(c, (long long)(dib_enc_fused_pack_bytes(h->F) + 3) / 4);
  if (h->oe) {
    h->oe_pe = make_buf(c, B, h->oe_ldpe, 1);
    h->oe_act.assign(h->oe_L + 1, Buf());
    h->oe_d.assign(h->oe_L + 1, Buf());
    for (int j = 1; j <= h->oe_L; ++j) h->oe_act[j] = make_buf(c, B, h->oe_arch[j - 1], 1);
    h->oe_out = make_buf(c, B, h->out, 1);
    h->oe_dout = make_buf(c, B, h->out, 1);
    for (int j = 1; j <= h->oe_L; ++j) h->oe_d[j] = make_buf(c, B, h->oe_arch[j - 1], 1);
    h->oe_shadow_off = take(c, h->oe_shadow_len);
    h->oe_part_off = take(c, (long long)kMaxSplits * h->oe_part_stride);
    h->oe_cont_off = take(c, 4 * B * h->out);    // unpadded [n, D] e1 | e2 | d e1 | d e2 for the heads
    h->nce_loss_off = take(c, 64);
  }
  h->ws_floats = c;
}

void build_problems(dib_model* h, std::vector<DibGemmProblem>& v) {
  auto zero = [] { DibGemmProblem p; memset(&p, 0, sizeof(p)); return p; };
  const int F = h->F, L = h->L, Li = h->Li;
  h->enc_fwd.assign(L + 1, -1); h->enc_dgrad.assign(L + 1, -1); h->enc_wgrad.assign(L + 1, -1);
  h->int_fwd.assign(Li + 1, -1); h->int_dgrad.assign(Li + 1, -1); h->int_wgrad.assign(Li + 1, -1);
  h->enc_maxK.assign(L + 1, 0);
  auto encA = [&](int f, int j, long long& off, int& ld) {   // input of encoder layer j (after Dropout when there is one)
    if (j == 0) { off = h->pe.off + h->pe_off[f]; ld = h->ldpe; }
    else {
      const Buf& b = h->drop > 0.f ? h->enc_drop[j] : h->enc_act[j];
      off = b.off + f * b.feat_stride; ld = b.ld;
    }
  };
  auto encDZ = [&](int f, int j, long long& off, int& ld) {  // grad wrt pre-activation output of layer j
    const Buf& b = j == L ? h->d_out : h->d_enc[j + 1];
    off = b.off + f * b.feat_stride; ld = b.ld;
  };
  for (int j = 0; j <= L && !h->simple; ++j) {
    h->enc_fwd[j] = (int)v.size();
    for (int f = 0; f < F; ++f) {
      DibGemmProblem p = zero();
      encA(f, j, p.a_off, p.lda);
      p.b_off = h->encW[f][j]; p.ldb = enc_fan_out(h, j);
      const Buf& o = j < L ? h->enc_act[j + 1] : h->enc_out;
      p.c_off = o.off + f * o.feat_stride; p.ldc = o.ld;
      p.x_off = h->encB[f][j];
      p.T = enc_fan_in(h, f, j); p.C = enc_fan_out(h, j); p.act = j < L ? h->act : DIB_ACT_LINEAR;
      if (p.T > h->enc_maxK[j]) h->enc_maxK[j] = p.T;
      v.push_back(p);
    }
  }
  for (int j = 1; j <= L && !h->simple; ++j) {
    h->enc_dgrad[j] = (int)v.size();
    for (int f = 0; f < F; ++f) {
      DibGemmProblem p = zero();
      encDZ(f, j, p.a_off, p.lda);
      p.b_off = h->encW[f][j]; p.ldb = enc_fan_out(h, j);
      p.c_off = h->d_enc[j].off + f * h->d_enc[j].feat_stride; p.ldc = h->d_enc[j].ld;
      p.x_off = h->enc_act[j].off + f * h->enc_act[j].feat_stride; p.ldx = h->enc_act[j].ld;
      p.T = enc_fan_out(h, j); p.C = enc_fan_in(h, f, j); p.act = h->act;
      v.push_back(p);
    }
  }
  for (int j = 0; j <= L && !h->simple; ++j) {
    h->enc_wgrad[j] = (int)v.size();
    for (int f = 0; f < F; ++f) {
      DibGemmProblem p = zero();
      encA(f, j, p.a_off, p.lda);
      encDZ(f, j, p.b_off, p.ldb);
      p.c_off = h->encW[f][j]; p.ldc = enc_fan_out(h, j);
      p.x_off = h->encB[f][j];
      p.R = enc_fan_in(h, f, j); p.C = enc_fan_out(h, j);
      v.push_back(p);
    }
  }
  auto intA = [&](int j, long long& off, int& ld) {
    if (j == 0) { off = h->emb.off; ld = h->emb.ld; } else { off = h->int_act[j].off; ld = h->int_act[j].ld; }
  };
  auto intDZ = [&](int j, long long& off, int& ld) {
    const Buf& b = j == Li ? h->d_pred : h->d_int[j + 1];
    off = b.off; ld = b.ld;
  };
  for (int j = 0; j <= Li; ++j) {
    h->int_fwd[j] = (int)v.size();
    DibGemmProblem p = zero();
    intA(j, p.a_off, p.lda);
    p.b_off = h->intW[j]; p.ldb = int_fan_out(h, j);
    const Buf& o = j < Li ? h->int_act[j + 1] : h->pred;
    p.c_off = o.off; p.ldc = o.ld;
    p.x_off = h->intB[j];
    p.T = int_fan_in(h, j); p.C = int_fan_out(h, j); p.act = j < Li ? h->act : h->out_act;
    v.push_back(p);
  }
  for (int j = 0; j <= Li; ++j) {
    h->int_dgrad[j] = (int)v.size();
    DibGemmProblem p = zero();
    intDZ(j, p.a_off, p.lda);
    p.b_off = h->intW[j]; p.ldb = int_fan_out(h, j);
    const Buf& o = j == 0 ? h->d_emb : h->d_int[j];
    p.c_off = o.off; p.ldc = o.ld;
    if (j > 0) { p.x_off = h->int_act[j].off; p.ldx = h->int_act[j].ld; p.act = h->act; }
    else { p.act = DIB_ACT_LINEAR; }
    p.T = int_fan_out(h, j); p.C = int_fan_in(h, j);
    v.push_back(p);
  }
  for (int j = 0; j <= Li; ++j) {
    h->int_wgrad[j] = (int)v.size();
    DibGemmProblem p = zero();
    intA(j, p.a_off, p.lda);
    intDZ(j, p.b_off, p.ldb);
    p.c_off = h->intW[j]; p.ldc = int_fan_out(h, j);
    p.x_off = h->intB[j];
    p.R = int_fan_in(h, j); p.C = int_fan_out(h, j);
    v.push_back(p);
  }
  if (!h->oe) return;
  // output encoder: weights / biases / weight gradients are offsets into its shadow and its partial rows (gemm_oe)
  const int Lo = h->oe_L;
  h->oe_fwd.assign(Lo + 1, -1); h->oe_dgrad.assign(Lo + 1, -1); h->oe_wgrad.assign(Lo + 1, -1);
  auto oeA = [&](int j, long long& off, int& ld) {
    const Buf& b = j == 0 ? h->oe_pe : h->oe_act[j];
    off = b.off; ld = b.ld;
  };
  auto oeDZ = [&](int j, long long& off, int& ld) {
    const Buf& b = j == Lo ? h->oe_dout : h->oe_d[j + 1];
    off = b.off; ld = b.ld;
  };
  for (int j = 0; j <= Lo; ++j) {
    h->oe_fwd[j] = (int)v.size();
    DibGemmProblem p = zero();
    oeA(j, p.a_off, p.lda);
    p.b_off = h->oeW[j]; p.ldb = oe_fan_out(h, j);
    const Buf& o = j < Lo ? h->oe_act[j + 1] : h->oe_out;
    p.c_off = o.off; p.ldc = o.ld;
    p.x_off = h->oeB[j];
    p.T = oe_fan_in(h, j); p.C = oe_fan_out(h, j); p.act = j < Lo ? h->act : DIB_ACT_LINEAR;
    v.push_back(p);
  }
  for (int j = 1; j <= Lo; ++j) {
    h->oe_dgrad[j] = (int)v.size();
    DibGemmProblem p = zero();
    oeDZ(j, p.a_off, p.lda);
    p.b_off = h->oeW[j]; p.ldb = oe_fan_out(h, j);
    p.c_off = h->oe_d[j].off; p.ldc = h->oe_d[j].ld;
    p.x_off = h->oe_act[j].off; p.ldx = h->oe_act[j].ld; p.act = h->act;
    p.T = oe_fan_out(h, j); p.C = oe_fan_in(h, j);
    v.push_back(p);
  }
  for (int j = 0; j <= Lo; ++j) {
    h->oe_wgrad[j] = (int)v.size();
    DibGemmProblem p = zero();
    oeA(j, p.a_off, p.lda);
    oeDZ(j, p.b_off, p.ldb);
    p.c_off = h->oeW[j]; p.ldc = oe_fan_out(h, j);
    p.x_off = h->oeB[j];
    p.R = oe_fan_in(h, j); p.C = oe_fan_out(h, j);
    v.push_back(p);
  }
}

struct Ctx {
  dib_model* h;
  const float* params;
  float* ws;
  cudaStream_t st;
  int n;
  bool dev_step = false;     // dib_train_step only: add *h->step_dev to the Philox step word (dib_set_noise_step_device)
  const uint32_t* step_dev() const { return dev_step ? h->step_dev : nullptr; }
};

void prof_begin(const Ctx& c, const char* label, int j = -1) {
  if (!c.h->profiling) return;
  dib_model::ProfRec r;
  r.label = label;
  if (j >= 0) r.label += std::to_string(j);
  cudaEventCreate(&r.a); cudaEventCreate(&r.b);
  cudaEventRecord(r.a, c.st);
  c.h->prof.push_back(r);
}
void prof_end(const Ctx& c) {
  if (!c.h->profiling) return;
  cudaEventRecord(c.h->prof.back().b, c.st);
}

int gemm(const Ctx& c, int mode, int first, int nprob, int maxC, int maxR, int nsplit, int rps) {
  DibGemmLaunch L;
  L.probs = c.h->d_probs + first;
  L.nprob = nprob;
  L.M = c.n;
  L.maxC = maxC; L.maxR = maxR;
  L.nsplit = nsplit; L.rows_per_split = rps; L.split_stride = c.h->Pp;
  L.alpha = c.h->alpha;
  float* part = c.ws + c.h->part_off;
  const bool tc = is_tc(c.h);
  L.round_out = tc ? 1 : 0;
  switch (mode) {
    case DIB_GEMM_FWD: L.baseA = c.ws; L.baseB = c.params; L.baseC = c.ws; L.baseX = nullptr; break;
    case DIB_GEMM_DGRAD: L.baseA = c.ws; L.baseB = c.params; L.baseC = c.ws; L.baseX = c.ws; break;
    default: L.baseA = c.ws; L.baseB = c.ws; L.baseC = part; L.baseX = part; break;
  }
  if (tc && dib_gemm_tc_eligible(mode, c.h->h_probs.data() + first, nprob, c.params)) {
    if (mode != DIB_GEMM_WGRAD) { L.baseB = c.ws + c.h->wshadow_off; L.baseBias = c.params; }
    DIB_CUDA_OK(dib_launch_gemm_tc(mode, L, c.h->h_probs.data() + first, c.st));
    return 0;
  }
  DIB_CUDA_OK(dib_launch_gemm_simt(mode, L, c.st));
  return 0;
}

// one output-encoder layer: the same kernels as gemm(), with the weights and biases read from the encoder's aligned shadow
// and the weight-gradient partials written to its own partial rows
int gemm_oe(const Ctx& c, int mode, int first, int maxC, int maxR, int nsplit, int rps) {
  dib_model* h = c.h;
  DibGemmLaunch L;
  L.probs = h->d_probs + first;
  L.nprob = 1;
  L.M = c.n;
  L.maxC = maxC; L.maxR = maxR;
  L.nsplit = nsplit; L.rows_per_split = rps; L.split_stride = h->oe_part_stride;
  L.alpha = h->alpha;
  const bool tc = is_tc(h);
  L.round_out = tc ? 1 : 0;
  float* sh = c.ws + h->oe_shadow_off;
  float* part = c.ws + h->oe_part_off;
  switch (mode) {
    case DIB_GEMM_FWD: L.baseA = c.ws; L.baseB = sh; L.baseC = c.ws; L.baseX = nullptr; L.baseBias = sh; break;
    case DIB_GEMM_DGRAD: L.baseA = c.ws; L.baseB = sh; L.baseC = c.ws; L.baseX = c.ws; break;
    default: L.baseA = c.ws; L.baseB = c.ws; L.baseC = part; L.baseX = part; break;
  }
  if (tc && dib_gemm_tc_eligible(mode, h->h_probs.data() + first, 1, sh)) {
    DIB_CUDA_OK(dib_launch_gemm_tc(mode, L, h->h_probs.data() + first, c.st));
    return 0;
  }
  DIB_CUDA_OK(dib_launch_gemm_simt(mode, L, c.st));
  return 0;
}

// output_encoder(y) (train.py:186-193) on n rows into the oe_out workspace buffer
int oe_forward(const Ctx& c, const float* y) {
  dib_model* h = c.h;
  const int rnd = is_tc(h) ? 1 : 0;
  prof_begin(c, "oe_fwd");
  DIB_CUDA_OK(dib_launch_oe_pack(c.params + h->P, c.ws + h->oe_shadow_off, h->oe_pack, c.st));
  DIB_CUDA_OK(dib_launch_pe(y, h->oe_dy, 0, h->d_oe_col_src, h->d_oe_col_freq, 0, h->oe_ldpe, c.ws + h->oe_pe.off, h->oe_ldpe, 0,
                            c.n, rnd, c.st));
  for (int j = 0; j <= h->oe_L; ++j)
    if (gemm_oe(c, DIB_GEMM_FWD, h->oe_fwd[j], oe_fan_out(h, j), 0, 1, 0)) return 1;
  prof_end(c);
  return 0;
}

// reverse mode of oe_forward from d e2 in oe_dout (the shadow and the activations as oe_forward left them) ->
// grads_q [Q] in Keras order
int oe_backward(const Ctx& c, int nsplit, int rps, float* grads_q) {
  dib_model* h = c.h;
  prof_begin(c, "oe_bwd");
  for (int j = h->oe_L; j >= 0; --j) {
    if (gemm_oe(c, DIB_GEMM_WGRAD, h->oe_wgrad[j], oe_fan_out(h, j), oe_fan_in(h, j), nsplit, rps)) return 1;
    if (j >= 1 && gemm_oe(c, DIB_GEMM_DGRAD, h->oe_dgrad[j], oe_fan_in(h, j), 0, 1, 0)) return 1;
  }
  // fixed-order sums of the batch-split partials, written straight to the Keras-ordered gradient
  const float* part = c.ws + h->oe_part_off;
  std::vector<DibReduceSeg> segs;
  for (int v = 0; v < h->oe_pack.nvar; ++v) {
    segs.push_back({part + h->oe_pack.dst_off[v], h->oe_part_stride, nsplit, h->oe_pack.count[v], 1.f,
                    grads_q + h->oe_pack.src_off[v]});
    if ((int)segs.size() == kDibMaxReduceSegs || v + 1 == h->oe_pack.nvar) {
      DIB_CUDA_OK(dib_launch_reduce_segments(segs.data(), (int)segs.size(), c.st));
      segs.clear();
    }
  }
  prof_end(c);
  return 0;
}

int check_call(const dib_model* h, const void* params, const void* x, int64_t n, const void* ws) {
  if (!h) return fail("null model handle");
  if (!params || !ws || (!x && n > 0)) return fail("null params / x / workspace pointer");
  if (n < 0 || n > h->maxB) return fail("n = " + std::to_string(n) + " exceeds config.max_batch = " + std::to_string(h->maxB));
  if (reinterpret_cast<uintptr_t>(ws) & 255) return fail("workspace must be 256-byte aligned");
  if (reinterpret_cast<uintptr_t>(params) & 15) return fail("params must be 16-byte aligned");
  return 0;
}

// PE -> encoder layers (all features) -> reparam/KL -> integration layers -> loss/metrics
struct NoiseKey { uint64_t seed; uint32_t step; uint64_t sample_offset; bool training; };
int encode_all(const Ctx& c, const float* x, int ldx, int rnd, const int* row_index, int64_t n_src, const NoiseKey* key = nullptr);

// the compiled loss on the prediction in the pred buffer (d_pred when training) and the statistics vector.  A
// DIB_LOSS_INFONCE handle runs the external-loss branch: y is then d L_infonce / d e1.
int loss_and_stats(const Ctx& c, const float* y, float inv_batch, bool training, float* user_pred, float* out_stats, int nblk_kl) {
  dib_model* h = c.h;
  const int rnd = is_tc(h) ? 1 : 0;
  const int loss = h->loss == DIB_LOSS_INFONCE ? DIB_LOSS_EXTERNAL : h->loss;
  prof_begin(c, "loss_stats");
  DIB_CUDA_OK(dib_launch_loss(loss, h->out_act, h->alpha, c.ws + h->pred.off, h->pred.ld, y, h->out, c.n, inv_batch,
                              training ? c.ws + h->d_pred.off : nullptr, user_pred, c.ws + h->loss_part_off,
                              c.ws + h->acc_part_off, rnd, c.st));
  const int nblk = (int)DIB_CEIL_DIV((long long)c.n, (long long)kRowsPerBlock);
  DIB_CUDA_OK(dib_launch_finalize_stats(c.ws + h->kl_part_off, h->kl_stride, nblk_kl, c.ws + h->loss_part_off,
                                        c.ws + h->acc_part_off, nblk, h->F, c.n, y != nullptr, out_stats, c.st));
  prof_end(c);
  return 0;
}

// stop_nblk_kl != nullptr: stop after the integration network (the prediction is in the pred buffer) and return the KL
// partial count that loss_and_stats needs -- the InfoNCE step computes the loss gradient in between
int run_forward(const Ctx& c, const float* x, const float* y, const float* eps, uint64_t seed, uint32_t step,
                uint64_t sample_offset, float inv_batch, bool training, float* user_pred, float* user_emb,
                float* out_stats, bool enc_only = false, int* stop_nblk_kl = nullptr) {
  dib_model* h = c.h;
  const int rnd = is_tc(h) ? 1 : 0;
  const bool fast_path = h->fused_ok && rnd && (!training || h->fused_bwd_ok) && !h->force_unfused && h->int16_ok && !h->force_int32;
  if (rnd && !fast_path) {
    prof_begin(c, "weights_tf32_shadow");
    DIB_CUDA_OK(dib_launch_round_copy(c.params, c.ws + h->wshadow_off, h->P, c.st));
    prof_end(c);
  }
  // fused encoder path: only when the backward does not need the per-layer activations in HBM
  const bool fused = h->fused_ok && rnd && (!training || h->fused_bwd_ok) && !h->force_unfused;
  int nblk_kl = (int)DIB_CEIL_DIV((long long)c.n, (long long)kRowsPerBlock);
  if (fused) {
    const int ntiles = (int)DIB_CEIL_DIV((long long)c.n, 128ll);
    long long want = (long long)h->F * ntiles;
    DibEncFusedDesc d = h->fdesc;
    d.logvar_offset = h->lv_off;
    const long long cap = (long long)h->num_sms * dib_enc_fused_fwd_ctas_per_sm();
    d.grid = (int)(want < cap ? want : cap);
    nblk_kl = DIB_CEIL_DIV(d.grid, h->F);
    prof_begin(c, "enc_pack_weights");
    {
      const long long zn = (long long)h->F * h->kl_stride, zcap = dib_enc_fused_pack_zero_capacity(h->F);
      // the pack kernel also clears the KL partial table when it fits its grid
      if (zn <= zcap) DIB_CUDA_OK(dib_enc_fused_pack(d, c.params, c.ws + h->pack_off, c.ws + h->kl_part_off, zn, c.st));
      else {
        DIB_CUDA_OK(dib_enc_fused_pack(d, c.params, c.ws + h->pack_off, nullptr, 0, c.st));
        DIB_CUDA_OK(cudaMemsetAsync(c.ws + h->kl_part_off, 0, sizeof(float) * (size_t)zn, c.st));
      }
    }
    prof_end(c);
    DibEncFusedIO io;
    io.params = c.params; io.packed = c.ws + h->pack_off; io.x = x; io.ldx = h->D; io.n = c.n;
    io.eps = eps; io.seed = seed; io.step = step; io.step_dev = c.step_dev(); io.sample_offset = sample_offset;
    io.emb = c.ws + h->emb.off; io.ldemb = h->emb.ld; io.user_emb = user_emb;
    io.kl_part = c.ws + h->kl_part_off; io.kl_stride = h->kl_stride;
    const bool i16 = h->int16_ok && !h->force_int32 && !enc_only;
    if (i16) { io.emb = nullptr; io.emb16 = c.ws + h->emb16_off; io.ldemb16 = h->F * h->E; }
    if (enc_only) io.emb = nullptr;      // the caller's network consumes user_emb; nothing downstream reads the workspace copy
    if (training && !eps && dib_enc_bwd_version() >= 2) { io.eps16 = c.ws + h->eps16_off; io.a0g = c.ws + h->a0g_off; }
    prof_begin(c, "enc_fused_fwd");
    DIB_CUDA_OK(dib_enc_fused_forward(d, io, c.st));
    prof_end(c);
    if (enc_only) {
      DIB_CUDA_OK(dib_launch_finalize_stats(c.ws + h->kl_part_off, h->kl_stride, nblk_kl, c.ws + h->loss_part_off,
                                            c.ws + h->acc_part_off, 0, h->F, c.n, 0, out_stats, c.st));
      return 0;
    }
    if (i16) {
      const int bf = h->precision == DIB_PREC_BF16 ? 1 : 0;
      // ---------------- integration network on 16-bit activations + fused output head
      prof_begin(c, "int16_pack_weights");
      {
        std::vector<const float*> wsrc; std::vector<void*> wdst; std::vector<long long> wn;
        for (int j = 0; j < h->Li; ++j) {
          wsrc.push_back(c.params + h->intW[j]); wdst.push_back(c.ws + h->w16_off[j]);
          wn.push_back((long long)int_fan_in(h, j) * int_fan_out(h, j));
        }
        DIB_CUDA_OK(dib_int16_convert_many(wsrc.data(), wdst.data(), wn.data(), h->Li, bf, c.st));
      }
      prof_end(c);
      const int Kh = h->int_arch[h->Li - 1];
      const float gscale = training ? exp2f(ceilf(log2f(1.f / inv_batch))) : 1.f;
      // single-output models: the last two hidden layers and the head run as ONE kernel (g2 stays on chip)
      const bool fwd2 = h->Li >= 2 && dib_int16_fwd2_ok(int_fan_in(h, h->Li - 2), int_fan_out(h, h->Li - 2), int_fan_out(h, h->Li - 1), h->out);
      const int n_plain = fwd2 ? h->Li - 2 : h->Li;
      for (int j = 0; j < n_plain; ++j) {
        prof_begin(c, "int16_fwd_l", j);
        DIB_CUDA_OK(dib_int16_fwd(j == 0 ? (const void*)(c.ws + h->emb16_off) : (const void*)(c.ws + h->g16_off[j]), int_fan_in(h, j),
                                  c.ws + h->w16_off[j], c.params + h->intB[j], c.ws + h->g16_off[j + 1], int_fan_out(h, j), c.n,
                                  int_fan_in(h, j), int_fan_out(h, j), h->act, h->alpha, bf, c.st));
        prof_end(c);
      }
      if (fwd2) {
        const int j0 = h->Li - 2, j1 = h->Li - 1;
        prof_begin(c, "int16_fwd2_head");
        DIB_CUDA_OK(dib_int16_fwd2_head(j0 == 0 ? (const void*)(c.ws + h->emb16_off) : (const void*)(c.ws + h->g16_off[j0]), int_fan_in(h, j0),
                                        int_fan_in(h, j0), c.ws + h->w16_off[j0], c.params + h->intB[j0], c.ws + h->w16_off[j1],
                                        c.params + h->intB[j1], c.ws + h->g16_off[j1], c.params + h->intW[h->Li], c.params + h->intB[h->Li],
                                        h->act, h->out_act, h->alpha, h->loss, y, c.n, inv_batch, gscale,
                                        training ? (void*)(c.ws + h->dg16_off[h->Li]) : nullptr, user_pred, c.ws + h->headpart_off,
                                        h->head_stride, c.ws + h->loss_part_off, c.ws + h->acc_part_off, &h->head_used, bf, c.st));
        DIB_CUDA_OK(dib_launch_finalize_stats(c.ws + h->kl_part_off, h->kl_stride, nblk_kl, c.ws + h->loss_part_off,
                                              c.ws + h->acc_part_off, h->head_used, h->F, c.n, y != nullptr, out_stats, c.st));
        prof_end(c);
        return 0;
      }
      h->head_used = h->head_blocks;
      prof_begin(c, "int16_head_loss");
      DIB_CUDA_OK(dib_int16_head(c.ws + h->g16_off[h->Li], Kh, Kh, c.params + h->intW[h->Li], c.params + h->intB[h->Li], h->out,
                                 h->out_act, h->act, h->alpha, h->loss, y, c.n, inv_batch, gscale,
                                 training ? (void*)(c.ws + h->dg16_off[h->Li]) : nullptr, Kh, user_pred, c.ws + h->headpart_off,
                                 h->head_stride, c.ws + h->loss_part_off, c.ws + h->acc_part_off, h->head_blocks, bf, c.st));
      DIB_CUDA_OK(dib_launch_finalize_stats(c.ws + h->kl_part_off, h->kl_stride, nblk_kl, c.ws + h->loss_part_off,
                                            c.ws + h->acc_part_off, h->head_blocks, h->F, c.n, y != nullptr, out_stats, c.st));
      prof_end(c);
      return 0;
    }
  } else {
  const NoiseKey nk{seed, step, sample_offset, training};
  if (encode_all(c, x, h->D, rnd, nullptr, 0, &nk)) return 1;
  DibReparamArgs ra;
  ra.enc_out = c.ws + h->enc_out.off; ra.feat_stride = h->enc_out.feat_stride; ra.ldo = h->enc_out.ld;
  ra.eps = eps; ra.seed = seed; ra.step = step; ra.step_dev = c.step_dev(); ra.sample_offset = sample_offset;
  ra.F = h->F; ra.E = h->E; ra.n = c.n; ra.round_out = rnd;
  prof_begin(c, "reparam_kl_fwd");
  DIB_CUDA_OK(dib_launch_reparam_fwd(ra, c.ws + h->emb.off, h->emb.ld, user_emb, c.ws + h->kl_part_off, h->kl_stride, c.st));
  prof_end(c);
  if (enc_only) {
    DIB_CUDA_OK(dib_launch_finalize_stats(c.ws + h->kl_part_off, h->kl_stride, nblk_kl, c.ws + h->loss_part_off,
                                          c.ws + h->acc_part_off, 0, h->F, c.n, 0, out_stats, c.st));
    return 0;
  }
  }
  for (int j = 0; j <= h->Li; ++j) {
    prof_begin(c, "int_fwd_l", j);
    if (gemm(c, DIB_GEMM_FWD, h->int_fwd[j], 1, int_fan_out(h, j), 0, 1, 0)) return 1;
    prof_end(c);
  }
  if (stop_nblk_kl) { *stop_nblk_kl = nblk_kl; return 0; }
  return loss_and_stats(c, y, inv_batch, training, user_pred, out_stats, nblk_kl);
}

// every feature encoder on n rows of x (deterministic part: mu | logvar incl. the offset) into the enc_out workspace
// buffer: positional encoding + grouped GEMMs (models.py:72-78,106), or nb-bool's SimpleEncoder constants
int encode_all(const Ctx& c, const float* x, int ldx, int rnd, const int* row_index, int64_t n_src, const NoiseKey* key) {
  dib_model* h = c.h;
  if (h->simple) {
    prof_begin(c, "simple_enc_fwd");
    DIB_CUDA_OK(dib_launch_simple_enc_fwd(x, ldx, h->d_xoff, c.params, c.ws + h->enc_out.off, h->enc_out.feat_stride,
                                          h->enc_out.ld, h->F, h->E, c.n, -1, 0, row_index, n_src, c.st));
    prof_end(c);
  } else {
    prof_begin(c, "pe");
    DIB_CUDA_OK(dib_launch_pe(x, ldx, 0, h->d_col_src, h->d_col_freq, 0, h->ldpe, c.ws + h->pe.off, h->ldpe, 0, c.n, rnd, c.st,
                              row_index, row_index ? h->d_col_feat : nullptr, n_src));
    prof_end(c);
    for (int j = 0; j <= h->L; ++j) {
      prof_begin(c, "enc_fwd_l", j);
      if (gemm(c, DIB_GEMM_FWD, h->enc_fwd[j], h->F, enc_fan_out(h, j), 0, 1, 0)) return 1;
      if (j < h->L && h->drop > 0.f) {     // Keras Dropout after the hidden Dense (training) / identity copy (inference)
        const bool tr = key && key->training;
        DIB_CUDA_OK(dib_launch_dropout(c.ws + h->enc_act[j + 1].off, c.ws + h->enc_drop[j + 1].off, h->enc_act[j + 1].feat_stride,
                                       h->enc_act[j + 1].ld, h->enc_arch[j], h->F, c.n, tr ? h->drop : 0.f, key ? key->seed : 0,
                                       key ? key->step : 0, tr ? c.step_dev() : nullptr, key ? key->sample_offset : 0, j + 1, -1, 0,
                                       rnd, c.st));
      }
      prof_end(c);
    }
  }
  DIB_CUDA_OK(dib_launch_add_logvar_offset(c.ws + h->enc_out.off, h->enc_out.feat_stride, h->enc_out.ld, h->F, h->E, c.n,
                                           h->lv_off, -1, c.st));
  return 0;
}

// weight for the per-sample KL gradients: beta itself (models.py:118) or d(beta*scale*KL^p)/dKL (nb-chaos cell 10)
int ib_weight(const Ctx& c, const float* beta_dev, const float* stats, float inv_global_batch, const float** out) {
  dib_model* h = c.h;
  *out = beta_dev;
  if (h->kl_exp == 1.f && h->kl_scale == 1.f) return 0;
  float* be = c.ws + h->beta_eff_off;
  DIB_CUDA_OK(dib_launch_beta_eff(stats, h->F, inv_global_batch, beta_dev, h->kl_exp, h->kl_scale, be, c.st));
  *out = be;
  return 0;
}

}  // namespace

// =================================================================================================
void dib_note_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

extern "C" {

uint64_t dib_launch_count(void) { return g_launches.load(); }

// bring-up switch: 1 = never use the fused encoder kernels (compare fused vs unfused tensor-core paths)
int dib_debug_force_unfused(dib_model* h, int32_t on) {
  if (!h) return fail("null model handle");
  h->force_unfused = (on & 1) != 0;      // bit 0: unfused encoder kernels
  h->force_int32 = (on & 2) != 0;        // bit 1: integration network on the fp32-storage TF32 kernels
  return 0;
}

// kernel-variant switch for A/B measurements: key 0 = fused encoder backward kernel (1 = single chain, 2 = two chains);
// key 1 = integration FWD/DGRAD GEMMs with the weight slice resident in shared memory (1, default) or re-streamed (0)
int dib_debug_set_variant(int32_t key, int32_t value) {
  if (key == 0) { dib_enc_bwd_set_version(value); return 0; }
  if (key == 1) { dib_int16_rb_set(value); return 0; }
  if (key == 2) { dib_int16_head1_set(value); return 0; }
  if (key == 3) { dib_int16_fwd2_set(value); return 0; }
  if (key == 4) { dib_int16_2sm_set(value); return 0; }
  if (key == 5) { dib_int16_dbg_set(value); return 0; }     // measurement only: wrong results
  return fail("dib_debug_set_variant: unknown key");
}

int dib_profile_enable(dib_model* h, int32_t on) {
  if (!h) return fail("null model handle");
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  h->prof.clear();
  h->profiling = on != 0;
  return 0;
}

int32_t dib_profile_read(dib_model* h, char* labels, size_t labels_bytes, float* ms, int32_t capacity) {
  if (!h) { fail("null model handle"); return -1; }
  std::string all;
  int32_t n = 0;
  for (auto& r : h->prof) {
    if (n >= capacity) break;
    if (cudaEventSynchronize(r.b) != cudaSuccess) { fail("dib_profile_read: event sync failed"); return -1; }
    float t = 0.f;
    cudaEventElapsedTime(&t, r.a, r.b);
    ms[n++] = t;
    all += r.label; all += '\n';
  }
  if (labels && labels_bytes) {
    const size_t k = all.size() < labels_bytes - 1 ? all.size() : labels_bytes - 1;
    memcpy(labels, all.data(), k); labels[k] = 0;
  }
  return n;
}

// single-problem GEMM through the tensor-core kernel (bring-up / unit tests): see DibGemmProblem for the modes
int dib_debug_gemm_tc(int32_t mode, const float* A, int32_t lda, const float* B, int32_t ldb, float* Cout, int32_t ldc,
                      float* X, int32_t ldx, int32_t M, int32_t T, int32_t Ccols, int32_t R, int32_t act,
                      int32_t nsplit, int32_t rows_per_split, int64_t split_stride, int32_t use_simt, void* stream) {
  DibGemmProblem p;
  memset(&p, 0, sizeof(p));
  p.lda = lda; p.ldb = ldb; p.ldc = ldc; p.ldx = ldx; p.T = T; p.C = Ccols; p.R = R; p.act = act;
  p.x_off = 0;
  DibGemmProblem* dp = nullptr;
  DIB_CUDA_OK(cudaMalloc(&dp, sizeof(p)));
  DIB_CUDA_OK(cudaMemcpy(dp, &p, sizeof(p), cudaMemcpyHostToDevice));
  DibGemmLaunch L;
  L.probs = dp; L.nprob = 1; L.baseA = A; L.baseB = B; L.baseC = Cout; L.baseX = X; L.M = M;
  L.maxC = Ccols; L.maxR = R; L.nsplit = nsplit < 1 ? 1 : nsplit; L.rows_per_split = rows_per_split;
  L.split_stride = split_stride; L.alpha = 0.2f;
  cudaError_t e;
  if (use_simt) e = dib_launch_gemm_simt(mode, L, static_cast<cudaStream_t>(stream));
  else if (!dib_gemm_tc_eligible(mode, &p, 1, nullptr)) { cudaFree(dp); return fail("dib_debug_gemm_tc: not eligible"); }
  else e = dib_launch_gemm_tc(mode, L, &p, static_cast<cudaStream_t>(stream));
  cudaError_t e2 = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
  cudaFree(dp);
  if (e != cudaSuccess) return fail(std::string("launch: ") + cudaGetErrorString(e));
  if (e2 != cudaSuccess) return fail(std::string("sync: ") + cudaGetErrorString(e2));
  return 0;
}

const char* dib_last_error(void) { return g_last_error.c_str(); }

const char* dib_build_info(void) {
  return "dib_b200 abi=2 arch=sm_100a paths=fp32-simt,tf32-tcgen05,fp16-fused-tcgen05,bf16-fused-tcgen05";
}

int32_t dib_model_info(const dib_model* h, char* out, size_t out_bytes) {
  if (!h || !out || out_bytes < 2) { fail("dib_model_info: bad arguments"); return -1; }
  static const char* pn[] = {"fp32", "tf32", "bf16", "fp16"};
  const bool fused = h->fused_ok && h->fused_bwd_ok && !h->force_unfused;
  const bool i16 = fused && h->int16_ok && !h->force_int32;
  const char* k16 = h->precision == DIB_PREC_BF16 ? "bf16" : "f16";
  std::string s = std::string("precision=") + pn[h->precision];
  if (!is_tc(h)) s += " encoders=simt-fp32 integration=simt-fp32 operands=fp32 accumulate=fp32";
  else {
    s += fused ? std::string(" encoders=fused-tcgen05-") + k16 : std::string(" encoders=grouped-tcgen05-tf32");
    s += i16 ? std::string(" integration=int16-tcgen05-") + k16 : std::string(" integration=tcgen05-tf32");
    s += fused ? std::string(" operands=") + (h->precision == DIB_PREC_BF16 ? "bf16" : "fp16") : std::string(" operands=tf32");
    s += " accumulate=fp32";
  }
  if (h->oe) {      // the kernel family of each output-encoder layer (narrow first layers stay on the SIMT kernel)
    s += " output_encoder=";
    for (int j = 0; j <= h->oe_L; ++j) {
      const bool tc = is_tc(h) && dib_gemm_tc_eligible(DIB_GEMM_FWD, &h->h_probs[h->oe_fwd[j]], 1, nullptr);
      s += std::string(j ? "," : "") + (tc ? "tcgen05-tf32" : "simt-fp32");
    }
  }
  const size_t k = s.size() < out_bytes - 1 ? s.size() : out_bytes - 1;
  memcpy(out, s.data(), k); out[k] = 0;
  return (int32_t)k;
}

int dib_create(const dib_config* cfg, dib_model** out) {
  if (!cfg || !out) return fail("dib_create: null argument");
  *out = nullptr;
  if (cfg->abi_version != DIB_ABI_VERSION) return fail("dib_create: abi_version mismatch");
  if (cfg->number_features < 1 || cfg->feature_embedding_dimension < 1 || cfg->output_dimensionality < 1 ||
      cfg->max_batch < 1 || cfg->number_encoder_layers < 0 || cfg->number_integration_layers < 0)
    return fail("dib_create: invalid sizes");
  if (cfg->max_batch > 0x7fffffffll) return fail("dib_create: max_batch too large");
  if (cfg->precision < DIB_PREC_FP32 || cfg->precision > DIB_PREC_FP16)
    return fail("dib_create: unknown precision");
  if (cfg->activation_fn < 0 || cfg->activation_fn > DIB_ACT_ELU || cfg->output_activation_fn < 0 ||
      cfg->output_activation_fn > DIB_ACT_ELU)
    return fail("dib_create: unknown activation");
  if (cfg->loss < 0 || cfg->loss > DIB_LOSS_INFONCE) return fail("dib_create: unknown loss");
  if (cfg->loss == DIB_LOSS_INFONCE && cfg->output_activation_fn != DIB_ACT_LINEAR)
    return fail("dib_create: DIB_LOSS_INFONCE needs a linear output activation (the model output is the embedding e1)");
  dib_model* h = new (std::nothrow) dib_model();
  if (!h) return fail("dib_create: out of host memory");
  h->F = cfg->number_features; h->L = cfg->number_encoder_layers; h->Li = cfg->number_integration_layers;
  h->E = cfg->feature_embedding_dimension; h->out = cfg->output_dimensionality;
  h->act = cfg->activation_fn; h->out_act = cfg->output_activation_fn; h->loss = cfg->loss;
  h->precision = cfg->precision; h->use_pe = cfg->use_positional_encoding ? 1 : 0;
  h->alpha = cfg->leaky_relu_alpha; h->maxB = cfg->max_batch;
  h->lv_off = cfg->logvar_offset;
  h->kl_exp = cfg->kl_loss_exponent == 0.f ? 1.f : cfg->kl_loss_exponent;
  h->kl_scale = cfg->kl_loss_scale == 0.f ? 1.f : cfg->kl_loss_scale;
  h->simple = cfg->encoder_kind == DIB_ENCODER_SIMPLE;
  h->drop = cfg->dropout_rate;
  if (!(h->drop >= 0.f && h->drop < 1.f)) { delete h; return fail("dib_create: dropout_rate must be in [0, 1)"); }
  if (cfg->encoder_kind != DIB_ENCODER_MLP && cfg->encoder_kind != DIB_ENCODER_SIMPLE) { delete h; return fail("dib_create: unknown encoder_kind"); }
  if (!(h->kl_exp > 0.f)) { delete h; return fail("dib_create: kl_loss_exponent must be > 0"); }
  if (h->simple) { h->L = 0; h->use_pe = 0; }
  // models.py:70: frequencies 2**arange(1, n) -> n-1 sinusoid blocks after the identity block
  h->nfreq = h->use_pe ? (cfg->number_positional_encoding_frequencies > 1 ? cfg->number_positional_encoding_frequencies : 1) : 1;
  h->fdims.assign(cfg->feature_dimensionalities, cfg->feature_dimensionalities + h->F);
  h->enc_arch.assign(cfg->feature_encoder_architecture, cfg->feature_encoder_architecture + h->L);
  if (h->simple) for (int d : h->fdims) if (d != h->E) { delete h; return fail("dib_create: SimpleEncoder needs d_i == feature_embedding_dimension"); }
  h->int_arch.assign(cfg->integration_network_architecture, cfg->integration_network_architecture + h->Li);
  for (int d : h->fdims) if (d < 1) { delete h; return fail("dib_create: feature dimensionality < 1"); }
  for (int d : h->enc_arch) if (d < 1) { delete h; return fail("dib_create: encoder width < 1"); }
  for (int d : h->int_arch) if (d < 1) { delete h; return fail("dib_create: integration width < 1"); }

  // first-layer operand layout: per feature a zero-padded block of width round_up(d_i * nfreq, 4)
  std::vector<int> col_src, col_freq, col_feat;
  h->D = 0;
  for (int f = 0; f < h->F; ++f) {
    const int d = h->fdims[f], w = d * h->nfreq;
    h->x_off.push_back(h->D);
    h->pe_off.push_back((int)col_src.size());
    h->w_in.push_back(w);
    for (int blk = 0; blk < h->nfreq; ++blk)
      for (int k = 0; k < d; ++k) { col_src.push_back(h->D + k); col_freq.push_back(blk == 0 ? 0 : (1 << blk)); }
    while (col_src.size() % 4) { col_src.push_back(-1); col_freq.push_back(0); }
    col_feat.resize(col_src.size(), f);
    h->D += d;
  }
  h->ldpe = (int)col_src.size();

  // flat parameter layout (Keras variable order: per feature W,b per layer; then the integration network)
  long long off = 0;
  auto add_var = [&](int rows, int cols) {
    h->var_off.push_back(off); h->var_rows.push_back(rows); h->var_cols.push_back(cols);
    const long long o = off; off += (long long)(rows ? rows : 1) * cols; return o;
  };
  h->encW.assign(h->F, {}); h->encB.assign(h->F, {});
  for (int f = 0; f < h->F; ++f) {
    if (h->simple) {                       // nb-bool cell 4: mu_scaling (1,1), logvar (1,1)
      h->encW[f].push_back(add_var(1, 1));
      h->encB[f].push_back(add_var(1, 1));
      continue;
    }
    for (int j = 0; j <= h->L; ++j) {
      h->encW[f].push_back(add_var(enc_fan_in(h, f, j), enc_fan_out(h, j)));
      h->encB[f].push_back(add_var(0, enc_fan_out(h, j)));
    }
  }
  for (int j = 0; j <= h->Li; ++j) {
    h->intW.push_back(add_var(int_fan_in(h, j), int_fan_out(h, j)));
    h->intB.push_back(add_var(0, int_fan_out(h, j)));
  }
  h->P = off; h->Pp = DIB_ROUND_UP(off, 64);
  {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || h->num_sms < 1)
      h->num_sms = 148;
  }
  plan(h);

  std::vector<DibGemmProblem> probs;
  build_problems(h, probs);
  h->h_probs = probs;
  cudaError_t e = cudaMalloc(&h->d_probs, probs.size() * sizeof(DibGemmProblem));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_col_src, col_src.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_col_freq, col_freq.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_col_feat, col_feat.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_xoff, h->x_off.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_xoff, h->x_off.data(), h->x_off.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_probs, probs.data(), probs.size() * sizeof(DibGemmProblem), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_col_src, col_src.data(), col_src.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_col_freq, col_freq.data(), col_freq.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_col_feat, col_feat.data(), col_feat.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    std::string msg = std::string("dib_create: CUDA error: ") + cudaGetErrorString(e);
    dib_destroy(h);
    return fail(msg);
  }
  // ---- fused encoder kernels: two hidden layers of 128, E = 32, first-layer fan-in (+ bias column) <= 16
  {
    bool ok = want16(h) && h->drop == 0.f && h->L == 2 && h->enc_arch[0] == 128 && h->enc_arch[1] == 128 && h->E == 32;
    for (int f = 0; ok && f < h->F; ++f) ok = h->w_in[f] + 1 <= 16;
    if (ok) {
      const int F = h->F;
      std::vector<long long> tab(6 * (size_t)F);
      std::vector<int> itab(2 * (size_t)F);
      for (int f = 0; f < F; ++f) {
        tab[0 * F + f] = h->encW[f][0]; tab[1 * F + f] = h->encB[f][0]; tab[2 * F + f] = h->encW[f][1];
        tab[3 * F + f] = h->encB[f][1]; tab[4 * F + f] = h->encW[f][2]; tab[5 * F + f] = h->encB[f][2];
        itab[f] = h->x_off[f]; itab[F + f] = h->fdims[f];
      }
      const size_t b1 = tab.size() * sizeof(long long), b2 = itab.size() * sizeof(int);
      cudaError_t fe = cudaMalloc(&h->d_fused_tables, b1 + b2);
      if (fe == cudaSuccess) fe = cudaMemcpy(h->d_fused_tables, tab.data(), b1, cudaMemcpyHostToDevice);
      if (fe == cudaSuccess) fe = cudaMemcpy(static_cast<char*>(h->d_fused_tables) + b1, itab.data(), b2, cudaMemcpyHostToDevice);
      if (fe == cudaSuccess) {
        const long long* lt = static_cast<const long long*>(h->d_fused_tables);
        const int* it = reinterpret_cast<const int*>(static_cast<const char*>(h->d_fused_tables) + b1);
        DibEncFusedDesc& d = h->fdesc;
        d.F = F; d.nfreq = h->nfreq; d.act = h->act; d.alpha = h->alpha; d.bf16 = h->precision == DIB_PREC_BF16 ? 1 : 0;
        d.w0_off = lt; d.b0_off = lt + F; d.w1_off = lt + 2 * F; d.b1_off = lt + 3 * F; d.w2_off = lt + 4 * F;
        d.b2_off = lt + 5 * F; d.x_off = it; d.fdim = it + F;
        h->fused_ok = true;
        h->fused_bwd_ok = true;
        // 16-bit integration path: hidden widths multiples of 128, last hidden width 256, narrow output head
        // (the fused head owns the compiled loss, so a caller-owned loss takes the TF32 integration kernels)
        bool iok = h->Li >= 1 && (h->F * h->E) % 64 == 0 && h->int_arch[h->Li - 1] == 256 && h->out <= 16 &&
                   h->loss != DIB_LOSS_EXTERNAL && h->loss != DIB_LOSS_INFONCE;
        for (int j = 0; iok && j < h->Li; ++j) iok = h->int_arch[j] % 128 == 0 && (h->intB[j] & 3) == 0;
        h->int16_ok = iok;
      }
    }
  }
  *out = h;
  return 0;
}

void dib_destroy(dib_model* h) {
  if (!h) return;
  if (h->d_probs) cudaFree(h->d_probs);
  if (h->d_col_src) cudaFree(h->d_col_src);
  if (h->d_col_freq) cudaFree(h->d_col_freq);
  if (h->d_col_feat) cudaFree(h->d_col_feat);
  if (h->d_xoff) cudaFree(h->d_xoff);
  if (h->d_fused_tables) cudaFree(h->d_fused_tables);
  if (h->d_oe_col_src) cudaFree(h->d_oe_col_src);
  if (h->d_oe_col_freq) cudaFree(h->d_oe_col_freq);
  for (auto& r : h->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  delete h;
}

int64_t dib_param_count(const dib_model* h) { return h ? h->P : -1; }

int dib_param_layout(const dib_model* h, int64_t* offsets, int32_t* rows, int32_t* cols, int32_t capacity) {
  if (!h) { fail("null model handle"); return -1; }
  const int nv = (int)h->var_off.size();
  if (!offsets || !rows || !cols) return nv;
  if (capacity < nv) { fail("dib_param_layout: capacity too small"); return -1; }
  for (int i = 0; i < nv; ++i) { offsets[i] = h->var_off[i]; rows[i] = h->var_rows[i]; cols[i] = h->var_cols[i]; }
  return nv;
}

size_t dib_workspace_bytes(const dib_model* h) { return h ? (size_t)h->ws_floats * sizeof(float) : 0; }

int32_t dib_stats_count(const dib_model* h) { return h ? h->F + 3 : -1; }

int dib_forward(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset, float* out_pred, float* out_emb,
                float* out_stats, void* workspace, void* stream) {
  (void)beta_dev;
  if (check_call(h, params, x, n, workspace)) return 1;
  if (!out_stats) return fail("dib_forward: out_stats is required");
  if (h->loss == DIB_LOSS_INFONCE && y) return fail("dib_forward: a DIB_LOSS_INFONCE handle takes y = NULL (the loss needs e2: dib_infonce_forward)");
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  if (n == 0) { DIB_CUDA_OK(cudaMemsetAsync(out_stats, 0, sizeof(float) * (h->F + 3), c.st)); return 0; }
  return run_forward(c, x, y, eps, seed, step, sample_offset, 0.f, false, out_pred, out_emb, out_stats);
}

int dib_encode_feature(dib_model* h, const float* params, int32_t feature, const float* x_i, int64_t n,
                       float* out_mu_logvar, void* workspace, void* stream) {
  if (check_call(h, params, x_i, n, workspace)) return 1;
  if (feature < 0 || feature >= h->F) return fail("dib_encode_feature: feature index out of range");
  if (!out_mu_logvar) return fail("dib_encode_feature: null output");
  if (n == 0) return 0;
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  const int f = feature, wpad = DIB_ROUND_UP(h->w_in[f], 4);
  const int rnd = is_tc(h) ? 1 : 0;
  if (h->simple) {
    DIB_CUDA_OK(dib_launch_simple_enc_fwd(x_i, h->fdims[f], h->d_xoff, c.params, c.ws + h->enc_out.off, h->enc_out.feat_stride,
                                          h->enc_out.ld, h->F, h->E, n, f, 1, nullptr, 0, c.st));
  } else {
    if (rnd) DIB_CUDA_OK(dib_launch_round_copy(c.params, c.ws + h->wshadow_off, h->P, c.st));
    DIB_CUDA_OK(dib_launch_pe(x_i, h->fdims[f], h->x_off[f], h->d_col_src, h->d_col_freq, h->pe_off[f], h->pe_off[f] + wpad,
                              c.ws + h->pe.off, h->ldpe, 0, n, rnd, c.st));
    for (int j = 0; j <= h->L; ++j) {
      if (gemm(c, DIB_GEMM_FWD, h->enc_fwd[j] + f, 1, enc_fan_out(h, j), 0, 1, 0)) return 1;
      if (j < h->L && h->drop > 0.f)       // inference: Dropout is the identity
        DIB_CUDA_OK(dib_launch_dropout(c.ws + h->enc_act[j + 1].off, c.ws + h->enc_drop[j + 1].off, h->enc_act[j + 1].feat_stride,
                                       h->enc_act[j + 1].ld, h->enc_arch[j], h->F, n, 0.f, 0, 0, nullptr, 0, j + 1, f, 0, rnd, c.st));
    }
  }
  DIB_CUDA_OK(dib_launch_add_logvar_offset(c.ws + h->enc_out.off, h->enc_out.feat_stride, h->enc_out.ld, h->F, h->E, n,
                                           h->lv_off, f, c.st));
  DIB_CUDA_OK(dib_launch_copy2d(c.ws + h->enc_out.off + f * h->enc_out.feat_stride, h->enc_out.ld, out_mu_logvar,
                                2 * h->E, 2 * h->E, n, c.st));
  return 0;
}

// phases: 1 = forward + compiled loss + integration-network backward (grads_flat[first integration parameter ..) final),
//         2 = encoder backward (grads_flat[0 .. first integration parameter) final); 3 = both (= dib_train_step).
// Phase 2 relies on the workspace exactly as phase 1 left it (same x, eps / seed / step, n).
}  // extern "C"

namespace {

// the body of dib_train_step_phased for n > 0.  forward_done: the caller already ran the forward, the loss gradient into
// d_pred and out_stats (the InfoNCE step); phase 1 then starts at the IB weight.
int train_phases(const Ctx& c, const float* x, const float* y, int64_t n, const float* beta_dev, float inv_global_batch,
                 const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset, float* grads_flat, float* out_stats,
                 int32_t phases, bool forward_done) {
  dib_model* h = c.h;
  const bool phA = (phases & 1) != 0, phB = (phases & 2) != 0;
  const long long p_enc = h->intW[0];                // encoder parameters occupy [0, p_enc)
  const bool nonlinear = h->kl_exp != 1.f || h->kl_scale != 1.f;
  if (phA) {
    if (!forward_done &&
        run_forward(c, x, y, eps, seed, step, sample_offset, inv_global_batch, true, nullptr, nullptr, out_stats)) return 1;
    const float* bw = nullptr;
    if (ib_weight(c, beta_dev, out_stats, inv_global_batch, &bw)) return 1;
  }
  // weight of the per-sample KL gradients in the encoder backward: beta, or d(beta*scale*KL^p)/dKL left in the workspace by phase 1
  const float* beta_w = nonlinear ? c.ws + h->beta_eff_off : beta_dev;

  // deterministic split of the batch for the weight gradients
  long long rps = DIB_CEIL_DIV((long long)n, (long long)kMaxSplits);
  if (rps < 256) rps = 256;
  rps = DIB_ROUND_UP(rps, 64);      // whole k-blocks of every WGRAD kernel (32 rows for the TF32 ones, 64 for the 16-bit ones)
  const int nsplit = (int)DIB_CEIL_DIV((long long)n, rps);
  float* part = c.ws + h->part_off;

  const bool fused_enc = h->fused_ok && h->fused_bwd_ok && !h->force_unfused;
  const bool i16 = fused_enc && h->int16_ok && !h->force_int32;
  const float gscale = exp2f(ceilf(log2f(1.f / inv_global_batch)));

  std::vector<DibReduceSeg> segs;          // fixed-order reductions of the step; whole steps (phases == 3) run them as ONE launch at the end
  // ---------------------------------------------------------------- phase 1: integration network backward
  if (phA && i16) {
    const int bf = h->precision == DIB_PREC_BF16 ? 1 : 0;
    const int Kh = h->int_arch[h->Li - 1];
    const int row_tiles = (int)DIB_CEIL_DIV((long long)n, 128ll);
    const long long p_head = h->intW[h->Li];
    // every fixed-order reduction of this phase runs as ONE launch at its end (bias gradients from the head / dgrad column sums,
    // batch-split weight-gradient partials, the output layer's per-CTA partials)
    // bias gradient of the last hidden layer: column sums of dg accumulated by the output head
    segs.push_back({c.ws + h->headpart_off + (long long)Kh * h->out + h->out, h->head_stride, h->head_used, Kh, 1.f / gscale,
                    grads_flat + h->intB[h->Li - 1]});
    // the dgrad chain first (layer j's dgrad produces the gradient layer j-1's wgrad consumes), then the weight gradients in PAIRS of
    // layers per launch: one layer's [K/128 x N/128 x splits] tiles do not fill the 2 x SMs CTA slots, two layers' tiles do
    for (int j = h->Li - 1; j >= 0; --j) {
      const int K = int_fan_in(h, j), N = int_fan_out(h, j);
      prof_begin(c, "int16_dgrad_l", j);
      DIB_CUDA_OK(dib_int16_dgrad(c.ws + h->dg16_off[j + 1], N, c.ws + h->w16_off[j], j > 0 ? (const void*)(c.ws + h->g16_off[j]) : nullptr,
                                  K, j > 0 ? (void*)(c.ws + h->dg16_off[j]) : (void*)(c.ws + h->demb16_off), K, (int)n, K, N, h->act,
                                  h->alpha, j > 0 ? c.ws + h->dbpart_off + (long long)j * h->dbpart_layer : nullptr, bf, c.st));
      if (j > 0)   // bias gradient of layer j-1 = column sums of the gradient this dgrad just produced
        segs.push_back({c.ws + h->dbpart_off + (long long)j * h->dbpart_layer, K, row_tiles, K, 1.f / gscale, grads_flat + h->intB[j - 1]});
      prof_end(c);
    }
    std::vector<int> nsplit_of(h->Li, nsplit);
    auto in_of = [&](int j) { return j == 0 ? (const void*)(c.ws + h->emb16_off) : (const void*)(c.ws + h->g16_off[j]); };
    auto tiles_of = [&](int j) { return DIB_CEIL_DIV(int_fan_in(h, j), 128) * DIB_CEIL_DIV(int_fan_out(h, j), 128); };
    int j = h->Li - 1;
    for (; j >= 1; j -= 2) {          // layers (j, j-1) together
      long long ns = (2ll * h->num_sms) / (tiles_of(j) + tiles_of(j - 1));
      if (ns > h->part_rows) ns = h->part_rows;
      if (ns > (long long)n / 256) ns = (long long)n / 256;
      if (ns < 1) ns = 1;
      const long long rps2 = DIB_ROUND_UP(DIB_CEIL_DIV((long long)n, ns), 64);
      const int ns2 = (int)DIB_CEIL_DIV((long long)n, rps2);
      nsplit_of[j] = nsplit_of[j - 1] = ns2;
      prof_begin(c, "int16_wgrad_pair_l", j - 1);
      DIB_CUDA_OK(dib_int16_wgrad_pair(in_of(j), int_fan_in(h, j), c.ws + h->dg16_off[j + 1], int_fan_out(h, j), part + h->intW[j], ns2, (int)rps2,
                                       in_of(j - 1), int_fan_in(h, j - 1), c.ws + h->dg16_off[j], int_fan_out(h, j - 1), part + h->intW[j - 1], ns2,
                                       (int)rps2, (int)n, h->Pp, 1.f / gscale, bf, c.st));
      prof_end(c);
    }
    if (j == 0) {
      prof_begin(c, "int16_wgrad_l", 0);
      DIB_CUDA_OK(dib_int16_wgrad(in_of(0), int_fan_in(h, 0), c.ws + h->dg16_off[1], int_fan_out(h, 0), part + h->intW[0], nullptr, (int)n,
                                  int_fan_in(h, 0), int_fan_out(h, 0), nsplit, (int)rps, h->Pp, 1.f / gscale, bf, c.st));
      prof_end(c);
    }
    prof_begin(c, "int_split_reduce");
    for (int q = 0; q < h->Li; ++q)     // hidden-layer kernels: batch-split partials
      segs.push_back({part + h->intW[q], h->Pp, nsplit_of[q], (long long)int_fan_in(h, q) * int_fan_out(h, q), 1.f, grads_flat + h->intW[q]});
    segs.push_back({c.ws + h->headpart_off, h->head_stride, h->head_used, h->P - p_head, 1.f, grads_flat + p_head});
    if (!(phB && fused_enc)) {               // phase-1-only call (or unfused encoders): reduce now
      DIB_CUDA_OK(dib_launch_reduce_segments(segs.data(), (int)segs.size(), c.st));
      segs.clear();
    }
    prof_end(c);
  } else if (phA) {
    // integration network backward (GradientTape through models.py:122)
    for (int j = h->Li; j >= 0; --j) {
      prof_begin(c, "int_wgrad_l", j);
      if (gemm(c, DIB_GEMM_WGRAD, h->int_wgrad[j], 1, int_fan_out(h, j), int_fan_in(h, j), nsplit, (int)rps)) return 1;
      prof_end(c);
      prof_begin(c, "int_dgrad_l", j);
      if (gemm(c, DIB_GEMM_DGRAD, h->int_dgrad[j], 1, int_fan_in(h, j), 0, 1, 0)) return 1;
      prof_end(c);
    }
    prof_begin(c, "int_split_reduce");
    DIB_CUDA_OK(dib_launch_reduce_partials(part + p_enc, h->Pp, nsplit, h->P - p_enc, grads_flat + p_enc, c.st));
    prof_end(c);
  }
  if (!phB) return 0;

  // ---------------------------------------------------------------- phase 2: encoder backward
  if (fused_enc) {
    const int ntiles = (int)DIB_CEIL_DIV((long long)n, 128ll);
    const long long want = (long long)h->F * ntiles;
    DibEncFusedDesc d = h->fdesc;
    d.grid = (int)(want < h->num_sms ? want : h->num_sms);
    const int slots_max = DIB_CEIL_DIV(d.grid, h->F), slots_min = d.grid / h->F;
    // features served by one CTA fewer leave their last slot unwritten: zero it (ENCODER range only -- the
    // integration network's batch-split partials live in the same rows beyond p_enc)
    for (int srow = slots_min; srow < slots_max; ++srow)
      DIB_CUDA_OK(cudaMemsetAsync(part + (long long)srow * h->Pp, 0, sizeof(float) * (size_t)p_enc, c.st));
    DibEncFusedIO io;
    io.params = c.params; io.packed = c.ws + h->pack_off; io.x = x; io.ldx = h->D; io.n = n;
    io.eps = eps; io.seed = seed; io.step = step; io.step_dev = c.step_dev(); io.sample_offset = sample_offset;
    io.emb = nullptr; io.ldemb = 0; io.user_emb = nullptr; io.kl_part = nullptr; io.kl_stride = 0;
    if (!eps && dib_enc_bwd_version() >= 2) { io.eps16 = c.ws + h->eps16_off; io.a0g = c.ws + h->a0g_off; }   // written by this step's forward
    DibEncFusedBwdIO b;
    if (i16) { b.d_emb = nullptr; b.ldd = 0; b.d_emb16 = c.ws + h->demb16_off; b.ldd16 = h->F * h->E; }
    else { b.d_emb = c.ws + h->d_emb.off; b.ldd = h->d_emb.ld; }
    b.beta_dev = beta_w; b.inv_batch = inv_global_batch; b.gscale = gscale; b.part = part; b.split_stride = h->Pp;
    prof_begin(c, "enc_fused_bwd");
    DIB_CUDA_OK(dib_enc_fused_backward(d, io, b, c.st));
    prof_end(c);
    prof_begin(c, "enc_split_reduce");
    segs.push_back({part, h->Pp, slots_max, p_enc, 1.f, grads_flat});
    DIB_CUDA_OK(dib_launch_reduce_segments(segs.data(), (int)segs.size(), c.st));
    prof_end(c);
    return 0;
  }
  DibReparamArgs ra;
  ra.enc_out = c.ws + h->enc_out.off; ra.feat_stride = h->enc_out.feat_stride; ra.ldo = h->enc_out.ld;
  ra.eps = eps; ra.seed = seed; ra.step = step; ra.step_dev = c.step_dev(); ra.sample_offset = sample_offset;
  ra.F = h->F; ra.E = h->E; ra.n = n; ra.round_out = is_tc(h) ? 1 : 0;
  prof_begin(c, "reparam_kl_bwd");
  DIB_CUDA_OK(dib_launch_reparam_bwd(ra, c.ws + h->d_emb.off, h->d_emb.ld, beta_w, inv_global_batch,
                                     c.ws + h->d_out.off, c.st));
  prof_end(c);
  if (h->simple) {
    prof_begin(c, "simple_enc_wgrad");
    DIB_CUDA_OK(dib_launch_simple_enc_wgrad(x, h->D, h->d_xoff, c.ws + h->d_out.off, h->d_out.feat_stride, h->d_out.ld, h->F, h->E,
                                            n, nsplit, (int)rps, part, h->Pp, c.st));
    prof_end(c);
  }
  for (int j = h->L; j >= 0 && !h->simple; --j) {
    prof_begin(c, "enc_wgrad_l", j);
    if (gemm(c, DIB_GEMM_WGRAD, h->enc_wgrad[j], h->F, enc_fan_out(h, j), h->enc_maxK[j], nsplit, (int)rps)) return 1;
    prof_end(c);
    if (j >= 1) {
      prof_begin(c, "enc_dgrad_l", j);
      if (gemm(c, DIB_GEMM_DGRAD, h->enc_dgrad[j], h->F, h->enc_arch[j - 1], 0, 1, 0)) return 1;
      if (h->drop > 0.f)                   // Dropout backward: the same keep mask, scaled
        DIB_CUDA_OK(dib_launch_dropout(nullptr, c.ws + h->d_enc[j].off, h->d_enc[j].feat_stride, h->d_enc[j].ld, h->enc_arch[j - 1],
                                       h->F, n, h->drop, seed, step, c.step_dev(), sample_offset, j, -1, 1, is_tc(h) ? 1 : 0, c.st));
      prof_end(c);
    }
  }
  prof_begin(c, "enc_split_reduce");
  DIB_CUDA_OK(dib_launch_reduce_partials(part, h->Pp, nsplit, p_enc, grads_flat, c.st));
  prof_end(c);
  return 0;
}

}  // namespace

extern "C" {

int dib_train_step_phased(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                          float inv_global_batch, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                          float* grads_flat, float* out_stats, void* workspace, int32_t phases, void* stream) {
  if (check_call(h, params, x, n, workspace)) return 1;
  if (h->loss == DIB_LOSS_INFONCE)
    return fail("dib_train_step: a DIB_LOSS_INFONCE handle trains with dib_infonce_train_step (the step needs the output encoder)");
  if ((!y && n > 0) || !beta_dev || !grads_flat || !out_stats)
    return fail("dib_train_step: y, beta_dev, grads_flat and out_stats are required");
  if (phases < 1 || phases > 3) return fail("dib_train_step_phased: phases must be 1, 2 or 3");
  const bool phA = (phases & 1) != 0, phB = (phases & 2) != 0;
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  c.dev_step = true;
  const long long p_enc = h->intW[0];                // encoder parameters occupy [0, p_enc)
  if (n == 0) {
    if (phB) DIB_CUDA_OK(cudaMemsetAsync(grads_flat, 0, sizeof(float) * p_enc, c.st));
    if (phA) {
      DIB_CUDA_OK(cudaMemsetAsync(grads_flat + p_enc, 0, sizeof(float) * (h->P - p_enc), c.st));
      DIB_CUDA_OK(cudaMemsetAsync(out_stats, 0, sizeof(float) * (h->F + 3), c.st));
    }
    return 0;
  }
  return train_phases(c, x, y, n, beta_dev, inv_global_batch, eps, seed, step, sample_offset, grads_flat, out_stats, phases,
                      false);
}

int dib_train_step(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                   float inv_global_batch, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                   float* grads_flat, float* out_stats, void* workspace, void* stream) {
  return dib_train_step_phased(h, params, x, y, n, beta_dev, inv_global_batch, eps, seed, step, sample_offset, grads_flat,
                               out_stats, workspace, 3, stream);
}

// Philox 'step' word from device memory (CUDA-Graph replay: a captured launch cannot carry a fresh by-value step):
// when set, every forward / train-step call uses step + *step_dev.  The caller owns and advances the counter.
int dib_set_noise_step_device(dib_model* h, const uint32_t* step_dev) {
  if (!h) return fail("null model handle");
  h->step_dev = step_dev;
  return 0;
}

int dib_adam_step(float* params, const float* grads, float* m, float* v, int64_t count, const float* lr_dev,
                  int32_t* step_dev, float beta_1, float beta_2, float epsilon, void* stream) {
  if (!params || !grads || !m || !v || !lr_dev || !step_dev) return fail("dib_adam_step: null pointer");
  if (count < 0) return fail("dib_adam_step: negative count");
  DIB_CUDA_OK(dib_launch_adam(params, grads, m, v, count, lr_dev, step_dev, beta_1, beta_2, epsilon,
                              static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_optimizer_step(int32_t kind, float* params, const float* grads, float* slot1, float* slot2, int64_t count,
                       const float* lr_dev, int32_t* step_dev, float hyper0, float hyper1, float hyper2, void* stream) {
  if (kind < 0 || kind > 1 || !params || !grads || !lr_dev || !step_dev || count < 0 || (kind == 1 && (!slot1 || !slot2)) ||
      (kind == 0 && hyper0 != 0.f && !slot1))
    return fail("dib_optimizer_step: bad arguments");
  DIB_CUDA_OK(dib_launch_optimizer(kind, params, grads, slot1, slot2, count, lr_dev, step_dev, hyper0, hyper1, hyper2,
                                   static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_integration_forward(dib_model* h, const float* params, const float* emb, int64_t n, float* out_pred,
                            void* workspace, void* stream) {
  if (check_call(h, params, emb, n, workspace)) return 1;
  if (!out_pred) return fail("dib_integration_forward: null output");
  if (n == 0) return 0;
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  const int FE = h->F * h->E;
  if (is_tc(h)) DIB_CUDA_OK(dib_launch_round_copy(c.params, c.ws + h->wshadow_off, h->P, c.st));
  DIB_CUDA_OK(dib_launch_copy2d(emb, FE, c.ws + h->emb.off, h->emb.ld, FE, n, c.st));
  if (h->emb.ld > FE)          // zero the padded operand columns
    DIB_CUDA_OK(cudaMemset2DAsync(c.ws + h->emb.off + FE, sizeof(float) * h->emb.ld, 0, sizeof(float) * (h->emb.ld - FE), (size_t)n, c.st));
  for (int j = 0; j <= h->Li; ++j)
    if (gemm(c, DIB_GEMM_FWD, h->int_fwd[j], 1, int_fan_out(h, j), 0, 1, 0)) return 1;
  DIB_CUDA_OK(dib_launch_copy2d(c.ws + h->pred.off, h->pred.ld, out_pred, h->out, h->out, n, c.st));
  return 0;
}

int dib_positional_encoding(const float* x, int64_t n, int32_t d, int32_t number_frequencies, float* out, void* stream) {
  if ((!x || !out) && n > 0) return fail("dib_positional_encoding: null pointer");
  if (n < 0 || d < 1 || number_frequencies < 1 || number_frequencies > 31) return fail("dib_positional_encoding: bad sizes");
  DIB_CUDA_OK(dib_launch_pe_plain(x, n, d, number_frequencies, out, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_metrics_update_ex(const float* stats, const float* beta_dev, float* acc, int32_t number_features,
                          float kl_loss_exponent, float kl_loss_scale, void* stream) {
  if (!stats || !beta_dev || !acc || number_features < 1) return fail("dib_metrics_update: bad arguments");
  DIB_CUDA_OK(dib_launch_metrics_update(stats, beta_dev, acc, number_features, kl_loss_exponent == 0.f ? 1.f : kl_loss_exponent,
                                        kl_loss_scale == 0.f ? 1.f : kl_loss_scale, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_metrics_update(const float* stats, const float* beta_dev, float* acc, int32_t number_features, void* stream) {
  return dib_metrics_update_ex(stats, beta_dev, acc, number_features, 1.f, 1.f, stream);
}

int dib_encoders_forward(dib_model* h, const float* params, const float* x, int64_t n, const float* eps, uint64_t seed,
                         uint32_t step, uint64_t sample_offset, float* out_emb, float* out_stats, void* workspace, void* stream) {
  if (check_call(h, params, x, n, workspace)) return 1;
  if (!out_emb || !out_stats) return fail("dib_encoders_forward: out_emb and out_stats are required");
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  if (n == 0) { DIB_CUDA_OK(cudaMemsetAsync(out_stats, 0, sizeof(float) * (h->F + 3), c.st)); return 0; }
  return run_forward(c, x, nullptr, eps, seed, step, sample_offset, 0.f, false, nullptr, out_emb, out_stats, true);
}

int dib_encoders_backward(dib_model* h, const float* params, const float* x, const float* d_emb, int64_t n,
                          const float* beta_dev, float inv_global_batch, const float* eps, uint64_t seed, uint32_t step,
                          uint64_t sample_offset, float* grads_flat, float* out_stats, void* workspace, void* stream) {
  if (check_call(h, params, x, n, workspace)) return 1;
  if ((!d_emb && n > 0) || !beta_dev || !grads_flat || !out_stats)
    return fail("dib_encoders_backward: d_emb, beta_dev, grads_flat and out_stats are required");
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  DIB_CUDA_OK(cudaMemsetAsync(grads_flat, 0, sizeof(float) * h->P, c.st));
  if (n == 0) { DIB_CUDA_OK(cudaMemsetAsync(out_stats, 0, sizeof(float) * (h->F + 3), c.st)); return 0; }
  // the forward is recomputed here (training mode keeps what the backward needs); user_emb is not needed again
  if (run_forward(c, x, nullptr, eps, seed, step, sample_offset, inv_global_batch, true, nullptr, nullptr, out_stats, true)) return 1;
  const float* bw = beta_dev;
  if (ib_weight(c, beta_dev, out_stats, inv_global_batch, &bw)) return 1;
  long long rps = DIB_CEIL_DIV((long long)n, (long long)kMaxSplits);
  if (rps < 256) rps = 256;
  rps = DIB_ROUND_UP(rps, 64);      // whole k-blocks of every WGRAD kernel (32 rows for the TF32 ones, 64 for the 16-bit ones)
  const int nsplit = (int)DIB_CEIL_DIV((long long)n, rps);
  const long long p_enc = h->intW[0];
  const int FE = h->F * h->E;
  const bool fused = h->fused_ok && h->fused_bwd_ok && !h->force_unfused;
  float* part = c.ws + h->part_off;
  if (fused) {
    const int ntiles = (int)DIB_CEIL_DIV((long long)n, 128ll);
    const long long want = (long long)h->F * ntiles;
    DibEncFusedDesc d = h->fdesc;
    d.logvar_offset = h->lv_off;
    d.grid = (int)(want < h->num_sms ? want : h->num_sms);
    const int slots_max = DIB_CEIL_DIV(d.grid, h->F), slots_min = d.grid / h->F;
    for (int srow = slots_min; srow < slots_max; ++srow)
      DIB_CUDA_OK(cudaMemsetAsync(part + (long long)srow * h->Pp, 0, sizeof(float) * (size_t)p_enc, c.st));
    DibEncFusedIO io;
    io.params = c.params; io.packed = c.ws + h->pack_off; io.x = x; io.ldx = h->D; io.n = n;
    io.eps = eps; io.seed = seed; io.step = step; io.step_dev = c.step_dev(); io.sample_offset = sample_offset;
    io.emb = nullptr; io.ldemb = 0; io.user_emb = nullptr; io.kl_part = nullptr; io.kl_stride = 0;
    if (!eps && dib_enc_bwd_version() >= 2) { io.eps16 = c.ws + h->eps16_off; io.a0g = c.ws + h->a0g_off; }   // written by this step's forward
    DibEncFusedBwdIO b;
    b.d_emb = d_emb; b.ldd = FE; b.beta_dev = bw; b.inv_batch = inv_global_batch;
    b.gscale = exp2f(ceilf(log2f(1.f / inv_global_batch)));
    b.part = part; b.split_stride = h->Pp;
    DIB_CUDA_OK(dib_enc_fused_backward(d, io, b, c.st));
    DIB_CUDA_OK(dib_launch_reduce_partials(part, h->Pp, slots_max, p_enc, grads_flat, c.st));
    return 0;
  }
  DibReparamArgs ra;
  ra.enc_out = c.ws + h->enc_out.off; ra.feat_stride = h->enc_out.feat_stride; ra.ldo = h->enc_out.ld;
  ra.eps = eps; ra.seed = seed; ra.step = step; ra.step_dev = c.step_dev(); ra.sample_offset = sample_offset;
  ra.F = h->F; ra.E = h->E; ra.n = n; ra.round_out = is_tc(h) ? 1 : 0;
  DIB_CUDA_OK(dib_launch_reparam_bwd(ra, d_emb, FE, bw, inv_global_batch, c.ws + h->d_out.off, c.st));
  if (h->simple) {
    DIB_CUDA_OK(dib_launch_simple_enc_wgrad(x, h->D, h->d_xoff, c.ws + h->d_out.off, h->d_out.feat_stride, h->d_out.ld, h->F, h->E,
                                            n, nsplit, (int)rps, part, h->Pp, c.st));
  } else {
    for (int j = h->L; j >= 0; --j) {
      if (gemm(c, DIB_GEMM_WGRAD, h->enc_wgrad[j], h->F, enc_fan_out(h, j), h->enc_maxK[j], nsplit, (int)rps)) return 1;
      if (j >= 1 && gemm(c, DIB_GEMM_DGRAD, h->enc_dgrad[j], h->F, h->enc_arch[j - 1], 0, 1, 0)) return 1;
      if (j >= 1 && h->drop > 0.f)
        DIB_CUDA_OK(dib_launch_dropout(nullptr, c.ws + h->d_enc[j].off, h->d_enc[j].feat_stride, h->d_enc[j].ld, h->enc_arch[j - 1],
                                       h->F, n, h->drop, seed, step, c.step_dev(), sample_offset, j, -1, 1, is_tc(h) ? 1 : 0, c.st));
    }
  }
  DIB_CUDA_OK(dib_launch_reduce_partials(part, h->Pp, nsplit, p_enc, grads_flat, c.st));
  return 0;
}

int dib_mi_sandwich_bounds(const float* mu_logvar, int64_t n, int32_t embedding_dimension, const float* eps, uint64_t seed,
                           uint32_t step, float* row_scratch, float* out_lower_upper, void* stream) {
  if (!mu_logvar || !row_scratch || !out_lower_upper || n < 1 || n > 0x7fffffffll || embedding_dimension < 1)
    return fail("dib_mi_sandwich_bounds: bad arguments");
  DIB_CUDA_OK(dib_launch_mi_sandwich(mu_logvar, n, embedding_dimension, eps, seed, step, row_scratch, out_lower_upper,
                                     static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_mi_sandwich_bounds_batched(const float* mu_logvar, int32_t groups, int64_t n, int32_t embedding_dimension, const float* eps,
                                   uint64_t seed, int32_t batches_per_feature, double* row_scratch, double* out_lower_upper,
                                   void* stream) {
  if (!mu_logvar || !row_scratch || !out_lower_upper || groups < 1 || groups > 65535 || n < 1 || n > 0x7fffffffll ||
      embedding_dimension < 1 || embedding_dimension > 64 || batches_per_feature < 1)
    return fail("dib_mi_sandwich_bounds_batched: bad arguments (1 <= groups <= 65535, 1 <= E <= 64)");
  DIB_CUDA_OK(dib_launch_mi_sandwich_batched(mu_logvar, groups, n, embedding_dimension, eps, seed, batches_per_feature,
                                             row_scratch, out_lower_upper, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_bhattacharyya(const float* mu_logvar, int64_t n, int32_t embedding_dimension, float* out_dist,
                      float* out_compression, void* stream) {
  if (!mu_logvar || n < 0 || embedding_dimension < 1) return fail("dib_bhattacharyya: bad arguments");
  const int64_t ld = 2 * (int64_t)embedding_dimension;
  DIB_CUDA_OK(dib_launch_pairwise_gauss(0, mu_logvar, ld, 0, n, mu_logvar, ld, 0, n, embedding_dimension, 1, out_dist,
                                        out_compression, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_pairwise_gaussian(int32_t kind, const float* mu_logvar_1, int64_t n, const float* mu_logvar_2, int64_t m,
                          int32_t embedding_dimension, float* out, float* out_exp_neg, void* stream) {
  if ((kind != 0 && kind != 1) || n < 0 || m < 0 || embedding_dimension < 1 ||
      ((!mu_logvar_1 || !mu_logvar_2) && n > 0 && m > 0))
    return fail("dib_pairwise_gaussian: bad arguments");
  const int64_t ld = 2 * (int64_t)embedding_dimension;
  DIB_CUDA_OK(dib_launch_pairwise_gauss(kind, mu_logvar_1, ld, 0, n, mu_logvar_2, ld, 0, m, embedding_dimension, 1, out,
                                        out_exp_neg, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_scaled_similarity(int32_t kind, const float* e1, int64_t n, const float* e2, int64_t m, int32_t d, float temperature,
                          float* out, void* stream) {
  if (kind < 0 || kind > 4 || n < 0 || m < 0 || d < 1 || !(temperature > 0.f) || ((!e1 || !e2 || !out) && n > 0 && m > 0))
    return fail("dib_scaled_similarity: bad arguments");
  DIB_CUDA_OK(dib_launch_similarity(kind, e1, n, e2, m, d, temperature, out, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_infonce_head(int32_t kind, const float* e1, const float* e2, int64_t n, int32_t d, float temperature, float* scratch,
                     float* out_loss, float* d_e1, float* d_e2, void* stream) {
  if (kind < 0 || kind > 4 || n < 1 || n > 32768 || d < 1 || d > 512 || !(temperature > 0.f) || !e1 || !e2 || !scratch ||
      !out_loss)
    return fail("dib_infonce_head: bad arguments (1 <= n <= 32768, 1 <= d <= 512, temperature > 0)");
  DIB_CUDA_OK(dib_launch_infonce_head(kind, e1, e2, n, d, temperature, scratch, out_loss, d_e1, d_e2,
                                      static_cast<cudaStream_t>(stream)));
  return 0;
}

int64_t dib_infonce_head_tc_scratch_bytes(int64_t n, int32_t d) {
  if (n < 1 || n > (1 << 26) || d < 1 || d > 256) return -1;
  return (int64_t)dib_infonce_head_tc_scratch(n, d);
}

int dib_infonce_head_tc(int32_t kind, const float* e1, const float* e2, int64_t n, int32_t d, float temperature, void* scratch,
                        float* out_loss, float* d_e1, float* d_e2, void* stream) {
  if ((kind != 0 && kind != 1 && kind != 4) || n < 1 || n > (1 << 26) || d < 1 || d > 256 || !(temperature > 0.f) || !e1 ||
      !e2 || !scratch || !out_loss)
    return fail("dib_infonce_head_tc: bad arguments (kind l2sq/l2/cosine, 1 <= n <= 2^26, 1 <= d <= 256, temperature > 0)");
  if (reinterpret_cast<uintptr_t>(scratch) % 128)
    return fail("dib_infonce_head_tc: scratch must be 128-byte aligned");
  if (!dib_infonce_head_tc_available()) return fail("dib_infonce_head_tc: cuTensorMapEncodeTiled is not available");
  DIB_CUDA_OK(dib_launch_infonce_head_tc(kind, e1, e2, n, d, temperature, scratch, out_loss, d_e1, d_e2,
                                         static_cast<cudaStream_t>(stream)));
  return 0;
}

int dib_compression_matrices(dib_model* h, const float* params, const float* x, int64_t n_total, const int32_t* row_index,
                             int64_t n, float* out_mu_logvar, float* out_dist, float* out_compression, void* workspace,
                             void* stream) {
  if (check_call(h, params, x, n, workspace)) return 1;
  if (n_total < 0 || (!row_index && n > n_total) || (row_index && n > 0 && n_total < 1))
    return fail("dib_compression_matrices: rows out of range");
  if (n == 0) return 0;
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  const int rnd = is_tc(h) ? 1 : 0;
  if (rnd) DIB_CUDA_OK(dib_launch_round_copy(c.params, c.ws + h->wshadow_off, h->P, c.st));
  // all F encoders as ONE grouped problem per layer (the reference loops over features in Python, visualization.py:14-35)
  if (encode_all(c, x, h->D, rnd, row_index, n_total)) return 1;
  const float* eo = c.ws + h->enc_out.off;
  if (out_mu_logvar)
    for (int f = 0; f < h->F; ++f)
      DIB_CUDA_OK(dib_launch_copy2d(eo + f * h->enc_out.feat_stride, h->enc_out.ld, out_mu_logvar + (int64_t)f * n * 2 * h->E,
                                    2 * h->E, 2 * h->E, n, c.st));
  if (out_dist || out_compression)
    DIB_CUDA_OK(dib_launch_pairwise_gauss(0, eo, h->enc_out.ld, h->enc_out.feat_stride, n, eo, h->enc_out.ld,
                                          h->enc_out.feat_stride, n, h->E, h->F, out_dist, out_compression, c.st));
  return 0;
}

// ---- InfoNCE training (train.py:180-289) ------------------------------------------------------------------------------
int dib_attach_output_encoder(dib_model* h, const dib_output_encoder_config* cfg) {
  if (!h || !cfg) return fail("dib_attach_output_encoder: null argument");
  if (h->loss != DIB_LOSS_INFONCE) return fail("dib_attach_output_encoder: the handle was not created with DIB_LOSS_INFONCE");
  if (h->oe) return fail("dib_attach_output_encoder: an output encoder is already attached");
  if (cfg->input_dimensionality < 1 || cfg->number_layers < 0 || cfg->number_layers > kDibMaxOeLayers ||
      (cfg->number_layers > 0 && !cfg->architecture))
    return fail("dib_attach_output_encoder: bad sizes (input_dimensionality >= 1, 0 <= number_layers <= " +
                std::to_string(kDibMaxOeLayers) + ")");
  for (int j = 0; j < cfg->number_layers; ++j)
    if (cfg->architecture[j] < 1) return fail("dib_attach_output_encoder: width < 1");
  h->oe_dy = cfg->input_dimensionality;
  h->oe_L = cfg->number_layers;
  h->oe_arch.assign(cfg->architecture, cfg->architecture + h->oe_L);
  // PE of y with the model's frequencies (train.py:187-189), columns padded to a multiple of 4
  std::vector<int> col_src, col_freq;
  for (int blk = 0; blk < h->nfreq; ++blk)
    for (int k = 0; k < h->oe_dy; ++k) { col_src.push_back(k); col_freq.push_back(blk == 0 ? 0 : (1 << blk)); }
  while (col_src.size() % 4) { col_src.push_back(-1); col_freq.push_back(0); }
  h->oe_ldpe = (int)col_src.size();
  // Keras-ordered parameters and their aligned shadow: kernels first (one TF32 rounding range), then biases
  h->oe_var_off.clear(); h->oe_var_rows.clear(); h->oe_var_cols.clear();
  h->oeW.assign(h->oe_L + 1, 0); h->oeB.assign(h->oe_L + 1, 0);
  long long off = 0, sh = 0;
  for (int j = 0; j <= h->oe_L; ++j) {
    const long long fi = oe_fan_in(h, j), fo = oe_fan_out(h, j);
    h->oe_var_off.push_back(off); h->oe_var_rows.push_back((int)fi); h->oe_var_cols.push_back((int)fo); off += fi * fo;
    h->oe_var_off.push_back(off); h->oe_var_rows.push_back(0); h->oe_var_cols.push_back((int)fo); off += fo;
    h->oeW[j] = sh; sh += DIB_ROUND_UP(fi * fo, 4ll);
  }
  h->oe_wlen = sh;
  for (int j = 0; j <= h->oe_L; ++j) { h->oeB[j] = sh; sh += DIB_ROUND_UP((long long)oe_fan_out(h, j), 4ll); }
  h->Q = off; h->oe_shadow_len = sh; h->oe_part_stride = DIB_ROUND_UP(sh, 64ll);
  DibOePackTable& t = h->oe_pack;
  t.nvar = 2 * (h->oe_L + 1);
  for (int j = 0; j <= h->oe_L; ++j) {
    t.src_off[2 * j] = h->oe_var_off[2 * j]; t.dst_off[2 * j] = h->oeW[j];
    t.count[2 * j] = (long long)oe_fan_in(h, j) * oe_fan_out(h, j); t.round[2 * j] = is_tc(h) ? 1 : 0;
    t.src_off[2 * j + 1] = h->oe_var_off[2 * j + 1]; t.dst_off[2 * j + 1] = h->oeB[j];
    t.count[2 * j + 1] = oe_fan_out(h, j); t.round[2 * j + 1] = 0;
  }
  // the workspace plan and the GEMM problem table grow by the encoder's buffers and problems
  h->oe = true;
  plan(h);
  std::vector<DibGemmProblem> probs;
  build_problems(h, probs);
  h->h_probs = probs;
  DibGemmProblem* dp = nullptr;
  cudaError_t e = cudaMalloc(&dp, probs.size() * sizeof(DibGemmProblem));
  if (e == cudaSuccess) e = cudaMemcpy(dp, probs.data(), probs.size() * sizeof(DibGemmProblem), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_oe_col_src, col_src.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_oe_col_freq, col_freq.size() * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_oe_col_src, col_src.data(), col_src.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_oe_col_freq, col_freq.data(), col_freq.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (dp) cudaFree(dp);
    return fail(std::string("dib_attach_output_encoder: CUDA error: ") + cudaGetErrorString(e));
  }
  cudaFree(h->d_probs);
  h->d_probs = dp;
  return 0;
}

int64_t dib_output_encoder_param_count(const dib_model* h) { return h && h->oe ? h->Q : -1; }

int dib_output_encoder_param_layout(const dib_model* h, int64_t* offsets, int32_t* rows, int32_t* cols, int32_t capacity) {
  if (!h || !h->oe) { fail("dib_output_encoder_param_layout: no output encoder attached"); return -1; }
  const int nv = (int)h->oe_var_off.size();
  if (!offsets || !rows || !cols) return nv;
  if (capacity < nv) { fail("dib_output_encoder_param_layout: capacity too small"); return -1; }
  for (int i = 0; i < nv; ++i) { offsets[i] = h->P + h->oe_var_off[i]; rows[i] = h->oe_var_rows[i]; cols[i] = h->oe_var_cols[i]; }
  return nv;
}

int dib_output_encoder_forward(dib_model* h, const float* params, const float* y, int64_t n, float* out_e2, void* workspace,
                               void* stream) {
  if (check_call(h, params, y, n, workspace)) return 1;
  if (!h->oe) return fail("dib_output_encoder_forward: no output encoder attached (dib_attach_output_encoder)");
  if (!out_e2) return fail("dib_output_encoder_forward: null output");
  if (n == 0) return 0;
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  if (oe_forward(c, y)) return 1;
  DIB_CUDA_OK(dib_launch_copy2d(c.ws + h->oe_out.off, h->oe_out.ld, out_e2, h->out, h->out, n, c.st));
  return 0;
}

int64_t dib_infonce_scratch_bytes(int32_t kind, int64_t n, int32_t d) {
  if (kind == 0 || kind == 1 || kind == 4) return dib_infonce_head_tc_scratch_bytes(n, d);
  if ((kind != 2 && kind != 3) || n < 1 || n > 32768 || d < 1 || d > 512) return -1;
  return (n * n + 4 * n) * (int64_t)sizeof(float);
}

}  // extern "C"

namespace {

// dib_infonce_train_step (training) / dib_infonce_forward: model forward to e1 -> output encoder -> head -> external-loss
// branch with y := d e1 -> [phased backward of the model -> output-encoder backward]
int infonce_call(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev, int32_t kind,
                 float temperature, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset, void* head_scratch,
                 float* grads_flat, float* out_stats, void* workspace, void* stream, bool training) {
  const char* who = training ? "dib_infonce_train_step" : "dib_infonce_forward";
  if (check_call(h, params, x, n, workspace)) return 1;
  if (h->loss != DIB_LOSS_INFONCE || !h->oe)
    return fail(std::string(who) + ": needs a DIB_LOSS_INFONCE handle with an attached output encoder");
  if (!y || !beta_dev || !out_stats || !head_scratch || (training && !grads_flat))
    return fail(std::string(who) + ": y, beta_dev, head_scratch, out_stats" + (training ? " and grads_flat" : "") + " are required");
  if (n < 1) return fail(std::string(who) + ": the InfoNCE loss needs n >= 1 rows");
  if (!(temperature > 0.f)) return fail(std::string(who) + ": temperature must be > 0");
  const int D = h->out;
  const bool gram = kind == 0 || kind == 1 || kind == 4;
  if (gram) {
    if (D > 256) return fail(std::string(who) + ": l2sq / l2 / cosine need output_dimensionality <= 256, got " + std::to_string(D));
    if (reinterpret_cast<uintptr_t>(head_scratch) % 128) return fail(std::string(who) + ": head_scratch must be 128-byte aligned");
    if (!dib_infonce_head_tc_available()) return fail(std::string(who) + ": cuTensorMapEncodeTiled is not available");
  } else if (kind == 2 || kind == 3) {
    if (n > 32768) return fail(std::string(who) + ": l1 / linf run the exact head, which holds n x n similarities: n <= 32768, got " +
                               std::to_string(n));
    if (D > 512) return fail(std::string(who) + ": l1 / linf need output_dimensionality <= 512");
  } else {
    return fail(std::string(who) + ": unknown similarity kind " + std::to_string(kind));
  }
  Ctx c{h, params, static_cast<float*>(workspace), static_cast<cudaStream_t>(stream), (int)n};
  c.dev_step = training;
  const float inv_batch = 1.f / (float)n;
  int nblk_kl = 0;
  if (run_forward(c, x, nullptr, eps, seed, step, sample_offset, inv_batch, training, nullptr, nullptr, out_stats, false, &nblk_kl))
    return 1;
  if (oe_forward(c, y)) return 1;
  // the heads take unpadded [n, D] rows
  float* cont = c.ws + h->oe_cont_off;
  const long long nD = (long long)h->maxB * D;
  float *e1 = c.ws + h->pred.off, *e2 = c.ws + h->oe_out.off, *de1 = cont + 2 * nD;
  float* de2 = training ? c.ws + h->oe_dout.off : nullptr;
  const bool padded = h->pred.ld != D;
  if (padded) {
    DIB_CUDA_OK(dib_launch_copy2d(e1, h->pred.ld, cont, D, D, n, c.st));
    DIB_CUDA_OK(dib_launch_copy2d(e2, h->oe_out.ld, cont + nD, D, D, n, c.st));
    e1 = cont; e2 = cont + nD;
    if (training) de2 = cont + 3 * nD;
  }
  float* loss_dev = c.ws + h->nce_loss_off;
  prof_begin(c, "infonce_head");
  if (gram)
    DIB_CUDA_OK(dib_launch_infonce_head_tc(kind, e1, e2, n, D, temperature, head_scratch, loss_dev, training ? de1 : nullptr, de2,
                                           c.st));
  else
    DIB_CUDA_OK(dib_launch_infonce_head(kind, e1, e2, n, D, temperature, static_cast<float*>(head_scratch), loss_dev,
                                        training ? de1 : nullptr, de2, c.st));
  prof_end(c);
  // d e2 into the output encoder's backward operand: rounded like d e1 (loss kernel) in the tensor-core modes, pads zeroed
  if (training && (padded || is_tc(h)))
    DIB_CUDA_OK(dib_launch_grad_handoff(de2, padded ? D : h->oe_dout.ld, c.ws + h->oe_dout.off, h->oe_dout.ld, D, n,
                                        is_tc(h) ? 1 : 0, c.st));
  if (loss_and_stats(c, training ? de1 : nullptr, inv_batch, training, nullptr, out_stats, nblk_kl)) return 1;
  DIB_CUDA_OK(dib_launch_infonce_stats(loss_dev, n, out_stats + h->F, c.st));
  if (!training) return 0;
  if (train_phases(c, x, de1, n, beta_dev, inv_batch, eps, seed, step, sample_offset, grads_flat, out_stats, 3, true)) return 1;
  long long rps = DIB_CEIL_DIV((long long)n, (long long)kMaxSplits);
  if (rps < 256) rps = 256;
  rps = DIB_ROUND_UP(rps, 64);
  return oe_backward(c, (int)DIB_CEIL_DIV((long long)n, rps), (int)rps, grads_flat + h->P);
}

}  // namespace

extern "C" {

int dib_infonce_train_step(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                           int32_t kind, float temperature, const float* eps, uint64_t seed, uint32_t step,
                           uint64_t sample_offset, void* head_scratch, float* grads_flat, float* out_stats, void* workspace,
                           void* stream) {
  return infonce_call(h, params, x, y, n, beta_dev, kind, temperature, eps, seed, step, sample_offset, head_scratch, grads_flat,
                      out_stats, workspace, stream, true);
}

int dib_infonce_forward(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                        int32_t kind, float temperature, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                        void* head_scratch, float* out_stats, void* workspace, void* stream) {
  return infonce_call(h, params, x, y, n, beta_dev, kind, temperature, eps, seed, step, sample_offset, head_scratch, nullptr,
                      out_stats, workspace, stream, false);
}

}  // extern "C"
