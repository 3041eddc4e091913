/* dib_b200.h -- C ABI of the B200-native Distributed-IB training engine.
 *
 * The reference (distributed-information-bottleneck.github.io) has no FFI/plugin interface: its
 * hot path is a tf.keras Model whose arithmetic executes inside TensorFlow.  Each entry point
 * below therefore names the reference *Python* interface it replaces (paths relative to the
 * reference root).  The PyTorch host shim (package dib_b200) binds these with ctypes and
 * reproduces the DistributedIBNet / compile / fit / callback surface on top of them;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer named *_dev / params / grads / x / y / eps / workspace is DEVICE memory owned by
 *     the caller (PyTorch tensors in the shim); the library never allocates user-visible memory.
 *     The only allocation it makes is a few KB of layer-descriptor tables inside dib_create.
 *   - every compute call is asynchronous on the caller's cudaStream_t (passed as void*), performs no
 *     host synchronisation and no allocation, and is CUDA-Graph capturable: beta, learning rate and
 *     the Adam step counter are read from device scalars.
 *   - return value: 0 = ok, non-zero = error (see dib_last_error()); no C++ exception crosses.
 *   - a handle is not thread-safe; use one host thread per handle (the reference is single-threaded).
 *   - all tensors are fp32, row-major.  Parameters live in ONE flat fp32 buffer; per feature
 *     (W1,b1,W2,b2,...,W_out,b_out) then the integration layers, kernels in Keras [in,out]
 *     orientation (tf.keras.layers.Dense, models.py:76-77,82-83).
 *   - sums, not means: statistics are returned as SUMS over the local samples so that data-parallel
 *     ranks combine them (and the gradients) with one all-reduce(sum); gradients are already scaled
 *     by inv_global_batch.
 */
#ifndef DIB_B200_H_
#define DIB_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIB_ABI_VERSION 2

/* activation_fn strings accepted by tf.keras.layers.Dense in the reference's call sites
 * (train.py:37 'relu', nb-radial 'tanh', nb-bool LeakyReLU, None). */
enum dib_activation {
  DIB_ACT_LINEAR = 0, DIB_ACT_RELU = 1, DIB_ACT_TANH = 2, DIB_ACT_LEAKY_RELU = 3,
  DIB_ACT_SIGMOID = 4, DIB_ACT_ELU = 5
};

/* compiled losses used by the reference's datasets (data.py:65, data.py:343, data.py:129). */
enum dib_loss {
  DIB_LOSS_BCE_LOGITS = 0,       /* tf.keras.losses.BinaryCrossentropy(from_logits=True)            */
  DIB_LOSS_SPARSE_CE_LOGITS = 1, /* tf.keras.losses.SparseCategoricalCrossentropy(from_logits=True) */
  DIB_LOSS_MSE = 2,
  /* NEXT ROW f3 -- custom training steps (GradientTape loops: train.py:201-220 InfoNCE, nb-bool cell 6, nb-particle
   * cell 7): the CALLER owns the task loss.  dib_forward returns the predictions; in dib_train_step the `y` argument
   * is reinterpreted as d(task loss)/d(predictions) [n, out], already carrying the caller's batch-mean scaling (it is
   * NOT multiplied by inv_global_batch; the beta*KL term still is).  Task-loss and accuracy statistics are 0. */
  DIB_LOSS_EXTERNAL = 3,
  /* tf.keras.losses.BinaryCrossentropy() on PROBABILITIES (from_logits=False, the Keras default; use with
   * output_activation_fn = sigmoid): -[y log(p~ + eps) + (1-y) log(1 - p~ + eps)], p~ = clip(p, eps, 1-eps), eps = 1e-7
   * (keras.backend.binary_crossentropy); the gradient is zero where p is clipped. */
  DIB_LOSS_BCE_PROBS = 4,
  /* the InfoNCE training path of train.py:180-289: the model output is the x-side embedding e1 (output_activation_fn must
   * be linear; dib_forward with y = NULL returns e1).  A trainable output encoder (dib_attach_output_encoder) maps y to e2
   * and dib_infonce_train_step trains both against the symmetric InfoNCE loss + beta * sum_i KL_i; dib_train_step refuses
   * such a handle. */
  DIB_LOSS_INFONCE = 5
};

/* arithmetic of the dense contractions; everything else (PE, exp, KL, loss, Adam, reductions) is fp32 in every mode
 * and all tensor-core modes accumulate in fp32 (TMEM).
 *   FP32: CUDA-core FMA -- the exact parity path (the reference's tf.keras fp32 graph on a CPU).
 *   TF32: tcgen05.mma kind::tf32 on fp32 storage (10-bit mantissa, 8-bit exponent operands, rounded not truncated):
 *         what stock TensorFlow does to an fp32 model on a tensor-core GPU.  Unfused grouped GEMMs.
 *   FP16: tcgen05.mma kind::f16 on fp16 operands (10-bit mantissa like TF32 but a 5-bit exponent: |value| <= 65504,
 *         saturating conversions, gradients carried under a power-of-two loss scale) -- the fused per-feature encoder
 *         kernels and the 16-bit integration path; shapes outside their envelope run on the TF32 kernels.
 *   BF16: the same fused kernels on bf16 operands (7-bit mantissa, fp32's exponent range).
 * dib_model_info() reports which kernel family a handle actually selected. */
enum dib_precision { DIB_PREC_FP32 = 0, DIB_PREC_TF32 = 1, DIB_PREC_BF16 = 2, DIB_PREC_FP16 = 3 };

/* feature encoders: the per-feature MLP of models.py:72-78, or nb-bool cell 4's SimpleEncoder -- two trainable (1,1)
 * constants per feature, output concat([x * mu_scaling, ones_like(x) * logvar]) (needs d_i == E, no positional encoding;
 * flat parameter order per feature: mu_scaling, logvar; feature_encoder_architecture is ignored). */
enum dib_encoder_kind { DIB_ENCODER_MLP = 0, DIB_ENCODER_SIMPLE = 1 };

/* Mirrors the constructor of models.DistributedIBNet (models.py:56-66). */
typedef struct dib_config {
  int32_t abi_version;               /* DIB_ABI_VERSION */
  int32_t number_features;           /* len(feature_dimensionalities)            models.py:69 */
  const int32_t* feature_dimensionalities;     /* [number_features]             models.py:68 */
  int32_t number_encoder_layers;     /* len(feature_encoder_architecture) */
  const int32_t* feature_encoder_architecture; /* hidden widths                  models.py:76 */
  int32_t number_integration_layers; /* len(integration_network_architecture) */
  const int32_t* integration_network_architecture; /*                            models.py:82 */
  int32_t output_dimensionality;     /*                                          models.py:83 */
  int32_t use_positional_encoding;   /*                                          models.py:74 */
  int32_t number_positional_encoding_frequencies; /* n -> frequencies 2^1..2^(n-1), models.py:70 */
  int32_t activation_fn;             /* enum dib_activation */
  float   leaky_relu_alpha;          /* slope for DIB_ACT_LEAKY_RELU */
  int32_t feature_embedding_dimension; /* E                                      models.py:64 */
  int32_t output_activation_fn;      /* enum dib_activation                      models.py:83 */
  int32_t loss;                      /* enum dib_loss (model.compile(loss=...), train.py:138-142) */
  int32_t precision;                 /* enum dib_precision */
  int64_t max_batch;                 /* largest n any call will pass (sizes the workspace) */
  /* ---- custom-step variants of the same front end (NEXT ROW f3); zero-initialised fields give models.py ---- */
  float   logvar_offset;             /* constant added to every encoder's log-variance before sampling / KL / any output
                                        (nb-particle cell 8: embs_logvars + logvar_initialization, -3 there) */
  float   kl_loss_exponent;          /* nonlinear IB (nb-chaos cell 10): loss_IB = beta * kl_loss_scale * (sum_i KL_i)^exponent; */
  float   kl_loss_scale;             /*   0 or 1 / 0 or 1 = the linear beta * sum_i KL_i of models.py:118 */
  int32_t encoder_kind;              /* enum dib_encoder_kind */
  float   dropout_rate;              /* nb-radial cell 5: tf.keras.layers.Dropout(rate) after every hidden Dense of the feature
                                        encoders, active in dib_train_step only (Keras training=True); masks from the Philox
                                        stream (oracle/philox.py :: dropout_keep).  Encoders then run on the unfused kernels. */
} dib_config;

typedef struct dib_model dib_model;

/* models.DistributedIBNet.__init__ (models.py:56-86).  Uses the current CUDA device. */
int dib_create(const dib_config* cfg, dib_model** out);
void dib_destroy(dib_model* h);

/* number of trainable parameters == sum over model.trainable_variables (train.py:198). */
int64_t dib_param_count(const dib_model* h);

/* For every variable v (in flat order) its offset and shape: offsets[v], rows[v] (fan-in, or 0 for a
 * bias), cols[v].  Pass NULLs to query the number of variables (return value, negative on error). */
int dib_param_layout(const dib_model* h, int64_t* offsets, int32_t* rows, int32_t* cols, int32_t capacity);

/* bytes of scratch the caller must provide to forward / train_step / encode calls.  The workspace pointer must be 256-byte
 * aligned and `params` 16-byte aligned (checked; cudaMalloc / torch allocations are). */
size_t dib_workspace_bytes(const dib_model* h);

/* number of floats in the statistics vector: [ sum_b KL_i (F) | sum_b task loss | sum_b accuracy | n ] */
int32_t dib_stats_count(const dib_model* h);

/* DistributedIBNet.call (models.py:96-123) + compiled loss/metrics, no gradient: the validation pass of
 * Model.fit (train.py:157-166; noise is sampled in validation too, train.py:264-265).
 *   x [n, sum d_i]; y [n, out] (class index as float for sparse CE) or NULL; eps [n, F, E] or NULL ->
 *   Philox4x32-10 keyed (seed, step, feature, sample_offset + row, dim), see oracle/philox.py;
 *   out_pred [n, out] or NULL; out_emb [n, F*E] or NULL; out_stats [dib_stats_count] (zeroed by the call). */
int dib_forward(dib_model* h, const float* params, const float* x, const float* y, int64_t n,
                const float* beta_dev, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                float* out_pred, float* out_emb, float* out_stats, void* workspace, void* stream);

/* model.feature_encoders[i](x_i) (models.py:79; consumers visualization.py:31, utils.py:38, nb-radial
 * StashEmbeddingsCallback): deterministic [n, d_i] -> [n, 2E] = (mu || logvar). */
int dib_encode_feature(dib_model* h, const float* params, int32_t feature, const float* x_i, int64_t n,
                       float* out_mu_logvar, void* workspace, void* stream);

/* One Keras train_step minus the optimizer: forward, loss = task + beta*sum_i KL_i (models.py:118),
 * reverse mode (GradientTape in Model.fit / nb-bool cell 6).  grads_flat [P] receives
 * d(loss)/d(params) * (n_local-sum scaled by inv_global_batch); out_stats as in dib_forward.
 * grads_flat and out_stats may be adjacent in one buffer so that one all-reduce covers both. */
int dib_train_step(dib_model* h, const float* params, const float* x, const float* y, int64_t n,
                   const float* beta_dev, float inv_global_batch,
                   const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                   float* grads_flat, float* out_stats, void* workspace, void* stream);

/* NEXT ROW f3 -- encoder-only custom steps (nb-particle cell 8: a shared particle encoder feeding the caller's own
 * network, e.g. a set transformer; nb-chaos cell 10): the model's integration network is not used.
 *   dib_encoders_forward : x [n, sum d_i] -> out_emb [n, F*E] (u = mu + exp(logvar/2) eps) and out_stats (KL sums; loss = acc = 0).
 *   dib_encoders_backward: recomputes that forward, then reverse mode from d_emb [n, F*E] = d(caller's loss)/d(emb)
 *     (already carrying the caller's batch scaling) plus the IB term d(beta * scale * (sum KL)^p)/d(params) with KL means
 *     over inv_global_batch; grads_flat [P]: encoder entries written, integration-network entries zeroed.
 * A shared-weight encoder over a particle axis is F = 1 on n = B * particles rows with inv_global_batch = 1/B (KL summed
 * over particles, averaged over the batch). */
int dib_encoders_forward(dib_model* h, const float* params, const float* x, int64_t n, const float* eps, uint64_t seed,
                         uint32_t step, uint64_t sample_offset, float* out_emb, float* out_stats, void* workspace, void* stream);
int dib_encoders_backward(dib_model* h, const float* params, const float* x, const float* d_emb, int64_t n,
                          const float* beta_dev, float inv_global_batch, const float* eps, uint64_t seed, uint32_t step,
                          uint64_t sample_offset, float* grads_flat, float* out_stats, void* workspace, void* stream);

/* dib_train_step in two halves, for overlapping the data-parallel collective with the encoder backward:
 *   phases = 1: forward + compiled loss + integration-network backward -> grads_flat[first integration parameter, P) and
 *               out_stats are final (bucket 1 can be all-reduced while phase 2 runs);
 *   phases = 2: encoder backward -> grads_flat[0, first integration parameter) final.  Same arguments as the phase-1 call;
 *   phases = 3: both (== dib_train_step).
 * The first integration parameter is offsets[v] of variable v = number_features * (encoder variables per feature). */
int dib_train_step_phased(dib_model* h, const float* params, const float* x, const float* y, int64_t n,
                          const float* beta_dev, float inv_global_batch,
                          const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                          float* grads_flat, float* out_stats, void* workspace, int32_t phases, void* stream);

/* CUDA-Graph replay: a captured launch cannot carry a fresh by-value `step`, so the Philox step word may come from device
 * memory: when step_dev != NULL every later dib_train_step[_phased] call of this handle uses step + *step_dev (dib_forward
 * and the encoder-only entry points keep the by-value step).  The caller owns the counter and advances it (on the stream)
 * between steps.  NULL restores the by-value behaviour. */
int dib_set_noise_step_device(dib_model* h, const uint32_t* step_dev);

/* tf.keras.optimizers.Adam dense update over the flat buffer (train.py:128-129, nb-radial Adam(lr)):
 *   t = *step_dev + 1 (the kernel increments *step_dev);  lr_t = lr*sqrt(1-b2^t)/(1-b1^t);
 *   m += (1-b1)(g-m); v += (1-b2)(g^2-v); w -= lr_t*m/(sqrt(v)+eps)   (eps outside the bias correction). */
int dib_adam_step(float* params, const float* grads, float* m, float* v, int64_t count,
                  const float* lr_dev, int32_t* step_dev, float beta_1, float beta_2, float epsilon,
                  void* stream);

/* the other optimizers tf.keras.optimizers.get(name) hands out (train.py:41,128); same device scalars as dib_adam_step.
 *   kind 0 SGD     : v = momentum * v - lr * g;  w += nesterov ? momentum * v - lr * g : v        (slot1 = v; slot2 unused)
 *   kind 1 RMSprop : ms = rho * ms + (1-rho) g^2;  mom = momentum * mom + lr * g / sqrt(ms + eps);  w -= mom   (TF ApplyRMSProp;
 *                    slot1 = ms, slot2 = mom)
 * hyper = {momentum, nesterov(0/1), 0} for SGD, {rho, momentum, epsilon} for RMSprop.  *step_dev is incremented. */
int dib_optimizer_step(int32_t kind, float* params, const float* grads, float* slot1, float* slot2, int64_t count,
                       const float* lr_dev, int32_t* step_dev, float hyper0, float hyper1, float hyper2, void* stream);

/* model.integration_network(emb) (models.py:84,122) as a stand-alone call: emb [n, F*E] -> out_pred [n, out] through the
 * Dense stack with the output activation, on the model's precision path (fp32 FMA / tf32 tcgen05). */
int dib_integration_forward(dib_model* h, const float* params, const float* emb, int64_t n, float* out_pred,
                            void* workspace, void* stream);

/* models.PositionalEncoding.call (models.py:12-23) as a stand-alone call: x [n, d] ->
 * out [n, d * number_frequencies] = concat([x] + [sin(2^k x) for k = 1 .. number_frequencies-1], -1), block-major. */
int dib_positional_encoding(const float* x, int64_t n, int32_t d, int32_t number_frequencies, float* out, void* stream);

/* Keras metric aggregation of one batch (Model.fit's Mean metrics; add_metric at models.py:115,121):
 *   acc[0..F)  += stats[i]/n              (KL_i batch mean; history['KL{i}'] = acc[i]/acc[F+3])
 *   acc[F]     += stats[F] + beta*sum_i stats[i]   (sample-weighted total loss; history['loss'] = acc[F]/acc[F+2])
 *   acc[F+1]   += stats[F+1]              (accuracy sum;  history['accuracy'] = acc[F+1]/acc[F+2])
 *   acc[F+2]   += n ;  acc[F+3] += 1      (samples, batches)
 * stats is the (all-reduced) vector written by dib_train_step / dib_forward; acc has F+4 floats. */
int dib_metrics_update(const float* stats, const float* beta_dev, float* acc, int32_t number_features, void* stream);
/* the same with the nonlinear IB term: acc[F] += stats[F] + n * beta * kl_loss_scale * (sum_i stats[i] / n)^kl_loss_exponent */
int dib_metrics_update_ex(const float* stats, const float* beta_dev, float* acc, int32_t number_features,
                          float kl_loss_exponent, float kl_loss_scale, void* stream);

/* utils.bhattacharyya_dist_mat (utils.py:177-212) followed by exp(-D) (visualization.py:34):
 * mu_logvar [n, 2E] -> out_dist [n, n] (may be NULL) and out_compression [n, n] (may be NULL). */
int dib_bhattacharyya(const float* mu_logvar, int64_t n, int32_t embedding_dimension,
                      float* out_dist, float* out_compression, void* stream);

/* NEXT ROW f2 -- pairwise closed forms between two sets of diagonal Gaussians, rows (mu || logvar):
 *   kind 0: utils.bhattacharyya_dist_mat(mus1, logvars1, mus2, logvars2)  (utils.py:177-212)
 *   kind 1: utils.kl_divergence_mat(mus1, logvars1, mus2, logvars2) = KL(N1_i || N2_j)  (utils.py:213-247)
 * mu_logvar_1 [n, 2E], mu_logvar_2 [m, 2E] -> out [n, m] and/or out_exp_neg [n, m] = exp(-out) (either may be NULL). */
int dib_pairwise_gaussian(int32_t kind, const float* mu_logvar_1, int64_t n, const float* mu_logvar_2, int64_t m,
                          int32_t embedding_dimension, float* out, float* out_exp_neg, void* stream);

/* NEXT ROW f2 -- visualization.save_compression_matrices (visualization.py:14-35) / SaveCompressionMatricesCallback
 * (models.py:152-186) / StashEmbeddingsCallback (nb-radial cell 5) for ALL features in one call: for feature i take
 * rows row_index[i, 0..n) of x [n_total, sum d_i] (row_index: device int32 [F, n], NULL = rows 0..n-1 for every
 * feature), run encoder i without noise, then Bhattacharyya and exp(-D).  Outputs (each may be NULL):
 * out_mu_logvar [F, n, 2E], out_dist [F, n, n], out_compression [F, n, n].  n <= config.max_batch. */
int dib_compression_matrices(dib_model* h, const float* params, const float* x, int64_t n_total,
                             const int32_t* row_index, int64_t n, float* out_mu_logvar, float* out_dist,
                             float* out_compression, void* workspace, void* stream);

/* NEXT ROW f3 -- utils.get_scaled_similarity (utils.py:127-175; distances utils.py:75-125):
 * kind 0 'l2sq' | 1 'l2' | 2 'l1' | 3 'linf' | 4 'cosine';  e1 [n, d], e2 [m, d] -> out [n, m] = similarity / temperature. */
int dib_scaled_similarity(int32_t kind, const float* e1, int64_t n, const float* e2, int64_t m, int32_t d,
                          float temperature, float* out, void* stream);

/* NEXT ROW f3 -- the InfoNCE head of the custom training loop (train.py:203-213) and its reverse mode (train.py:216-219):
 *   S = get_scaled_similarity(e1, e2);  out_loss[0] = mean_i CE(i, S[i,:]) + mean_i CE(i, S^T[i,:])   (nats)
 *   d_e1, d_e2 [n, d] = d loss / d e1, d e2 (either may be NULL).  e1 = model(x) (feed d_e1 to dib_train_step of a
 *   DIB_LOSS_EXTERNAL model), e2 = the caller's output encoder.  scratch: n*n + 4n floats.  n <= 32768, d <= 512. */
int dib_infonce_head(int32_t kind, const float* e1, const float* e2, int64_t n, int32_t d, float temperature,
                     float* scratch, float* out_loss, float* d_e1, float* d_e2, void* stream);

/* The same head, streamed on the tensor cores (tcgen05) for the similarities with a Gram form: kind 0 'l2sq' | 1 'l2' |
 * 4 'cosine'.  The n x n similarity matrix is never stored: scratch is O(n d) bytes, as returned by
 * dib_infonce_head_tc_scratch_bytes (-1 for arguments out of range), and must be 128-byte aligned.  1 <= n <= 2^26,
 * 1 <= d <= 256.  Products use bf16 hi + lo split operands with fp32 accumulation, the positive pairs s_ii are exact
 * fp32; deterministic (identical calls give identical bytes).  No allocation, no host synchronisation. */
int64_t dib_infonce_head_tc_scratch_bytes(int64_t n, int32_t d);
int dib_infonce_head_tc(int32_t kind, const float* e1, const float* e2, int64_t n, int32_t d, float temperature,
                        void* scratch, float* out_loss, float* d_e1, float* d_e2, void* stream);

/* ---- InfoNCE training (train.py:180-289) on a DIB_LOSS_INFONCE handle ----------------------------------------------
 * The output encoder of train.py:186-193: y [n, input_dimensionality] -> PositionalEncoding(2**arange(1, nfreq)) when the
 * model uses it -> Dense(architecture[j], activation_fn) per width -> Dense(output_dimensionality) (linear), with the
 * model's positional-encoding settings and activation.  Attach it once per handle, before the first call that uses it;
 * dib_workspace_bytes then includes its buffers.  Its Q parameters follow the model's P ones: every call below takes
 * params [P + Q], the encoder's variables in Keras order [W0, b0, W1, b1, ...] with [in, out] kernels at params[P, P+Q). */
typedef struct dib_output_encoder_config {
  int32_t input_dimensionality;      /* width of y */
  int32_t number_layers;             /* len(infonce_y_encoder_architecture) (may be 0) */
  const int32_t* architecture;       /* hidden widths */
} dib_output_encoder_config;

int dib_attach_output_encoder(dib_model* h, const dib_output_encoder_config* cfg);
/* Q, or -1 (no encoder attached / null handle) */
int64_t dib_output_encoder_param_count(const dib_model* h);
/* as dib_param_layout; offsets index the [P + Q] buffer, so the first is P */
int dib_output_encoder_param_layout(const dib_model* h, int64_t* offsets, int32_t* rows, int32_t* cols, int32_t capacity);
/* output_encoder(y): y [n, input_dimensionality] -> out_e2 [n, output_dimensionality] */
int dib_output_encoder_forward(dib_model* h, const float* params, const float* y, int64_t n, float* out_e2, void* workspace,
                               void* stream);

/* eval_batch_infonce(training=True) of train.py:201-219 minus the optimizer, with ONE model forward:
 *   e1 = model(x) (noise as dib_train_step, including dib_set_noise_step_device), e2 = output_encoder(y),
 *   L = mean_i CE(i, S[i,:]) + mean_i CE(i, S^T[i,:]) with S = get_scaled_similarity(e1, e2, kind, temperature),
 *   loss = L + beta * sum_i KL_i.
 * kind 0 'l2sq' | 1 'l2' | 4 'cosine' run the streaming tensor-core head (dib_infonce_head_tc: any n, output_dimensionality
 * <= 256); 2 'l1' | 3 'linf' the exact head (n <= 32768).  head_scratch: dib_infonce_scratch_bytes(kind, n, D) bytes,
 * 128-byte aligned.  grads_flat [P + Q] = d loss / d params, already batch-mean scaled; out_stats [F + 3] =
 * [ sum_b KL_i (F) | n * L | 0 | n ], so dib_metrics_update_ex accumulates loss = L + IB term.  No allocation, no host
 * synchronisation: CUDA-Graph capturable. */
int dib_infonce_train_step(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                           int32_t kind, float temperature, const float* eps, uint64_t seed, uint32_t step,
                           uint64_t sample_offset, void* head_scratch, float* grads_flat, float* out_stats, void* workspace,
                           void* stream);
/* the same without gradients: the validation pass (train.py:266); the by-value step is used, as in dib_forward */
int dib_infonce_forward(dib_model* h, const float* params, const float* x, const float* y, int64_t n, const float* beta_dev,
                        int32_t kind, float temperature, const float* eps, uint64_t seed, uint32_t step, uint64_t sample_offset,
                        void* head_scratch, float* out_stats, void* workspace, void* stream);
/* head_scratch bytes of the two calls above; -1 where they refuse (unknown kind, d > 256 for a Gram kind, n > 32768 for
 * l1 / linf) */
int64_t dib_infonce_scratch_bytes(int32_t kind, int64_t n, int32_t d);

/* NEXT ROW f1 -- utils.estimate_mi_sandwich_bounds' per-batch kernel (utils.py:36-65): InfoNCE lower and leave-one-out
 * upper bound (nats) of I(U;X) for one encoder on one batch of n samples.  mu_logvar [n, 2E] (dib_encode_feature
 * output); eps [n, E] or NULL -> Philox(seed, step, row, feature 0, dim); row_scratch [2n] floats; out [2]. */
int dib_mi_sandwich_bounds(const float* mu_logvar, int64_t n, int32_t embedding_dimension, const float* eps, uint64_t seed,
                           uint32_t step, float* row_scratch, float* out_lower_upper, void* stream);

/* NEXT ROW f1, batched -- the whole of utils.estimate_mi_sandwich_bounds / InfoPerFeatureCallback (models.py:188-223) in one
 * launch: `groups` = features x evaluation batches independent problems of n rows each, mu_logvar [groups, n, 2E] (the
 * out_mu_logvar of dib_compression_matrices with n = batches * batch size rows per feature is exactly this layout),
 * accumulated in float64 as the reference does (utils.py:40-41).  eps [groups, n, E] or NULL -> Philox keyed
 * ((seed << 8) + g / batches_per_feature; step g % batches_per_feature; row; feature 0; dim), i.e. the streams of the
 * per-feature, per-batch calls.  row_scratch: groups * n * 2 doubles; out: [groups, 2] doubles (lower, upper) in nats. */
int dib_mi_sandwich_bounds_batched(const float* mu_logvar, int32_t groups, int64_t n, int32_t embedding_dimension,
                                   const float* eps, uint64_t seed, int32_t batches_per_feature, double* row_scratch,
                                   double* out_lower_upper, void* stream);

/* NEXT ROW f4 -- ctw.estimate_entropy(seq, alphabet_size) (chaos/ctw.pyx:2-3 -> chaos/cppctw.cpp:163-171): infinite-depth
 * Context-Tree-Weighting entropy-rate estimate in bits/symbol.  HOST functions on HOST memory (the suffix-tree build is
 * irregular pointer chasing; SURVEY 8f keeps it on the CPU): symbols are int8 in [0, alphabet_size), alphabet_size <= 127.
 * The batch form runs `count` independent sequences (sequences + offsets[i] .. offsets[i+1]) on num_threads host threads
 * (<= 0: all cores).  Results are bit-identical to the reference (double carrying a float-rounded value). */
int dib_ctw_estimate_entropy(const int8_t* sequence, int64_t length, int32_t alphabet_size, double* out_bits_per_symbol);
int dib_ctw_estimate_entropy_batch(const int8_t* sequences, const int64_t* offsets, int32_t count, int32_t alphabet_size,
                                   int32_t num_threads, double* out_bits_per_symbol);
const char* dib_ctw_last_error(void);

/* ---- observability (no reference counterpart) ---------------------------------------------------------
 * dib_launch_count: kernels launched by this library in this process.
 * dib_profile_enable(h,1): bracket every launch group of subsequent forward/train_step calls with CUDA events
 * recorded on the caller's stream; dib_profile_read waits for them and returns up to `capacity` durations (ms)
 * with '\n'-separated labels; dib_profile_enable(h,0) turns it off and frees the events. */
uint64_t dib_launch_count(void);
int dib_profile_enable(dib_model* h, int32_t on);
int32_t dib_profile_read(dib_model* h, char* labels, size_t labels_bytes, float* ms, int32_t capacity);

/* bring-up / unit-test hook: ONE GEMM problem through the tensor-core kernel (use_simt=0) or the fp32 SIMT kernel
 * (use_simt=1); mode 0 FWD (bias = X, act), 1 DGRAD (X = activation source), 2 WGRAD (X = bias-grad partials).
 * Synchronises the stream. */
int dib_debug_gemm_tc(int32_t mode, const float* A, int32_t lda, const float* B, int32_t ldb, float* Cout, int32_t ldc,
                      float* X, int32_t ldx, int32_t M, int32_t T, int32_t Ccols, int32_t R, int32_t act,
                      int32_t nsplit, int32_t rows_per_split, int64_t split_stride, int32_t use_simt, void* stream);

/* bring-up switch (bit mask): 1 = unfused encoder kernels, 2 = integration network on fp32-storage TF32 kernels. */
int dib_debug_force_unfused(dib_model* h, int32_t on);

/* process-wide kernel-variant switch for A/B measurements.  key 0: fused encoder backward kernel, value 1 = the
 * single-chain kernel of round 1, 2 = two chains on consecutive tiles (default; also DIB_ENC_BWD=1|2 in the environment).
 * key 1: 16-bit integration FWD / DGRAD GEMMs, 1 = weight slice resident in shared memory, 0 = re-streamed per tile (default:
 * measured faster; also DIB_INT16_RB=0|1).
 * key 2: fused output head for output_dimensionality == 1, 1 = eight rows per pass with a lane-parallel loss (default), 0 = the
 * generic kernel.
 * key 3: single-output models whose last two hidden integration layers are 256 wide, 1 = those layers + the head + the loss as one
 * kernel (default; also DIB_INT16_FWD2=0|1), 0 = one kernel per layer and the head kernel of key 2.
 * key 4: 16-bit integration GEMMs whose output width is a multiple of 256, 1 = CTA-pair kernels (tcgen05 cta_group::2, 256 x 256 tile
 * per pair; also DIB_INT16_2SM=1), 0 = single-CTA 128 x 128 kernels (default: measured the same or faster).
 * key 5: MEASUREMENT ONLY, wrong results: 1 = the 16-bit GEMM epilogues skip their global stores (cost of the store path). */
int dib_debug_set_variant(int32_t key, int32_t value);

/* text of the last error raised on this thread ("" if none). */
const char* dib_last_error(void);

/* "sm_100a" etc: the architecture the kernels were compiled for, and the ABI version. */
const char* dib_build_info(void);

/* one line describing what THIS handle runs, e.g.
 * "precision=fp16 encoders=fused-tcgen05-f16 integration=int16-tcgen05-f16 operands=fp16 accumulate=fp32".
 * Returns the number of bytes written (excluding the terminator), negative on error. */
int32_t dib_model_info(const dib_model* h, char* out, size_t out_bytes);

#ifdef __cplusplus
}
#endif
#endif /* DIB_B200_H_ */
