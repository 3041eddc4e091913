"""TEST INFRASTRUCTURE ONLY -- CPU (numpy) restatement of the reference's Distributed-IB hot path.

PARITY STATUS: "parity unpinned" against TensorFlow itself.  The reference has no tests and
TensorFlow/Keras (unpinned 2.x, third-party, absent from /root/reference and from this image)
cannot be run here.  This oracle is pinned instead by
  (i)  the closed-form known answers derivable from the reference's own formulas
       (SURVEY.md section 4: beta schedule, KL, Bhattacharyya, PE layout, circuit truth table),
  (ii) golden vectors produced by executing the reference's OWN model code
       (/root/reference/models.py ``DistributedIBNet.call``, ``InfoBottleneckAnnealingCallback``,
       /root/reference/utils.py ``bhattacharyya_dist_mat``) on a numpy stand-in for the ``tf``
       namespace -- tests/golden/make_golden.py, fixtures committed under tests/golden/.
Keras behaviours that live in the third-party dependency are restated from its published
semantics and each is marked [KERAS] below.

Each function cites the reference lines it follows (paths relative to /root/reference).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module;
the product path (dib_b200) never does.
"""
from __future__ import annotations

import ast
import hashlib
import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence

import numpy as np

LOSS_BCE_LOGITS = "bce_logits"          # tf.keras.losses.BinaryCrossentropy(from_logits=True)  data.py:65
LOSS_SPARSE_CE_LOGITS = "sparse_ce_logits"  # SparseCategoricalCrossentropy(from_logits=True)   data.py:343
LOSS_MSE = "mse"                        # regression targets (data.py:129 implies it)
LOSS_BCE_PROBS = "bce_probs"            # [KERAS] BinaryCrossentropy() on probabilities (from_logits=False, the Keras default)
_KERAS_EPS = 1e-7                       # keras.backend.epsilon()


# ----------------------------------------------------------------------------------------------
# activations ([KERAS] tf.keras.activations.get(name)); derivatives are written in terms of the
# OUTPUT h = act(z) because that is what the CUDA backward has at hand.
# ----------------------------------------------------------------------------------------------
def act_fwd(name, z, alpha=0.2):
    if name in (None, "linear"):
        return z
    if name == "relu":
        return np.maximum(z, 0)
    if name == "tanh":
        return np.tanh(z)
    if name == "leaky_relu":
        return np.where(z > 0, z, alpha * z)
    if name == "sigmoid":
        return 1.0 / (1.0 + np.exp(-z))
    if name == "elu":
        return np.where(z > 0, z, np.expm1(np.minimum(z, 0)))
    raise ValueError(f"unknown activation {name!r}")


def act_grad_from_output(name, h, alpha=0.2):
    if name in (None, "linear"):
        return np.ones_like(h)
    if name == "relu":
        return (h > 0).astype(h.dtype)
    if name == "tanh":
        return 1.0 - h * h
    if name == "leaky_relu":
        return np.where(h > 0, 1.0, alpha).astype(h.dtype)
    if name == "sigmoid":
        return h * (1.0 - h)
    if name == "elu":
        return np.where(h > 0, 1.0, h + 1.0).astype(h.dtype)
    raise ValueError(f"unknown activation {name!r}")


# ----------------------------------------------------------------------------------------------
# model description + parameters
# ----------------------------------------------------------------------------------------------
@dataclass
class DIBConfig:
    """Constructor arguments of DistributedIBNet (models.py:56-66; dropout-free)."""
    feature_dimensionalities: Sequence[int]
    feature_encoder_architecture: Sequence[int]
    integration_network_architecture: Sequence[int]
    output_dimensionality: int
    use_positional_encoding: bool = True
    number_positional_encoding_frequencies: int = 5
    activation_fn: Optional[str] = "relu"
    feature_embedding_dimension: int = 32
    output_activation_fn: Optional[str] = None
    leaky_alpha: float = 0.2
    # ---- custom-step variants of the same front end (SURVEY 8f3) ----
    # logvar_offset: constant added to every encoder's log-variance output before sampling and KL
    #   (nb-particle cell 8: `embs_logvars = embs_logvars + logvar_initialization`, -3 there)
    logvar_offset: float = 0.0
    # nonlinear IB: loss_IB = beta * kl_loss_scale * (sum_i KL_i) ** kl_loss_exponent
    #   (nb-chaos cell 10: `loss = beta_var * number_states * kl ** kl_loss_exponent`); (1, 1) = models.py:118
    kl_loss_exponent: float = 1.0
    kl_loss_scale: float = 1.0
    # 'mlp' (models.py:72-78) or 'simple': nb-bool cell 4 SimpleEncoder -- two trainable (1,1) constants per feature,
    #   output concat([x * mu_scaling, ones_like(x) * logvar]); needs d_i == feature_embedding_dimension
    encoder_kind: str = "mlp"
    # nb-radial cell 5: tf.keras.layers.Dropout(dropout_rate) after every hidden Dense of the feature encoders (training only)
    dropout_rate: float = 0.0

    @property
    def number_features(self):
        return len(self.feature_dimensionalities)

    @property
    def frequencies(self):
        # models.py:70 -- 2**np.arange(1, n): n-1 sinusoid blocks (off-by-one vs the docstring)
        return [2 ** k for k in range(1, self.number_positional_encoding_frequencies)]

    def encoder_input_width(self, i):
        d = self.feature_dimensionalities[i]
        return d * (1 + len(self.frequencies)) if self.use_positional_encoding else d

    def encoder_layer_dims(self, i):
        dims = [self.encoder_input_width(i)] + list(self.feature_encoder_architecture)
        dims.append(2 * self.feature_embedding_dimension)           # models.py:77
        return dims

    def integration_layer_dims(self):
        return ([self.number_features * self.feature_embedding_dimension]  # models.py:81
                + list(self.integration_network_architecture) + [self.output_dimensionality])

    def param_shapes(self):
        """Flat order: feature 0 (W1,b1,W2,b2,...), feature 1 ..., integration (W,b)...  Kernels are
        Keras-oriented [in, out] (tf.keras.layers.Dense)."""
        shapes = []
        for i in range(self.number_features):
            if self.encoder_kind == "simple":
                shapes += [(1, 1), (1, 1)]                      # mu_scaling, logvar (nb-bool cell 4)
                continue
            d = self.encoder_layer_dims(i)
            for k in range(len(d) - 1):
                shapes += [(d[k], d[k + 1]), (d[k + 1],)]
        d = self.integration_layer_dims()
        for k in range(len(d) - 1):
            shapes += [(d[k], d[k + 1]), (d[k + 1],)]
        return shapes

    def param_count(self):
        return int(sum(int(np.prod(s)) for s in self.param_shapes()))


def glorot_uniform_params(cfg: DIBConfig, rng: np.random.Generator, dtype=np.float32) -> np.ndarray:
    """[KERAS] Dense default init: kernel glorot_uniform (limit sqrt(6/(fan_in+fan_out))), bias zeros.
    The RNG stream is ours (numpy Generator); Keras' own stream is irreproducible without TF."""
    out = []
    n_simple = 2 * cfg.number_features if cfg.encoder_kind == "simple" else 0
    for idx, s in enumerate(cfg.param_shapes()):
        if idx < n_simple:                                       # nb-bool cell 4: mu_scaling = 1, logvar = -3
            out.append(np.full(1, 1.0 if idx % 2 == 0 else -3.0, dtype=dtype))
        elif len(s) == 2:
            lim = math.sqrt(6.0 / (s[0] + s[1]))
            out.append(rng.uniform(-lim, lim, size=s).astype(dtype).ravel())
        else:
            out.append(np.zeros(s, dtype=dtype))
    return np.concatenate(out)


def golden_case_params(cfg: DIBConfig, seed: int):
    """Weights of a tests/golden/ref_forward_*.npz case: glorot-uniform kernels and N(0, 0.05^2) biases (non-zero, so
    that bias handling is pinned) drawn from default_rng(seed).  Returns (weights, rng); the case's inputs come next."""
    rng = np.random.default_rng(seed)
    flat = glorot_uniform_params(cfg, rng, dtype=np.float32)
    flat = flat + (rng.standard_normal(flat.size) * 0.05).astype(np.float32) * (flat == 0)
    return flat, rng


def load_forward_golden(path):
    """(cfg, arrays) of a tests/golden/ref_forward_*.npz case.  The weights are not stored (C0's alone are 2.4 MB of
    incompressible floats): they are regenerated from the stored seed and checked against the SHA-256 of the weights
    the reference computed the case with, so a change in numpy's random streams fails loudly instead of comparing
    against the wrong model."""
    z = dict(np.load(path))
    cfg = DIBConfig(**ast.literal_eval(str(z["cfg"])))
    params, _ = golden_case_params(cfg, int(z["seed"]))
    if hashlib.sha256(params.tobytes()).hexdigest() != str(z["params_sha256"]):
        raise RuntimeError(f"{path}: the weights regenerated from seed {int(z['seed'])} are not the golden's")
    z["params"] = params
    return cfg, z


def unflatten(cfg: DIBConfig, flat: np.ndarray):
    """-> (encoders: list over features of [(W,b),...], integration: [(W,b),...])"""
    views, off = [], 0
    for s in cfg.param_shapes():
        n = int(np.prod(s))
        views.append(flat[off:off + n].reshape(s))
        off += n
    assert off == flat.size
    it = iter(views)
    n_enc_layers = 1 if cfg.encoder_kind == "simple" else len(cfg.feature_encoder_architecture) + 1
    encoders = [[(next(it), next(it)) for _ in range(n_enc_layers)] for _ in range(cfg.number_features)]
    n_int_layers = len(cfg.integration_network_architecture) + 1
    integration = [(next(it), next(it)) for _ in range(n_int_layers)]
    return encoders, integration


# ----------------------------------------------------------------------------------------------
# forward pieces
# ----------------------------------------------------------------------------------------------
def positional_encoding(x, frequencies):
    """models.py:22-23: concat([x] + [sin(f*x) for f in frequencies], -1)  (block-major)."""
    return np.concatenate([x] + [np.sin(f * x) for f in frequencies], axis=-1)


def split_features(cfg: DIBConfig, x):
    """models.py:101: tf.split(inputs, feature_dimensionalities, axis=-1)."""
    offs = np.cumsum([0] + list(cfg.feature_dimensionalities))
    assert x.shape[-1] == offs[-1]                                   # models.py:89
    return [x[:, offs[i]:offs[i + 1]] for i in range(cfg.number_features)]


def encoder_forward(cfg: DIBConfig, layers, x_i, keep=False, drop=None):
    """models.py:72-78 Sequential: [PE] -> Dense(h,act)... -> Dense(2E) (linear).  a15 contract.
    ``drop(layer, shape)`` (training with dropout_rate > 0, nb-radial cell 5) returns the Keras Dropout scale mask
    (0 or 1/(1-rate)) applied to the OUTPUT of hidden layer ``layer`` (1-based: the activation that feeds layer ``layer``).
    With ``keep``: returns (out, acts, pres, masks) where acts[k] feeds layer k (after dropout), pres[k] is the same
    activation before dropout (what act' is taken from), masks[k] the scale mask (None where there is none)."""
    h = positional_encoding(x_i, cfg.frequencies) if cfg.use_positional_encoding else x_i
    acts, pres, masks = [h], [h], [None]
    for k, (W, b) in enumerate(layers):
        z = h @ W + b
        if k < len(layers) - 1:
            hh = act_fwd(cfg.activation_fn, z, cfg.leaky_alpha)
            m = drop(k + 1, hh.shape) if drop is not None else None
            h = hh * m if m is not None else hh
            pres.append(hh); masks.append(m)
        else:
            h = z
            pres.append(z); masks.append(None)
        acts.append(h)
    return (h, acts, pres, masks) if keep else h


def task_loss_per_sample(loss, pred, y):
    """[KERAS] per-sample loss value; the compiled loss is its mean over the batch."""
    if loss == LOSS_BCE_LOGITS:
        yy = y.reshape(pred.shape).astype(pred.dtype)
        l = np.maximum(pred, 0) - pred * yy + np.log1p(np.exp(-np.abs(pred)))
        return l.mean(axis=-1)
    if loss == LOSS_SPARSE_CE_LOGITS:
        m = pred.max(axis=-1, keepdims=True)
        lse = (m + np.log(np.exp(pred - m).sum(axis=-1, keepdims=True)))[:, 0]
        return lse - pred[np.arange(pred.shape[0]), y.astype(np.int64).ravel()]
    if loss == LOSS_MSE:
        yy = y.reshape(pred.shape).astype(pred.dtype)
        return ((pred - yy) ** 2).mean(axis=-1)
    if loss == LOSS_BCE_PROBS:      # keras.backend.binary_crossentropy: clip to [eps, 1-eps], then log(p + eps)
        yy = y.reshape(pred.shape).astype(pred.dtype)
        pc = np.clip(pred, _KERAS_EPS, 1.0 - _KERAS_EPS)
        return (-(yy * np.log(pc + _KERAS_EPS) + (1.0 - yy) * np.log(1.0 - pc + _KERAS_EPS))).mean(axis=-1)
    raise ValueError(loss)


def task_loss_grad(loss, pred, y):
    """d(sum_b per-sample loss)/d pred  (caller scales by 1/B)."""
    if loss == LOSS_BCE_LOGITS:
        yy = y.reshape(pred.shape).astype(pred.dtype)
        return (1.0 / (1.0 + np.exp(-pred)) - yy) / pred.shape[-1]
    if loss == LOSS_SPARSE_CE_LOGITS:
        m = pred.max(axis=-1, keepdims=True)
        p = np.exp(pred - m)
        p /= p.sum(axis=-1, keepdims=True)
        p[np.arange(pred.shape[0]), y.astype(np.int64).ravel()] -= 1.0
        return p
    if loss == LOSS_MSE:
        yy = y.reshape(pred.shape).astype(pred.dtype)
        return 2.0 * (pred - yy) / pred.shape[-1]
    if loss == LOSS_BCE_PROBS:
        yy = y.reshape(pred.shape).astype(pred.dtype)
        pc = np.clip(pred, _KERAS_EPS, 1.0 - _KERAS_EPS)
        g = -yy / (pc + _KERAS_EPS) + (1.0 - yy) / (1.0 - pc + _KERAS_EPS)
        return np.where((pred > _KERAS_EPS) & (pred < 1.0 - _KERAS_EPS), g, 0.0) / pred.shape[-1]
    raise ValueError(loss)


def accuracy_count(loss, pred, y):
    """[KERAS] metrics=['accuracy'] resolution: binary_accuracy (threshold 0.5 applied to the RAW
    model output, logits included) for a BCE loss; sparse_categorical_accuracy for sparse CE.
    Returns the SUM over the batch of per-sample accuracies."""
    if loss == LOSS_SPARSE_CE_LOGITS:
        return float((pred.argmax(axis=-1) == y.astype(np.int64).ravel()).sum())
    yy = y.reshape(pred.shape)
    return float(((pred > 0.5).astype(np.float64) == yy).mean(axis=-1).sum())


@dataclass
class ForwardResult:
    pred: np.ndarray
    emb: np.ndarray               # [B, F*E] concat of u_i (models.py:122)
    kl_per_feature: np.ndarray    # [F], mean over batch (models.py:111-112), nats
    task_loss: float              # mean over batch
    loss: float                   # task + beta*sum KL (models.py:118 + compiled loss)
    acc_sum: float
    cache: dict = field(default_factory=dict)


def dropout_fn(cfg: DIBConfig, seed, step, sample_ids, feature, dtype=np.float64):
    """The Philox-keyed Dropout masks of one feature encoder for a training step (see oracle/philox.py :: dropout_keep)."""
    from . import philox
    rate = np.float32(cfg.dropout_rate)
    scale = dtype(1.0) / (dtype(1.0) - dtype(rate))
    return lambda layer, shape: philox.dropout_keep(seed, step, sample_ids, feature, layer, shape[1], rate).astype(dtype) * scale


def forward(cfg: DIBConfig, flat_params, x, eps, beta, y=None, loss=None, keep=False, dtype=np.float64, dropout=None):
    """models.py:96-123 with eps explicit: u = mu + exp(logvar/2)*eps  (== tf.random.normal(mean=mu,
    stddev=exp(logvar/2)), models.py:108).  eps: [B, F, E]."""
    p = np.asarray(flat_params, dtype=dtype)
    x = np.asarray(x, dtype=dtype)
    eps = np.asarray(eps, dtype=dtype)
    encoders, integration = unflatten(cfg, p)
    E = cfg.feature_embedding_dimension
    xs = split_features(cfg, x)
    embs, kls, enc_cache = [], [], []
    for i in range(cfg.number_features):
        if cfg.encoder_kind == "simple":                              # nb-bool cell 4: concat([x*mu_scaling, 1*logvar])
            ms, lvc = encoders[i][0]
            assert xs[i].shape[1] == E, "SimpleEncoder needs d_i == feature_embedding_dimension"
            o, acts = np.concatenate([xs[i] * ms, np.ones_like(xs[i]) * lvc], axis=-1), [xs[i]]
        else:
            # dropout = (seed, step, global sample ids) of a TRAINING step; None = inference (Keras: Dropout is the identity)
            drop = dropout_fn(cfg, dropout[0], dropout[1], dropout[2], i, dtype) if (dropout is not None and cfg.dropout_rate > 0) else None
            o, acts, pres, masks = encoder_forward(cfg, encoders[i], xs[i], keep=True, drop=drop)
        mu, lv = o[:, :E], o[:, E:] + cfg.logvar_offset               # models.py:106 tf.split(.,2,-1); nb-particle offset
        u = mu + np.exp(lv / 2.0) * eps[:, i, :]                      # models.py:108
        kl = (0.5 * (mu ** 2 + np.exp(lv) - lv - 1.0)).sum(axis=-1).mean()   # models.py:111-112
        embs.append(u)
        kls.append(kl)
        if cfg.encoder_kind == "simple":
            pres, masks = acts, [None] * len(acts)
        enc_cache.append((acts, mu, lv, pres, masks))
    emb = np.concatenate(embs, axis=-1)                               # models.py:122
    h = emb
    int_acts = [h]
    for k, (W, b) in enumerate(integration):
        z = h @ W + b
        if k < len(integration) - 1:
            h = act_fwd(cfg.activation_fn, z, cfg.leaky_alpha)
        else:
            h = act_fwd(cfg.output_activation_fn, z, cfg.leaky_alpha)  # models.py:83
        int_acts.append(h)
    pred = h
    kls = np.asarray(kls, dtype=dtype)
    res = ForwardResult(pred=pred, emb=emb, kl_per_feature=kls, task_loss=float("nan"),
                        loss=float("nan"), acc_sum=float("nan"))
    if y is not None and loss != "external":
        res.task_loss = float(task_loss_per_sample(loss, pred, y).mean())
        res.loss = res.task_loss + ib_loss(cfg, beta, kls)            # models.py:118 / nb-chaos nonlinear IB
        res.acc_sum = accuracy_count(loss, pred, y)
    if keep:
        res.cache = dict(enc=enc_cache, int_acts=int_acts, encoders=encoders, integration=integration)
    return res


def ib_loss(cfg: DIBConfig, beta, kls):
    """beta * sum_i KL_i (models.py:118), or the nonlinear IB beta * L * KL**p of nb-chaos cell 10."""
    return float(beta) * cfg.kl_loss_scale * float(np.sum(kls)) ** cfg.kl_loss_exponent


def effective_beta(cfg: DIBConfig, beta, kls):
    """d(ib_loss)/d(sum KL): the weight the per-sample KL gradients carry in reverse mode."""
    p = cfg.kl_loss_exponent
    return float(beta) * cfg.kl_loss_scale * (1.0 if p == 1.0 else p * float(np.sum(kls)) ** (p - 1.0))


def train_grads(cfg: DIBConfig, flat_params, x, y, eps, beta, loss, dtype=np.float64, batch_for_mean=None, d_emb=None,
                dropout=None):
    """Reverse mode through forward() (what GradientTape does inside Keras' train_step).
    Returns (flat grads of mean-loss, ForwardResult).  ``batch_for_mean`` lets a shard of a larger
    global batch produce its additive share (grads scale 1/B_global)."""
    fr = forward(cfg, flat_params, x, eps, beta, y=y, loss=loss, keep=True, dtype=dtype, dropout=dropout)
    B = x.shape[0] if batch_for_mean is None else batch_for_mean
    beta = effective_beta(cfg, beta, fr.kl_per_feature * (x.shape[0] / B))   # KL means are over the GLOBAL batch
    E = cfg.feature_embedding_dimension
    c = fr.cache
    eps = np.asarray(eps, dtype=dtype)
    # integration network backward
    int_acts, integration = c["int_acts"], c["integration"]
    # loss == "external": y is the caller's d(task loss)/d(pred), already batch-scaled (custom GradientTape loops)
    if d_emb is not None:
        dz = np.zeros_like(fr.pred)           # encoder-only step: the integration network is not part of the caller's graph
    else:
        dz = np.asarray(y, dtype=dtype).reshape(fr.pred.shape) if loss == "external" else task_loss_grad(loss, fr.pred, y) / B
    dz = dz * act_grad_from_output(cfg.output_activation_fn, int_acts[-1], cfg.leaky_alpha)
    int_grads = [None] * len(integration)
    for k in reversed(range(len(integration))):
        W, _ = integration[k]
        int_grads[k] = (int_acts[k].T @ dz, dz.sum(axis=0))
        dh = dz @ W.T
        if k > 0:
            dz = dh * act_grad_from_output(cfg.activation_fn, int_acts[k], cfg.leaky_alpha)
    if d_emb is not None:     # encoder-only custom steps (nb-particle cell 8): the caller's network produced d loss / d emb
        d_emb = np.asarray(d_emb, dtype=dtype).reshape(fr.emb.shape)
        int_grads = [(np.zeros_like(W), np.zeros_like(b)) for W, b in integration]
    else:
        d_emb = dh
    enc_grads = []
    for i in range(cfg.number_features):
        acts, mu, lv, pres, masks = c["enc"][i]
        layers = c["encoders"][i]
        du = d_emb[:, i * E:(i + 1) * E]
        sig = np.exp(lv / 2.0)
        dmu = du + beta * mu / B
        dlv = du * eps[:, i, :] * 0.5 * sig + beta * 0.5 * (np.exp(lv) - 1.0) / B
        dz = np.concatenate([dmu, dlv], axis=-1)
        if cfg.encoder_kind == "simple":
            enc_grads.append([(np.sum(dmu * acts[0]).reshape(1, 1), np.sum(dlv).reshape(1, 1))])
            continue
        g = [None] * len(layers)
        for k in reversed(range(len(layers))):
            W, _ = layers[k]
            g[k] = (acts[k].T @ dz, dz.sum(axis=0))
            if k > 0:
                dh = dz @ W.T
                if masks[k] is not None:
                    dh = dh * masks[k]                               # Dropout backward: the same scale mask
                dz = dh * act_grad_from_output(cfg.activation_fn, pres[k], cfg.leaky_alpha)
        enc_grads.append(g)
    flat = []
    for g in enc_grads:
        for gw, gb in g:
            flat += [gw.ravel(), gb.ravel()]
    for gw, gb in int_grads:
        flat += [gw.ravel(), gb.ravel()]
    return np.concatenate(flat), fr


# ----------------------------------------------------------------------------------------------
# optimizer / schedule / fit
# ----------------------------------------------------------------------------------------------
@dataclass
class AdamState:
    m: np.ndarray
    v: np.ndarray
    t: int = 0


def adam_step(params, grads, st: AdamState, lr, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
    """[KERAS] tf.keras.optimizers.Adam (non-amsgrad) dense update:
        t += 1; lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v EMA; w -= lr_t * m / (sqrt(v) + eps)
    (epsilon OUTSIDE the bias correction, default 1e-7; lr from train.py:129 / nb-radial Adam(lr))."""
    st.t += 1
    dt = params.dtype.type
    lr_t = dt(lr) * dt(math.sqrt(1.0 - beta_2 ** st.t)) / dt(1.0 - beta_1 ** st.t)
    # Keras casts beta_1/beta_2 to the variable dtype first and forms (1 - beta) in that dtype
    st.m += (grads - st.m) * (dt(1.0) - dt(beta_1))
    st.v += (grads * grads - st.v) * (dt(1.0) - dt(beta_2))
    params -= lr_t * st.m / (np.sqrt(st.v) + dt(epsilon))
    return params


def sgd_step(params, grads, velocity, lr, momentum=0.0, nesterov=False):
    """[KERAS] tf.keras.optimizers.SGD: v = momentum*v - lr*g; w += momentum*v - lr*g (nesterov) or v."""
    dt = params.dtype.type
    if momentum == 0.0:
        params -= dt(lr) * grads
        return params
    velocity *= dt(momentum)
    velocity -= dt(lr) * grads
    params += (dt(momentum) * velocity - dt(lr) * grads) if nesterov else velocity
    return params


def rmsprop_step(params, grads, ms, mom, lr, rho=0.9, momentum=0.0, epsilon=1e-7):
    """[KERAS/TF] non-centered RMSprop as TensorFlow's ApplyRMSProp kernel computes it:
    ms = rho*ms + (1-rho)*g^2; mom = momentum*mom + lr*g/sqrt(ms + eps); w -= mom."""
    dt = params.dtype.type
    ms *= dt(rho)
    ms += (dt(1.0) - dt(rho)) * grads * grads
    mom *= dt(momentum)
    mom += dt(lr) * grads / np.sqrt(ms + dt(epsilon))
    params -= mom
    return params


def beta_schedule(epoch, beta_start, beta_end, number_pretraining_epochs, number_annealing_epochs):
    """models.py:147-149, evaluated in float32 like the TF ops there."""
    f = np.float32
    frac = f(max(epoch - number_pretraining_epochs, 0)) / f(number_annealing_epochs)
    return f(np.exp(np.log(f(beta_start)) + frac * (np.log(f(beta_end)) - np.log(f(beta_start)))))


def fit(cfg: DIBConfig, flat_params, x, y, *, loss, epochs, batch_size, lr,
        eps_fn: Callable[[int, np.ndarray], np.ndarray],
        perm_fn: Optional[Callable[[int, int], np.ndarray]] = None,
        beta_fn: Optional[Callable[[int], float]] = None,
        validation_data=None, dtype=np.float64, adam_kwargs=None, dropout_seed=None):
    """[KERAS] Model.fit epoch mechanics around the reference's call() (train.py:157-166):
      * per epoch: on_epoch_begin sets beta (models.py:147); indices shuffled (perm_fn(epoch, N));
        consecutive batches incl. a short last one;
      * history['loss'] = sample-weighted running mean of (task + beta*sumKL); history['accuracy']
        = sample-weighted mean; history['KL{i}'] and ['beta'] = UNWEIGHTED mean over batches
        (add_metric -> Mean with weight 1, models.py:115,121);
      * validation after every epoch with the same call() -- noise still sampled (train.py:264-265)
        -- in batches of batch_size, giving val_* twins.
    eps_fn(step, sample_ids) -> eps [n, F, E].  Noise contract of the engine: a training batch is keyed by
    (optimizer step counted from 0, ROW POSITION inside the global batch); a validation pass is keyed by
    (2**31 + epoch, row position inside the validation set).
    """
    p = np.array(flat_params, dtype=dtype, copy=True)
    st = AdamState(np.zeros_like(p), np.zeros_like(p))
    N = x.shape[0]
    F = cfg.number_features
    hist = {k: [] for k in ["loss", "accuracy", "beta"] + [f"KL{i}" for i in range(F)]}
    if validation_data is not None:
        for k in list(hist):
            hist["val_" + k] = []
    step = 0
    beta = 1.0                                                         # models.py:86
    adam_kwargs = adam_kwargs or {}
    for epoch in range(epochs):
        if beta_fn is not None:
            beta = float(beta_fn(epoch))
        perm = perm_fn(epoch, N) if perm_fn is not None else np.arange(N)
        sums = dict(loss=0.0, acc=0.0, n=0, kl=np.zeros(F), nb=0)
        for b0 in range(0, N, batch_size):
            idx = perm[b0:b0 + batch_size]
            eps = eps_fn(step, np.arange(len(idx)))
            # Dropout (nb-radial cell 5) is active in the training steps only; its masks share the step / row keying of the noise
            drop = (dropout_seed, step, np.arange(len(idx))) if (dropout_seed is not None and cfg.dropout_rate > 0) else None
            g, fr = train_grads(cfg, p, x[idx], y[idx], eps, beta, loss, dtype=dtype, dropout=drop)
            adam_step(p, g.astype(dtype), st, lr, **adam_kwargs)
            n = len(idx)
            sums["loss"] += fr.loss * n
            sums["acc"] += fr.acc_sum
            sums["n"] += n
            sums["kl"] += fr.kl_per_feature
            sums["nb"] += 1
            step += 1
        hist["loss"].append(sums["loss"] / sums["n"])
        hist["accuracy"].append(sums["acc"] / sums["n"])
        hist["beta"].append(beta)
        for i in range(F):
            hist[f"KL{i}"].append(sums["kl"][i] / sums["nb"])
        if validation_data is not None:
            xv, yv = validation_data
            vs = dict(loss=0.0, acc=0.0, n=0, kl=np.zeros(F), nb=0)
            for b0 in range(0, xv.shape[0], batch_size):
                idx = np.arange(b0, min(b0 + batch_size, xv.shape[0]))
                eps = eps_fn(2 ** 31 + epoch, idx)
                fr = forward(cfg, p, xv[idx], eps, beta, y=yv[idx], loss=loss, dtype=dtype)
                vs["loss"] += fr.loss * len(idx)
                vs["acc"] += fr.acc_sum
                vs["n"] += len(idx)
                vs["kl"] += fr.kl_per_feature
                vs["nb"] += 1
            hist["val_loss"].append(vs["loss"] / vs["n"])
            hist["val_accuracy"].append(vs["acc"] / vs["n"])
            hist["val_beta"].append(beta)
            for i in range(F):
                hist[f"val_KL{i}"].append(vs["kl"][i] / vs["nb"])
    return p, hist


# ----------------------------------------------------------------------------------------------
# compression matrices (a14)
# ----------------------------------------------------------------------------------------------
def bhattacharyya_dist_mat(mus1, logvars1, mus2, logvars2):
    """utils.py:177-212 in its O(N*M*E) closed form (the reference materialises N*M*E*E diagonals):
       D = 1/8 sum_e (mu1-mu2)^2/sbar + 1/2 [ sum_e ln sbar - 1/2 (sum lv1 + sum lv2) ],
       sbar = (exp(lv1)+exp(lv2))/2."""
    mus1, logvars1, mus2, logvars2 = [np.asarray(a, dtype=np.float64) for a in (mus1, logvars1, mus2, logvars2)]
    d = mus1[:, None, :] - mus2[None, :, :]
    sbar = 0.5 * (np.exp(logvars1)[:, None, :] + np.exp(logvars2)[None, :, :])
    term1 = 0.125 * (d * d / sbar).sum(-1)
    term2 = 0.5 * (np.log(sbar).sum(-1) - 0.5 * (logvars1.sum(-1)[:, None] + logvars2.sum(-1)[None, :]))
    return term1 + term2


def kl_divergence_mat(mus1, logvars1, mus2, logvars2):
    """utils.py:213-247 in closed form: KL(N1_i || N2_j) =
       1/2 [ sum lv2_j - sum lv1_i - E + sum_e exp(lv1_i - lv2_j) + sum_e (mu2_j - mu1_i)^2 exp(-lv2_j) ]."""
    mus1, logvars1, mus2, logvars2 = [np.asarray(a, dtype=np.float64) for a in (mus1, logvars1, mus2, logvars2)]
    E = mus1.shape[1]
    d = mus2[None, :, :] - mus1[:, None, :]
    term1 = np.exp(logvars1[:, None, :] - logvars2[None, :, :]).sum(-1)
    term2 = (d * d * np.exp(-logvars2)[None, :, :]).sum(-1)
    return 0.5 * (logvars2.sum(-1)[None, :] - logvars1.sum(-1)[:, None] - E + term1 + term2)


def compression_matrices(cfg: DIBConfig, flat_params, x, row_index=None, dtype=np.float64):
    """visualization.save_compression_matrices (visualization.py:14-35) for every feature: rows row_index[i] of x
    -> encoder i -> Bhattacharyya -> exp(-D).  Returns (mu_logvar [F,n,2E], dist [F,n,n], comp [F,n,n])."""
    encoders, _ = unflatten(cfg, np.asarray(flat_params, dtype=dtype))
    x = np.asarray(x, dtype=dtype)
    E = cfg.feature_embedding_dimension
    offs = np.cumsum([0] + list(cfg.feature_dimensionalities))
    outs, dists = [], []
    for i in range(cfg.number_features):
        rows = x if row_index is None else x[np.asarray(row_index[i])]
        o = encoder_forward(cfg, encoders[i], rows[:, offs[i]:offs[i + 1]])
        outs.append(o)
        dists.append(bhattacharyya_dist_mat(o[:, :E], o[:, E:], o[:, :E], o[:, E:]))
    dists = np.stack(dists)
    return np.stack(outs), dists, np.exp(-dists)


def compression_matrix(cfg: DIBConfig, flat_params, feature_ind, x_rows, dtype=np.float64):
    """visualization.py:31-34: encoder forward (no noise) -> Bhattacharyya -> exp(-D)."""
    encoders, _ = unflatten(cfg, np.asarray(flat_params, dtype=dtype))
    o = encoder_forward(cfg, encoders[feature_ind], np.asarray(x_rows, dtype=dtype))
    E = cfg.feature_embedding_dimension
    mu, lv = o[:, :E], o[:, E:]
    return np.exp(-bhattacharyya_dist_mat(mu, lv, mu, lv))


# ----------------------------------------------------------------------------------------------
# next row f3: InfoNCE head of the custom training loop (train.py:201-213, utils.py:75-175)
# ----------------------------------------------------------------------------------------------
SIMILARITY_TYPES = ("l2sq", "l2", "l1", "linf", "cosine")


def get_scaled_similarity(embeddings1, embeddings2, similarity_type, temperature):
    """utils.py:127-175 (+ the pairwise distances utils.py:75-125): [N, d], [M, d] -> [N, M] similarities / temperature."""
    a, b = np.asarray(embeddings1, dtype=np.float64), np.asarray(embeddings2, dtype=np.float64)
    diff = a[:, None, :] - b[None, :, :]
    if similarity_type in ("l2sq", "l2"):
        # the reference expands |a|^2 + |b|^2 - 2ab and clamps at 0 (utils.py:85-90)
        d2 = np.maximum((a * a).sum(-1)[:, None] + (b * b).sum(-1)[None, :] - 2.0 * a @ b.T, 0.0)
        sim = -d2 if similarity_type == "l2sq" else -np.sqrt(d2 + 1e-9)
    elif similarity_type == "l1":
        sim = -np.abs(diff).sum(-1)
    elif similarity_type == "linf":
        sim = -np.abs(diff).max(-1)
    elif similarity_type == "cosine":
        sim = (a / np.linalg.norm(a, axis=-1, keepdims=True)) @ (b / np.linalg.norm(b, axis=-1, keepdims=True)).T
    else:
        raise ValueError(f"Similarity type not implemented: {similarity_type}")
    return sim / temperature


def _logsumexp(s, axis):
    m = s.max(axis=axis, keepdims=True)
    return (m + np.log(np.exp(s - m).sum(axis=axis, keepdims=True))).squeeze(axis)


def infonce_loss_and_grads(embeddings1, embeddings2, similarity_type, temperature):
    """train.py:203-213: S = get_scaled_similarity(e1, e2); loss = mean_i CE(i, S[i,:]) + mean_i CE(i, S^T[i,:]).
    Returns (loss, d loss/d e1, d loss/d e2, S) with the analytic reverse mode GradientTape would produce."""
    a, b = np.asarray(embeddings1, dtype=np.float64), np.asarray(embeddings2, dtype=np.float64)
    n = a.shape[0]
    assert b.shape[0] == n, "the InfoNCE loss needs full, equal batches (train.py:222-223)"
    T = float(temperature)
    S = get_scaled_similarity(a, b, similarity_type, T)
    row, col = _logsumexp(S, 1), _logsumexp(S, 0)
    diag = np.diag(S)
    loss = float((row - diag).mean() + (col - diag).mean())
    dS = (np.exp(S - row[:, None]) + np.exp(S - col[None, :]) - 2.0 * np.eye(n)) / n
    diff = a[:, None, :] - b[None, :, :]
    if similarity_type == "l2sq":
        g = -2.0 * diff / T                                          # d s_ij / d a_i  (= -d s_ij / d b_j)
    elif similarity_type == "l2":
        g = -diff / (-S * T)[:, :, None] / T                         # sqrt(d2 + eps) = -S T
    elif similarity_type == "l1":
        g = -np.sign(diff) / T
    elif similarity_type == "linf":
        k = np.abs(diff).argmax(-1)
        g = np.zeros_like(diff)
        ii, jj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        g[ii, jj, k] = -np.sign(diff[ii, jj, k]) / T
    if similarity_type == "cosine":
        na, nb = np.linalg.norm(a, axis=-1), np.linalg.norm(b, axis=-1)
        ah, bh = a / na[:, None], b / nb[:, None]
        c = ah @ bh.T
        ga = (bh[None, :, :] - c[:, :, None] * ah[:, None, :]) / na[:, None, None] / T
        gb = (ah[:, None, :] - c[:, :, None] * bh[None, :, :]) / nb[None, :, None] / T
    else:
        ga, gb = g, -g
    return loss, np.einsum("ij,ijk->ik", dS, ga), np.einsum("ij,ijk->jk", dS, gb), S


# ----------------------------------------------------------------------------------------------
# fixture: the paper's Boolean circuit (data.py:21-57) -- deterministic known answer
# ----------------------------------------------------------------------------------------------
def boolean_circuit_truth_table():
    spec = [[1, 0, 1], [2, 8, 7], [0, 4, 3], [1, 11, 5], [2, 6, 12], [2, 13, 9], [1, 14, 10],
            [0, 15, 2], [0, 17, 16]]                                   # data.py:40
    gates = [np.logical_and, np.logical_or, np.logical_xor]            # data.py:25
    grids = np.meshgrid(*[[0, 1]] * 10)                                # data.py:50-52
    tt = np.stack(grids, -1).reshape(-1, 10)
    for g, a, b in spec:
        tt = np.concatenate([tt, gates[g](tt[:, a], tt[:, b]).astype(np.int32)[:, None]], -1)
    x = 2 * tt[:, :10] - 1                                             # data.py:56
    y = tt[:, -1]
    return x.astype(np.float32), y.astype(np.float32)


# ----------------------------------------------------------------------------------------------
# next row f1: InfoNCE / leave-one-out sandwich bounds on I(U;X) of one encoder (utils.py:10-73)
# ----------------------------------------------------------------------------------------------
def mi_sandwich_batch(mu, logvar, eps):
    """utils.py:36-65 ``compute_batch`` with the sample u = mu + exp(logvar/2)*eps explicit, evaluated in log space
    (the reference forms the densities directly in float64; identical up to underflow):
        log p(u_i|x_j) = -1/2 sum_e ((u_i - mu_j)/sigma_j)^2 - 1/2 sum_e logvar_j - E/2 log(2 pi)          (:48-57)
        InfoNCE lower  = mean_i [ log p_ii - log mean_j p_ij ]                                            (:59-61)
        LOO upper      = mean_i [ log p_ii - log ( (1/bs) sum_{j != i} p_ij ) ]    (diagonal zeroed, still /bs; :63-64)
    Returns (lower, upper) in nats."""
    mu, logvar, eps = [np.asarray(a, dtype=np.float64) for a in (mu, logvar, eps)]
    bs, E = mu.shape
    sig = np.exp(logvar / 2.0)
    u = mu + sig * eps
    nd = (u[:, None, :] - mu[None, :, :]) / sig[None, :, :]
    logp = -0.5 * (nd ** 2).sum(-1) - 0.5 * logvar.sum(-1)[None, :] - 0.5 * E * np.log(2.0 * np.pi)
    diag = np.diag(logp)

    def lse(a):
        m = a.max(axis=1, keepdims=True)
        return (m + np.log(np.exp(a - m).sum(axis=1, keepdims=True)))[:, 0]
    lower = np.mean(diag - (lse(logp) - np.log(bs)))
    off = logp.copy()
    off[np.arange(bs), np.arange(bs)] = -np.inf
    upper = np.mean(diag - (lse(off) - np.log(bs)))
    return float(lower), float(upper)


def estimate_mi_sandwich_bounds(cfg: DIBConfig, flat_params, feature_ind, x_i, batches, eps_list, dtype=np.float64):
    """utils.py:10-73: average of compute_batch over the given batches (lists of row indices into x_i) with the given
    noise; the reference draws the batches with an unseeded tf.data shuffle, so batch composition is an input here."""
    encoders, _ = unflatten(cfg, np.asarray(flat_params, dtype=dtype))
    E = cfg.feature_embedding_dimension
    out = []
    for idx, eps in zip(batches, eps_list):
        o = encoder_forward(cfg, encoders[feature_ind], np.asarray(x_i, dtype=dtype)[idx])
        out.append(mi_sandwich_batch(o[:, :E], o[:, E:], eps))
    return np.mean(np.asarray(out), axis=0)
