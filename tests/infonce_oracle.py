"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the reference's InfoNCE training path (train.py:180-289) on top of
oracle.dib_oracle: the output encoder (train.py:186-193), one eval_batch_infonce(training=True) step minus the optimizer
(train.py:201-219) and the fit mechanics of compile(loss=InfoNCE) + fit (dib_b200.models.DistributedIBNet._fit_infonce)."""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import numpy as np

from oracle import dib_oracle as O


@dataclass
class OutputEncoderConfig:
    """train.py:186-193: Input((dy,)) -> [PositionalEncoding] -> Dense(w, activation_fn) per width -> Dense(D)."""
    input_dimensionality: int
    architecture: Sequence[int] = field(default_factory=lambda: [128, 128])


def output_encoder_param_shapes(cfg: O.DIBConfig, ocfg: OutputEncoderConfig):
    """Keras order [W0, b0, W1, b1, ...] with [in, out] kernels; the input width is dy * (1 + len(frequencies)) when the
    model uses positional encoding (the same frequencies, train.py:188), and the last width is output_dimensionality."""
    din = ocfg.input_dimensionality * (1 + len(cfg.frequencies)) if cfg.use_positional_encoding else ocfg.input_dimensionality
    dims = [din] + list(ocfg.architecture) + [cfg.output_dimensionality]
    shapes = []
    for k in range(len(dims) - 1):
        shapes += [(dims[k], dims[k + 1]), (dims[k + 1],)]
    return shapes


def output_encoder_glorot(cfg, ocfg, rng, dtype=np.float32):
    out = []
    for s in output_encoder_param_shapes(cfg, ocfg):
        if len(s) == 2:
            lim = math.sqrt(6.0 / (s[0] + s[1]))
            out.append(rng.uniform(-lim, lim, size=s).astype(dtype).ravel())
        else:
            out.append(np.zeros(s, dtype=dtype))
    return np.concatenate(out)


def _layers(cfg, ocfg, q):
    views, off = [], 0
    for s in output_encoder_param_shapes(cfg, ocfg):
        n = int(np.prod(s))
        views.append(q[off:off + n].reshape(s))
        off += n
    assert off == q.size
    return [(views[2 * k], views[2 * k + 1]) for k in range(len(views) // 2)]


def output_encoder_forward(cfg: O.DIBConfig, ocfg: OutputEncoderConfig, q, y, keep=False, dtype=np.float64):
    """output_encoder(y) (train.py:186-193).  With ``keep``: (e2, acts) where acts[k] is the input of layer k."""
    q = np.asarray(q, dtype=dtype)
    y = np.asarray(y, dtype=dtype).reshape(-1, ocfg.input_dimensionality)
    h = O.positional_encoding(y, cfg.frequencies) if cfg.use_positional_encoding else y
    layers = _layers(cfg, ocfg, q)
    acts = [h]
    for k, (W, b) in enumerate(layers):
        z = h @ W + b
        h = O.act_fwd(cfg.activation_fn, z, cfg.leaky_alpha) if k < len(layers) - 1 else z
        acts.append(h)
    return (h, acts) if keep else h


def output_encoder_backward(cfg: O.DIBConfig, ocfg: OutputEncoderConfig, q, acts, d_e2, dtype=np.float64):
    """Reverse mode of output_encoder_forward from d e2: the flat gradient in Keras order."""
    layers = _layers(cfg, ocfg, np.asarray(q, dtype=dtype))
    dz = np.asarray(d_e2, dtype=dtype)
    g = [None] * len(layers)
    for k in reversed(range(len(layers))):
        W, _ = layers[k]
        g[k] = (acts[k].T @ dz, dz.sum(axis=0))
        if k > 0:
            dz = (dz @ W.T) * O.act_grad_from_output(cfg.activation_fn, acts[k], cfg.leaky_alpha)
    return np.concatenate([a.ravel() for gw, gb in g for a in (gw, gb)])


def infonce_train_grads(cfg: O.DIBConfig, ocfg: OutputEncoderConfig, p, q, x, y, eps, beta, kind, T, dtype=np.float64):
    """eval_batch_infonce(training=True) minus apply_gradients (train.py:201-219): e1 = model(x) with noise eps, e2 =
    output_encoder(y), loss = InfoNCE(e1, e2) + beta * sum_i KL_i.  Returns (d loss / d p, d loss / d q, InfoNCE loss,
    ForwardResult of the model)."""
    e1 = O.forward(cfg, p, x, eps, beta, dtype=dtype).pred
    e2, acts = output_encoder_forward(cfg, ocfg, q, y, keep=True, dtype=dtype)
    loss, d_e1, d_e2, _ = O.infonce_loss_and_grads(e1, e2, kind, T)
    gp, fr = O.train_grads(cfg, p, x, d_e1, eps, beta, "external", dtype=dtype)
    gq = output_encoder_backward(cfg, ocfg, q, acts, d_e2, dtype=dtype)
    return gp, gq, loss, fr


def infonce_forward(cfg, ocfg, p, q, x, y, eps, beta, kind, T, dtype=np.float64):
    """eval_batch_infonce(training=False): (InfoNCE loss, ForwardResult)."""
    fr = O.forward(cfg, p, x, eps, beta, dtype=dtype)
    e2 = output_encoder_forward(cfg, ocfg, q, y, dtype=dtype)
    loss, _, _, _ = O.infonce_loss_and_grads(fr.pred, e2, kind, T)
    return loss, fr


def epoch_boundaries(N, B, epochs):
    """r(e) = np.round(e N / B): the first optimizer step of epoch e (train.py:222-236's repeated stream)."""
    return [int(np.round(e * N / B)) for e in range(epochs + 1)]


def fit_infonce(cfg: O.DIBConfig, ocfg: OutputEncoderConfig, p, q, x, y, *, kind, T, epochs, batch_size, lr,
                eps_fn: Callable[[int, np.ndarray], np.ndarray],
                perm_fn: Optional[Callable[[int, int], np.ndarray]] = None,
                beta_fn: Optional[Callable[[int], float]] = None,
                validation_data=None, dtype=np.float64, adam_kwargs=None):
    """compile(loss=InfoNCE) + fit:
      * full batches only: step s reads rows [sB, (s+1)B) of perm_0 || perm_1 || ... (perm_fn(k, N), or arange(N));
      * epoch e runs steps [r(e), r(e+1)), r(e) = np.round(e N / B);
      * beta from beta_fn(epoch) at the start of the epoch (the Keras callback; train.py:241-250 switches after the epoch's
        first step instead);
      * ONE Adam state over [p || q] (train.py:219 applies one apply_gradients to all variables: one iteration count);
      * history: loss = mean over batches of (InfoNCE + beta sum KL), KL{i}, beta, and val_ twins from floor(Nv/B) + 1
        full batches of consecutive rows of the repeated validation set, noise keyed (2**31 + epoch, stream position).
    Returns (p, q, history, number of optimizer steps)."""
    P = len(p)
    w = np.concatenate([np.asarray(p, dtype=dtype), np.asarray(q, dtype=dtype)])
    st = O.AdamState(np.zeros_like(w), np.zeros_like(w))
    N, B, F = x.shape[0], batch_size, cfg.number_features
    hist = {k: [] for k in ["loss", "beta"] + [f"KL{i}" for i in range(F)]}
    if validation_data is not None:
        for k in list(hist):
            hist["val_" + k] = []
    r = epoch_boundaries(N, B, epochs)
    beta = 1.0
    perms = {}

    def rows(s):
        ids = np.arange(s * B, (s + 1) * B)
        out = np.empty(B, dtype=np.int64)
        for j, g in enumerate(ids):
            k, i = divmod(int(g), N)
            if k not in perms:
                perms[k] = np.asarray(perm_fn(k, N)) if perm_fn is not None else np.arange(N)
            out[j] = perms[k][i]
        return out

    step = 0
    for epoch in range(epochs):
        if beta_fn is not None:
            beta = float(beta_fn(epoch))
        sums = dict(loss=0.0, kl=np.zeros(F), nb=0)
        for s in range(r[epoch], r[epoch + 1]):
            idx = rows(s)
            eps = eps_fn(step, np.arange(B))
            gp, gq, loss, fr = infonce_train_grads(cfg, ocfg, w[:P], w[P:], x[idx], y[idx], eps, beta, kind, T, dtype=dtype)
            O.adam_step(w, np.concatenate([gp, gq]).astype(dtype), st, lr, **(adam_kwargs or {}))
            sums["loss"] += loss + beta * float(np.sum(fr.kl_per_feature))
            sums["kl"] += fr.kl_per_feature
            sums["nb"] += 1
            step += 1
        hist["loss"].append(sums["loss"] / sums["nb"])
        hist["beta"].append(beta)
        for i in range(F):
            hist[f"KL{i}"].append(sums["kl"][i] / sums["nb"])
        if validation_data is not None:
            xv, yv = validation_data
            Nv = xv.shape[0]
            vs = dict(loss=0.0, kl=np.zeros(F), nb=0)
            for b in range(Nv // B + 1):
                pos = np.arange(b * B, (b + 1) * B)
                idx = pos % Nv
                loss, fr = infonce_forward(cfg, ocfg, w[:P], w[P:], xv[idx], yv[idx], eps_fn(2 ** 31 + epoch, pos), beta, kind,
                                           T, dtype=dtype)
                vs["loss"] += loss + beta * float(np.sum(fr.kl_per_feature))
                vs["kl"] += fr.kl_per_feature
                vs["nb"] += 1
            hist["val_loss"].append(vs["loss"] / vs["nb"])
            hist["val_beta"].append(beta)
            for i in range(F):
                hist[f"val_KL{i}"].append(vs["kl"][i] / vs["nb"])
    return w[:P], w[P:], hist, step


def infonce_case_params(cfg: O.DIBConfig, ocfg: OutputEncoderConfig, seed: int):
    """Weights of a ref_infonce_step.npz case: the model's as O.golden_case_params (glorot kernels, N(0, 0.05^2) biases),
    then the output encoder's from the same generator (glorot kernels, N(0, 0.05^2) biases).  Returns (p, q, rng)."""
    p, rng = O.golden_case_params(cfg, seed)
    q = output_encoder_glorot(cfg, ocfg, rng, dtype=np.float32)
    q = q + (rng.standard_normal(q.size) * 0.05).astype(np.float32) * (q == 0)
    return p, q, rng


def load_infonce_golden(path):
    """{case name: (cfg, ocfg, arrays)} of tests/golden/ref_infonce_step.npz; the weights are regenerated from the seed and
    checked against the SHA-256 the golden was computed with."""
    import ast
    import hashlib
    z = dict(np.load(path))
    out = {}
    for name in z["cases"]:
        a = {k.split("__", 1)[1]: v for k, v in z.items() if k.startswith(f"{name}__")}
        cfg = O.DIBConfig(**ast.literal_eval(str(a["cfg"])))
        ocfg = OutputEncoderConfig(**ast.literal_eval(str(a["ocfg"])))
        p, q, _ = infonce_case_params(cfg, ocfg, int(a["seed"]))
        if hashlib.sha256(np.concatenate([p, q]).tobytes()).hexdigest() != str(a["params_sha256"]):
            raise RuntimeError(f"{path}:{name}: the weights regenerated from seed {int(a['seed'])} are not the golden's")
        a["p"], a["q"] = p, q
        out[str(name)] = (cfg, ocfg, a)
    return out
