"""Golden vectors for the InfoNCE training path (train.py:180-289) by executing the REFERENCE'S OWN CODE on the numpy tf
stand-in of make_golden.py: train.py's output-encoder construction (train.py:186-193) and its eval_batch_infonce
(train.py:201-219) are cut out of train.py's text and exec'd verbatim, with the reference's models.DistributedIBNet and
utils.get_scaled_similarity imported unmodified.  The golden uses training=False, so GradientTape.gradient is never
called.  Additions to the stand-in:
  * tf.range, tf.transpose, a no-op tf.function, a GradientTape context whose gradient() raises;
  * [KERAS] tf.keras.losses.sparse_categorical_crossentropy(labels, logits, from_logits=True) = log-softmax CE per row;
  * [KERAS] Layer.__call__ drops the `training` argument for layers whose call() does not take it, and `list / Variable`
    divides elementwise (kl_loss / model.beta, train.py:220).
`args` supplies infonce_space_dimensionality, the name train.py:116,192 reads but never defines.

Run here (needs /root/reference; never on the GPU box):   python tests/golden/make_infonce_golden.py
Writes tests/golden/ref_infonce_step.npz (committed).  Weights are not stored: each case keeps its seed and the SHA-256 of
[model weights | output-encoder weights] (tests/infonce_oracle.py :: infonce_case_params / load_infonce_golden)."""
import hashlib
import inspect
import os
import sys
import textwrap
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "..", ".."))
import make_golden as G                                                # noqa: E402
from oracle import dib_oracle as O                                     # noqa: E402
from tests import infonce_oracle as NO                                 # noqa: E402

TRAIN = os.path.join(G.REF, "train.py")

CASES = [   # (name, y width, similarity, temperature, use PE, seed)
    ("y6_l2", 6, "l2", 0.7, True, 51),
    ("y1_cosine", 1, "cosine", 1.3, True, 52),
    ("y6_cosine_nope", 6, "cosine", 0.5, False, 53),
    ("y1_l2", 1, "l2", 1.0, True, 54),
]


def _sparse_ce_from_logits(labels, logits, from_logits=False):
    """[KERAS] sparse_categorical_crossentropy(from_logits=True): -log_softmax(logits)[label] per row."""
    assert from_logits
    z = np.asarray(logits, dtype=np.float64)
    m = z.max(axis=-1, keepdims=True)
    lse = (m + np.log(np.exp(z - m).sum(axis=-1, keepdims=True)))[:, 0]
    return lse - z[np.arange(z.shape[0]), np.asarray(labels).astype(np.int64)]


class _Tape:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def gradient(self, *a, **k):
        raise AssertionError("the golden runs eval_batch_infonce(training=False)")


def _extract(src):
    a = src.index("    output_encoder_layers = [tf.keras.layers.Input(")
    b = src.index("    output_encoder = tf.keras.Sequential(output_encoder_layers)")
    b = src.index("\n", b) + 1
    c = src.index("    @tf.function\n    def eval_batch_infonce(")
    d = src.index("      return loss_infonce, kl_loss / model.beta", c)
    d = src.index("\n", d) + 1
    return textwrap.dedent(src[a:b]), textwrap.dedent(src[c:d])


def main():
    models, utils = G.load_reference()
    tf = sys.modules["tensorflow"]
    tf.range = np.arange
    tf.transpose = np.transpose
    tf.GradientTape = _Tape
    tf.keras.losses = types.SimpleNamespace(sparse_categorical_crossentropy=_sparse_ce_from_logits)

    layer_call = G._Layer.__call__

    def _call(self, x, *a, **k):                                     # [KERAS] `training` only reaches calls that take it
        if "training" in k and "training" not in inspect.signature(self.call).parameters:
            k = {kk: v for kk, v in k.items() if kk != "training"}
        return layer_call(self, x, *a, **k)

    G._Layer.__call__ = _call
    G._Variable.__rtruediv__ = lambda self, o: np.asarray(o) / self._v
    G._Sequential.call = lambda self, x, training=None: _seq(self, x)

    oe_src, eval_src = _extract(open(TRAIN).read())
    out = {}
    for name, dy, kind, T, use_pe, seed in CASES:
        cfg_kwargs = dict(feature_dimensionalities=[2, 1, 2, 1], feature_encoder_architecture=[16, 8],
                          integration_network_architecture=[12], output_dimensionality=5,
                          use_positional_encoding=use_pe, number_positional_encoding_frequencies=3,
                          activation_fn="relu", feature_embedding_dimension=4, output_activation_fn=None)
        cfg = O.DIBConfig(**cfg_kwargs)
        ocfg = NO.OutputEncoderConfig(dy, [10, 7])
        p, q, rng = NO.infonce_case_params(cfg, ocfg, seed)
        B, beta = 9, 0.02
        x = rng.standard_normal((B, 6)).astype(np.float32)
        y = rng.standard_normal((B, dy)).astype(np.float32)
        eps = rng.standard_normal((B, cfg.number_features, cfg.feature_embedding_dimension)).astype(np.float32)

        ref = dict(cfg_kwargs)
        fd, fea, ina, od = (ref.pop(k) for k in ("feature_dimensionalities", "feature_encoder_architecture",
                                                 "integration_network_architecture", "output_dimensionality"))
        model = models.DistributedIBNet(fd, fea, ina, od, **ref)            # train.py:118-126
        G.inject_weights(model, cfg, p)
        model.beta.assign(beta)
        args = types.SimpleNamespace(infonce_y_encoder_architecture=list(ocfg.architecture), infonce_space_dimensionality=od,
                                     infonce_similarity=kind, infonce_temperature=T)
        ns = dict(tf=tf, np=np, models=models, utils=utils, args=args, activation_fn="relu",
                  use_positional_encoding=use_pe, number_positional_encoding_frequencies=3,
                  dataset_dict={"y_train": y}, model=model, batch_size=B, optimizer=None, all_trainable_variables=None)
        exec(oe_src, ns)                                                    # train.py:186-193, verbatim
        dense = [l for l in ns["output_encoder"].layers if isinstance(l, G._Dense)]
        off = 0
        for l, (ws, bs) in zip(dense, zip(*[iter(NO.output_encoder_param_shapes(cfg, ocfg))] * 2)):
            assert l.units == ws[1]
            l.kernel = q[off:off + ws[0] * ws[1]].reshape(ws).astype(np.float64); off += ws[0] * ws[1]
            l.bias = q[off:off + bs[0]].astype(np.float64); off += bs[0]
        assert off == q.size
        exec(eval_src, ns)                                                  # train.py:201-219, verbatim
        feed = lambda: setattr(G.EPS, "q", [eps[:, i, :].astype(np.float64) for i in range(cfg.number_features)])
        feed()
        model.losses = []
        loss_infonce, kl = ns["eval_batch_infonce"](x.astype(np.float64), y.astype(np.float64), training=False)
        assert not G.EPS.q
        feed()
        model.losses = []
        e1 = np.asarray(model(x.astype(np.float64)))
        e2 = np.asarray(ns["output_encoder"](y.astype(np.float64)))
        digest = hashlib.sha256(np.concatenate([p, q]).tobytes()).hexdigest()
        for k, v in dict(cfg=np.array(repr(cfg_kwargs)), ocfg=np.array(repr(dict(input_dimensionality=dy,
                         architecture=list(ocfg.architecture)))), kind=np.array(kind), temperature=np.float64(T),
                         seed=np.int64(seed), params_sha256=np.array(digest), beta=np.float32(beta), x=x, y=y, eps=eps,
                         e1=e1, e2=e2, loss_infonce=np.float64(loss_infonce), kl=np.asarray(kl, np.float64).ravel()).items():
            out[f"{name}__{k}"] = v
        print(f"{name}: loss_infonce={float(loss_infonce):.6f} kl={np.asarray(kl).ravel()[:2]} e2[0,:2]={e2[0, :2]}")
    out["cases"] = np.array([c[0] for c in CASES])
    np.savez_compressed(os.path.join(HERE, "ref_infonce_step.npz"), **out)


def _seq(self, x):
    for l in self.layers:
        x = l(x)
    return x


if __name__ == "__main__":
    main()
