"""Generate golden vectors by executing the REFERENCE'S OWN CODE on a numpy stand-in for ``tf``.

TensorFlow is not installed in this image, so the reference cannot be run as shipped.  What can
be done, and is done here, is to import /root/reference/models.py and /root/reference/utils.py
unmodified with a tiny numpy-backed ``tensorflow`` module in ``sys.modules`` that provides just
the symbols those files touch (tf.split/concat/exp/..., tf.keras.layers.Dense, Sequential,
Model.add_loss/add_metric, tf.random.normal fed from an explicit epsilon queue).  Everything
that is *reference logic* -- layer construction order (models.py:56-86), the forward pass, KL,
beta-scaled loss assembly and metric names (models.py:96-123), the beta schedule
(models.py:147-149) and utils.bhattacharyya_dist_mat (utils.py:177-212) -- is therefore executed
from the reference files themselves; only the third-party arithmetic primitives are numpy.

Run here (needs /root/reference; never run on the GPU box):
    python tests/golden/make_golden.py
Writes tests/golden/*.npz, which are committed.
"""
import hashlib
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
DT = np.float64


# ------------------------------------------------------------------------------------------
# numpy stand-in for the handful of tf symbols the reference's models.py / utils.py touch
# ------------------------------------------------------------------------------------------
class _EpsQueue:
    """tf.random.normal(shape, mean, stddev) == mean + stddev * eps with eps popped from here."""
    def __init__(self):
        self.q = []
        self.used = []

    def pop(self, shape):
        e = self.q.pop(0)
        assert tuple(e.shape) == tuple(shape), (e.shape, shape)
        self.used.append(e)
        return e


EPS = _EpsQueue()


class _Variable:
    def __init__(self, value, dtype=None, trainable=True):
        self._v = np.asarray(value, dtype=np.float32 if dtype is None else dtype)

    def assign(self, v):
        self._v = np.asarray(v, dtype=self._v.dtype)

    def value(self):
        return self._v

    def numpy(self):
        return self._v

    def __mul__(self, o):
        return self._v * o

    __rmul__ = __mul__

    def __float__(self):
        return float(self._v)

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self._v, dtype=dtype)


class _Layer:
    def __init__(self, *a, **k):
        pass

    def __call__(self, x, *a, **k):
        return self.call(x, *a, **k)


class _Input:
    def __init__(self, shape):
        self.shape = shape


_ACT = {None: lambda z: z, "relu": lambda z: np.maximum(z, 0), "tanh": np.tanh,
        "sigmoid": lambda z: 1 / (1 + np.exp(-z)),
        "leaky_relu": lambda z: np.where(z > 0, z, 0.2 * z)}


class _Dense(_Layer):
    def __init__(self, units, activation=None):
        self.units, self.activation = units, activation
        self.kernel = self.bias = None

    def call(self, x):
        assert self.kernel is not None, "weights are injected by the golden script"
        return _ACT[self.activation](x @ self.kernel + self.bias)


class _Sequential(_Layer):
    def __init__(self, layers):
        self.layers = [l for l in layers if not isinstance(l, _Input)]

    def build(self, *a, **k):
        pass

    def call(self, x):
        for l in self.layers:
            x = l(x)
        return x


class _Model(_Layer):
    def __init__(self):
        self.losses, self.metrics_log = [], {}

    def add_loss(self, v):
        self.losses.append(np.asarray(v))

    def add_metric(self, v, name=None):
        self.metrics_log[name] = np.asarray(v.value() if isinstance(v, _Variable) else v)


class _Callback:
    model = None


def _split(x, sizes, axis=-1):
    if isinstance(sizes, int):
        return np.split(x, sizes, axis=axis)
    return np.split(x, np.cumsum(sizes)[:-1], axis=axis)


class _Dataset:
    """tf.data.Dataset stand-in: repeat/shuffle/batch/take over the rows of an array; the (random, unseeded in the
    reference) shuffle is replaced by the identity so that the batches are the consecutive row blocks."""
    def __init__(self, arr, bs=None, n=None):
        self.arr, self.bs, self.n = arr, bs, n

    def repeat(self): return self
    def shuffle(self, _): return self
    def batch(self, bs): return _Dataset(self.arr, bs, self.n)
    def take(self, n): return _Dataset(self.arr, self.bs, n)

    def __iter__(self):
        N = self.arr.shape[0]
        for b in range(self.n):
            idx = (np.arange(self.bs) + b * self.bs) % N
            yield self.arr[idx]


def _random_normal(shape, mean=0.0, stddev=1.0, dtype=None):
    return mean + stddev * EPS.pop(tuple(int(s) for s in shape))


def install_tf_shim():
    tf = types.ModuleType("tensorflow")
    tf.float32, tf.float64 = np.float32, np.float64
    tf.concat = lambda xs, axis: np.concatenate(xs, axis=axis)
    tf.split = _split
    tf.exp, tf.square = np.exp, np.square
    tf.reduce_mean = lambda x, axis=None: np.mean(x, axis=axis)
    tf.reduce_sum = lambda x, axis=None, keepdims=False: np.sum(np.asarray(x), axis=axis, keepdims=keepdims)
    tf.reduce_max = lambda x, axis=None: np.max(np.asarray(x), axis=axis)
    tf.expand_dims = lambda x, axis: np.expand_dims(x, axis)
    tf.maximum, tf.abs, tf.sqrt = np.maximum, np.abs, np.sqrt
    tf.matmul = lambda a, b, transpose_b=False: np.matmul(a, np.swapaxes(b, -1, -2) if transpose_b else b)
    tf.tile = lambda x, reps: np.tile(x, [int(r) for r in reps])
    tf.shape = lambda x: x.shape
    tf.cast = lambda x, dt: np.asarray(x).astype(dt)
    tf.Variable = _Variable
    tf.function = lambda f=None, **k: f if f is not None else (lambda g: g)
    tf.math = types.SimpleNamespace(sin=np.sin, log=lambda v: np.log(v) if isinstance(v, np.ndarray) and v.dtype == np.float64
                                    else np.log(np.float32(v)))
    tf.reshape = lambda x, shape: np.reshape(x, [int(s) for s in shape])
    tf.eye = lambda n, dtype=None: np.eye(int(n), dtype=dtype)
    def _normalize(x, ord=2, axis=-1):
        assert ord == 2
        nrm = np.sqrt(np.sum(np.square(x), axis=axis, keepdims=True))
        return x / nrm, nrm
    tf.linalg = types.SimpleNamespace(diag_part=lambda x: np.diag(x).copy(),   # tf tensors are immutable: no view
                                      normalize=_normalize)
    tf.random = types.SimpleNamespace(normal=_random_normal)
    keras = types.SimpleNamespace(
        layers=types.SimpleNamespace(Layer=_Layer, Input=_Input, Dense=_Dense),
        Sequential=_Sequential, Model=_Model,
        callbacks=types.SimpleNamespace(Callback=_Callback))
    tf.keras = keras
    sys.modules["tensorflow"] = tf
    return tf


def load_reference():
    install_tf_shim()
    sys.path.insert(0, REF)
    import importlib
    utils = importlib.import_module("utils")
    models = importlib.import_module("models")
    sys.path.remove(REF)
    assert os.path.dirname(models.__file__) == REF
    return models, utils


# ------------------------------------------------------------------------------------------
def inject_weights(model, cfg, flat, dtype=DT):
    off = 0
    shapes = iter(cfg.param_shapes())
    for enc in list(model.feature_encoders) + [model.integration_network]:
        for l in enc.layers:
            if isinstance(l, _Dense):
                ws, bs = next(shapes), next(shapes)
                assert ws[1] == l.units == bs[0]
                nW, nb = int(np.prod(ws)), int(np.prod(bs))
                l.kernel = flat[off:off + nW].reshape(ws).astype(dtype)
                off += nW
                l.bias = flat[off:off + nb].astype(dtype)
                off += nb
    assert off == flat.size


def run_case(models, name, cfg_kwargs, B, beta, seed):
    sys.path.insert(0, os.path.join(HERE, "..", ".."))
    from oracle import dib_oracle as O
    cfg = O.DIBConfig(**cfg_kwargs)
    flat, rng = O.golden_case_params(cfg, seed)
    D = int(np.sum(cfg.feature_dimensionalities))
    x = rng.standard_normal((B, D)).astype(np.float32)
    eps = rng.standard_normal((B, cfg.number_features, cfg.feature_embedding_dimension)).astype(np.float32)

    ref_kwargs = dict(cfg_kwargs)
    ref_kwargs.pop("leaky_alpha", None)
    fd = ref_kwargs.pop("feature_dimensionalities")
    fea = ref_kwargs.pop("feature_encoder_architecture")
    ina = ref_kwargs.pop("integration_network_architecture")
    od = ref_kwargs.pop("output_dimensionality")
    model = models.DistributedIBNet(fd, fea, ina, od, **ref_kwargs)        # models.py:56
    inject_weights(model, cfg, flat)
    model.beta.assign(beta)
    EPS.q = [eps[:, i, :].astype(DT) for i in range(cfg.number_features)]
    pred = model.call(x.astype(DT))                                         # models.py:96-123
    assert not EPS.q
    kls = np.array([model.metrics_log[f"KL{i}"] for i in range(cfg.number_features)])
    enc_out = [model.feature_encoders[i](_split(x.astype(DT), list(fd))[i]) for i in range(len(fd))]
    # the weights are regenerated from the seed when loaded (oracle.dib_oracle.load_forward_golden): only their digest is kept
    out = dict(seed=np.int64(seed), params_sha256=np.array(hashlib.sha256(flat.tobytes()).hexdigest()),
               x=x, eps=eps, beta=np.float32(beta), pred=np.asarray(pred),
               kl=kls, ib_loss=np.asarray(model.losses[0]), beta_metric=model.metrics_log["beta"],
               cfg=np.array(repr(cfg_kwargs)))
    for i, o in enumerate(enc_out):
        out[f"enc{i}"] = np.asarray(o)
    np.savez_compressed(os.path.join(HERE, f"ref_forward_{name}.npz"), **out)
    print(f"{name}: pred[0]={np.asarray(pred)[0]}, KL={kls[:3]}, ib_loss={model.losses[0]:.6g}")


def main():
    models, utils = load_reference()

    # --- forward goldens through the reference's DistributedIBNet.call ---
    run_case(models, "c0_small", dict(
        feature_dimensionalities=[1] * 16, feature_encoder_architecture=[128, 128],
        integration_network_architecture=[256, 256], output_dimensionality=1,
        use_positional_encoding=True, number_positional_encoding_frequencies=5,
        activation_fn="relu", feature_embedding_dimension=32, output_activation_fn=None),
        B=96, beta=0.03, seed=11)
    run_case(models, "pendulum_like", dict(
        feature_dimensionalities=[2, 1, 2, 1], feature_encoder_architecture=[128, 128],
        integration_network_architecture=[256, 256], output_dimensionality=6,
        use_positional_encoding=True, number_positional_encoding_frequencies=5,
        activation_fn="relu", feature_embedding_dimension=32, output_activation_fn=None),
        B=37, beta=1e-3, seed=12)
    run_case(models, "radial_like", dict(
        feature_dimensionalities=[1] * 10, feature_encoder_architecture=[128, 128],
        integration_network_architecture=[256, 256, 256], output_dimensionality=1,
        use_positional_encoding=False, activation_fn="tanh",
        feature_embedding_dimension=32, output_activation_fn=None),
        B=64, beta=0.5, seed=13)
    run_case(models, "odd_shapes", dict(
        feature_dimensionalities=[3, 1, 4], feature_encoder_architecture=[24, 40, 8],
        integration_network_architecture=[20], output_dimensionality=3,
        use_positional_encoding=True, number_positional_encoding_frequencies=3,
        activation_fn="leaky_relu", feature_embedding_dimension=6, output_activation_fn=None),
        B=19, beta=2.0, seed=14)

    # --- beta schedule through the reference's callback (models.py:125-149) ---
    class _M:
        pass
    sched = {}
    for tag, (b0, b1, npre, nann, epochs) in {
            "train_py_defaults": (1e-4, 3e0, 1000, 10000, [0, 1000, 1001, 6000, 10999]),
            "nb_radial": (1e-6, 1.0, 0, 250, [0, 125, 249]),
            "bench": (1e-4, 3.0, 2, 8, list(range(10)))}.items():
        cb = models.InfoBottleneckAnnealingCallback(b0, b1, npre, nann)
        cb.model = _M()
        cb.model.beta = _Variable(1.0, dtype=np.float32)
        vals = []
        for e in epochs:
            cb.on_epoch_begin(e)
            vals.append(np.float32(cb.model.beta.value()))
        sched[tag + "_args"] = np.array([b0, b1, npre, nann], dtype=np.float64)
        sched[tag + "_epochs"] = np.array(epochs)
        sched[tag + "_beta"] = np.array(vals, dtype=np.float32)
        print(tag, vals[:5])
    np.savez_compressed(os.path.join(HERE, "ref_beta_schedule.npz"), **sched)

    # --- Bhattacharyya through the reference's utils.bhattacharyya_dist_mat (utils.py:177-212) ---
    rng = np.random.default_rng(21)
    mu = rng.standard_normal((40, 32))
    lv = rng.standard_normal((40, 32)) * 0.7 - 0.5
    D = utils.bhattacharyya_dist_mat(mu, lv, mu, lv)
    mu2 = np.array([[1., -2.], [0., .5]])
    lv2 = np.array([[0., np.log(4.)], [-1., 1.]])
    D2 = utils.bhattacharyya_dist_mat(mu2, lv2, mu2, lv2)
    mu3, lv3 = rng.standard_normal((7, 5)), rng.standard_normal((7, 5))
    mu4, lv4 = rng.standard_normal((3, 5)), rng.standard_normal((3, 5))
    D34 = utils.bhattacharyya_dist_mat(mu3, lv3, mu4, lv4)
    np.savez_compressed(os.path.join(HERE, "ref_bhattacharyya.npz"), mu=mu, lv=lv, D=D, mu2=mu2, lv2=lv2,
                        D2=D2, mu3=mu3, lv3=lv3, mu4=mu4, lv4=lv4, D34=D34)
    print("bhattacharyya KAT off-diagonal:", D2[0, 1], np.exp(-D2[0, 1]))

    # --- KL matrix through the reference's utils.kl_divergence_mat (utils.py:213-247) ---
    rng = np.random.default_rng(22)
    kmu1, klv1 = rng.standard_normal((9, 6)), rng.standard_normal((9, 6)) * 0.6
    kmu2, klv2 = rng.standard_normal((4, 6)), rng.standard_normal((4, 6)) * 0.6 - 0.3
    KL12 = utils.kl_divergence_mat(kmu1, klv1, kmu2, klv2)
    KL11 = utils.kl_divergence_mat(kmu1, klv1, kmu1, klv1)
    np.savez_compressed(os.path.join(HERE, "ref_kl_divergence.npz"), mu1=kmu1, lv1=klv1, mu2=kmu2, lv2=klv2, KL12=KL12,
                        KL11=KL11)
    print("kl_divergence_mat[0,:3]:", KL12[0, :3])

    # --- similarity matrices through the reference's utils.get_scaled_similarity (utils.py:75-175) ---
    rng = np.random.default_rng(41)
    e1, e2 = rng.standard_normal((11, 6)), rng.standard_normal((7, 6))
    sims = {"e1": e1, "e2": e2, "temperature": np.float64(0.7)}
    for kind in ("l2sq", "l2", "l1", "linf", "cosine"):
        sims[kind] = utils.get_scaled_similarity(e1, e2, kind, 0.7)
    np.savez_compressed(os.path.join(HERE, "ref_scaled_similarity.npz"), **sims)
    print("similarity l2sq[0,:3]:", sims["l2sq"][0, :3], "cosine[0,:3]:", sims["cosine"][0, :3])

    # --- MI sandwich bounds through the reference's utils.estimate_mi_sandwich_bounds (utils.py:10-73) ---
    rng = np.random.default_rng(31)
    bs, E, nb = 64, 8, 3
    x_feat = rng.standard_normal((bs * nb, 1))
    Wenc = rng.standard_normal((1, 2 * E)) * 0.8
    benc = rng.standard_normal(2 * E) * 0.3
    encoder = lambda xb: np.concatenate([np.tanh(xb @ Wenc[:, :E] + benc[:E]) * 2.0, xb @ Wenc[:, E:] * 0.3 + benc[E:] - 1.0], -1)
    eps_mi = [rng.standard_normal((bs, E)) for _ in range(nb)]
    EPS.q = [e.copy() for e in eps_mi]
    bounds = utils.estimate_mi_sandwich_bounds(encoder, _Dataset(x_feat), evaluation_batch_size=bs, number_evaluation_batches=nb)
    assert not EPS.q
    enc_out = encoder(x_feat)
    np.savez_compressed(os.path.join(HERE, "ref_mi_sandwich.npz"), mu=enc_out[:, :E], lv=enc_out[:, E:], eps=np.stack(eps_mi),
                        bounds=np.asarray(bounds), bs=bs, nb=nb)
    print("MI sandwich (nats) lower/upper:", bounds)


if __name__ == "__main__":
    main()
