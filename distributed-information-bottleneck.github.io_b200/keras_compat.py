"""The slice of the tf.keras surface that the reference's training driver touches (train.py:128-172,
nb-radial cell 10): optimizer/loss objects handed to ``model.compile``, the ``Callback`` protocol and ``History``.
These are thin descriptions -- the arithmetic they name runs in the CUDA library."""
from __future__ import annotations


class Adam:
    """tf.keras.optimizers.Adam(learning_rate, beta_1, beta_2, epsilon) -- Keras defaults; epsilon is applied
    outside the bias correction (dib_adam_step)."""

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, name="adam"):
        self.learning_rate = learning_rate
        self.beta_1, self.beta_2, self.epsilon = beta_1, beta_2, epsilon
        self.name = name

    lr = property(lambda self: self.learning_rate, lambda self, v: setattr(self, "learning_rate", v))


class SGD:
    """tf.keras.optimizers.SGD(learning_rate=0.01, momentum=0.0, nesterov=False):
    v = momentum * v - lr * g;  w += momentum * v - lr * g if nesterov else v   (dib_optimizer_step kind 0)."""
    kind = 0

    def __init__(self, learning_rate=0.01, momentum=0.0, nesterov=False, name="SGD"):
        self.learning_rate, self.momentum, self.nesterov, self.name = learning_rate, float(momentum), bool(nesterov), name

    lr = property(lambda self: self.learning_rate, lambda self, v: setattr(self, "learning_rate", v))

    def hyper(self):
        return self.momentum, 1.0 if self.nesterov else 0.0, 0.0


class RMSprop:
    """tf.keras.optimizers.RMSprop(learning_rate=0.001, rho=0.9, momentum=0.0, epsilon=1e-7) (non-centered), TensorFlow's
    ApplyRMSProp: ms = rho ms + (1-rho) g^2;  mom = momentum mom + lr g / sqrt(ms + eps);  w -= mom  (kind 1)."""
    kind = 1

    def __init__(self, learning_rate=0.001, rho=0.9, momentum=0.0, epsilon=1e-7, centered=False, name="RMSprop"):
        if centered:
            raise NotImplementedError("RMSprop(centered=True) is not implemented")
        self.learning_rate, self.rho, self.momentum, self.epsilon, self.name = learning_rate, float(rho), float(momentum), float(epsilon), name

    lr = property(lambda self: self.learning_rate, lambda self, v: setattr(self, "learning_rate", v))

    def hyper(self):
        return self.rho, self.momentum, self.epsilon


class optimizers:
    Adam = Adam
    SGD = SGD
    RMSprop = RMSprop

    @staticmethod
    def get(identifier):
        """tf.keras.optimizers.get(name) as used at train.py:128 (the --optimizer flag, train.py:41)."""
        if isinstance(identifier, (Adam, SGD, RMSprop)):
            return identifier
        if isinstance(identifier, str):
            table = {"adam": Adam, "sgd": SGD, "rmsprop": RMSprop}
            if identifier.lower() in table:
                return table[identifier.lower()]()
        raise ValueError(f"optimizer {identifier!r} is not implemented by the B200 engine (adam, sgd, rmsprop are)")


class _Loss:
    kind = None

    def __init__(self, from_logits=False, name=None):
        self.from_logits = from_logits
        self.name = name


class BinaryCrossentropy(_Loss):
    """data.py:65 / nb-radial: BinaryCrossentropy(from_logits=True); from_logits=False (the Keras default) is the
    clipped-probability form for models with output_activation_fn='sigmoid'."""
    kind = "bce_logits"
    kind_probs = "bce_probs"


class SparseCategoricalCrossentropy(_Loss):
    """data.py:343: SparseCategoricalCrossentropy(from_logits=True)."""
    kind = "sparse_ce_logits"


class MeanSquaredError(_Loss):
    kind = "mse"

    def __init__(self, name=None):
        super().__init__(from_logits=True, name=name)


class InfoNCE(_Loss):
    """The InfoNCE training path of train.py:180-289 as a compiled loss: the model output e1 and a trainable output encoder's
    e2 = output_encoder(y) (train.py:186-193) are compared with utils.get_scaled_similarity, and both networks are trained on
    mean_i CE(i, S[i,:]) + mean_i CE(i, S^T[i,:]) + beta * sum_i KL_i (train.py:201-219).  Defaults are train.py:57-62's."""
    kind = "infonce"

    def __init__(self, similarity_type='l2', temperature=1.0, output_encoder_architecture=(128, 128), name=None):
        from . import _lib
        if similarity_type not in _lib.SIMILARITIES:
            raise ValueError('Similarity type not implemented: ', similarity_type)          # utils.py:172
        if not float(temperature) > 0.0:
            raise ValueError(f"InfoNCE temperature must be > 0, got {temperature!r}")
        arch = [int(w) for w in output_encoder_architecture]
        if any(w < 1 for w in arch):
            raise ValueError(f"output encoder widths must be >= 1, got {arch}")
        super().__init__(from_logits=True, name=name)
        self.similarity_type = similarity_type
        self.temperature = float(temperature)
        self.output_encoder_architecture = arch


class losses:
    BinaryCrossentropy = BinaryCrossentropy
    SparseCategoricalCrossentropy = SparseCategoricalCrossentropy
    MeanSquaredError = MeanSquaredError
    InfoNCE = InfoNCE


def resolve_loss(loss):
    if isinstance(loss, _Loss):
        if not loss.from_logits:
            if getattr(loss, "kind_probs", None):
                return loss.kind_probs
            raise NotImplementedError(
                f"{type(loss).__name__}(from_logits=False) is not implemented: the reference's call sites pass logits")
        return loss.kind
    if isinstance(loss, str):
        key = loss.lower()
        if key in ("mse", "mean_squared_error"):
            return "mse"
        if key in ("bce_logits", "sparse_ce_logits", "bce_probs"):
            return key
        if key == "binary_crossentropy":               # the Keras string means from_logits=False
            return "bce_probs"
        if key in ("external", "custom"):       # GradientTape-style loops: the caller owns the task loss
            return "external"
        if key == "infonce":                    # dataset_dict['loss'] of the pendulum dataset (data.py:131)
            return "infonce"
    raise ValueError(f"unsupported loss {loss!r}")


class Callback:
    """tf.keras.callbacks.Callback protocol (models.py:125,152,188): the trainer sets ``.model``."""
    model = None

    def set_model(self, model):
        self.model = model

    def on_train_begin(self, logs=None): pass
    def on_train_end(self, logs=None): pass
    def on_epoch_begin(self, epoch, logs=None): pass
    def on_epoch_end(self, epoch, logs=None): pass
    def on_train_batch_begin(self, batch, logs=None): pass
    def on_train_batch_end(self, batch, logs=None): pass


class callbacks:
    Callback = Callback


class History(Callback):
    """Return value of Model.fit: ``.history`` maps metric name -> list over epochs (train.py:169-172)."""

    def __init__(self):
        self.history = {}
        self.epoch = []

    def on_epoch_end(self, epoch, logs=None):
        self.epoch.append(epoch)
        for k, v in (logs or {}).items():
            self.history.setdefault(k, []).append(v)
