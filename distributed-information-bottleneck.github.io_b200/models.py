"""Host-side mirror of the reference's ``models.py`` (PositionalEncoding, DistributedIBNet, the annealing /
compression-matrix / embedding-stash callbacks) on top of the C ABI in include/dib_b200.h.

Same names, constructor arguments and call protocol as /root/reference/models.py:12-223 and the corrected copy
in nb-radial cell 5, so ``train.py``-style drivers and the notebooks' ``model.compile / model.fit`` code run
unchanged with ``import dib_b200.models as models``.  PyTorch is used for device memory, streams and
``torch.distributed`` only; every FLOP of the hot path runs in libdib_b200.so.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import parallel
from .keras_compat import Adam, InfoNCE, RMSprop, SGD, Callback, History, optimizers, resolve_loss


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.DibError("dib_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _as_numpy_like(ref, t):
    """Return ``t`` in the kind of container ``ref`` was (numpy in -> numpy out, tensor in -> tensor out)."""
    if isinstance(ref, torch.Tensor):
        return t
    return t.detach().cpu().numpy()


class PositionalEncoding:
    """models.py:12-23.  Kept for API parity; inside DistributedIBNet the encoding is fused into the first-layer
    operand by the library.  Calling it directly is a convenience (plain torch ops, not the hot path)."""

    def __init__(self, frequencies):
        self.frequencies = list(frequencies)

    def __call__(self, inputs):
        freqs = [int(f) for f in self.frequencies]
        if freqs != [2 ** k for k in range(1, len(freqs) + 1)]:
            raise NotImplementedError("the library's positional encoding uses the reference's frequencies 2**arange(1, n)")
        _require_cuda()
        t = torch.as_tensor(inputs, dtype=torch.float32)
        dev = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device())
        x = t.to(dev).reshape(-1, t.shape[-1]).contiguous()
        out = torch.empty(x.shape[0], x.shape[1] * (len(freqs) + 1), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().dib_positional_encoding(_lib.ptr(x), x.shape[0], x.shape[1], len(freqs) + 1, _lib.ptr(out),
                                                           _stream()))
        return _as_numpy_like(inputs, out.reshape(*t.shape[:-1], out.shape[-1]))

    call = __call__


class _Beta:
    """``tf.Variable(1., dtype=tf.float32, trainable=False)`` surface used by the callbacks (models.py:86,148,177)."""

    def __init__(self, device):
        self._host = np.float32(1.0)
        self._dev = torch.ones(1, dtype=torch.float32, device=device)

    def assign(self, value):
        self._host = np.float32(value)
        self._dev.fill_(float(self._host))
        return self

    def value(self):
        return self._host

    numpy = value

    def __float__(self):
        return float(self._host)

    def __array__(self, dtype=None, copy=None):
        return np.asarray(self._host, dtype=dtype)

    # arithmetic the reference's drivers do with the variable: ``kl_loss / model.beta`` (train.py:214),
    # ``self.beta * tensor`` (models.py:118), ``beta * 2.0`` -- delegate to the float32 host value
    def _other(self, o):
        return o.to(torch.float32) if isinstance(o, torch.Tensor) else o

    def __mul__(self, o): return float(self._host) * self._other(o)
    __rmul__ = __mul__
    def __truediv__(self, o): return float(self._host) / self._other(o)
    def __rtruediv__(self, o): return self._other(o) / float(self._host)
    def __add__(self, o): return float(self._host) + self._other(o)
    __radd__ = __add__
    def __sub__(self, o): return float(self._host) - self._other(o)
    def __rsub__(self, o): return self._other(o) - float(self._host)
    def __neg__(self): return -float(self._host)
    def __repr__(self): return f"<beta {float(self._host)!r}>"


class _Network:
    """A view of one Dense stack inside the flat parameter buffer (model.feature_encoders[i] /
    model.integration_network): ``.weights`` are torch views [W, b, W, b, ...] in Keras order."""

    def __init__(self, model, var_slice):
        self._model = model
        self._vars = var_slice

    @property
    def weights(self):
        return [self._model._var_view(i) for i in self._vars]

    trainable_variables = weights

    def get_weights(self):
        return [w.detach().cpu().numpy() for w in self.weights]


class _FeatureEncoder(_Network):
    """model.feature_encoders[i]: deterministic [n, d_i] -> [n, 2E] (mu || logvar), the contract used by
    visualization.py:31, utils.py:38 and StashEmbeddingsCallback.  Runs dib_encode_feature."""

    def __init__(self, model, index, var_slice):
        super().__init__(model, var_slice)
        self.index = index

    def __call__(self, x_i, training=None):
        return _as_numpy_like(x_i, self._model._encode_feature(self.index, x_i))


class _IntegrationNetwork(_Network):
    """model.integration_network (models.py:84).  Direct calls are rare (the fused step never materialises this
    boundary); they run dib_integration_forward on the model's precision path."""

    def __call__(self, emb, training=None):
        m = self._model
        with torch.cuda.device(m.device):
            e = m._to_device(emb, m.number_features * m.feature_embedding_dimension)
            n = e.shape[0]
            m._ensure_handle(n)
            out = torch.empty(n, m.output_dimensionality, dtype=torch.float32, device=m.device)
            _lib.check(m._lib.dib_integration_forward(m._handle, _lib.ptr(m._params), _lib.ptr(e), n, _lib.ptr(out),
                                                      _lib.ptr(m._workspace), _stream()))
        return _as_numpy_like(emb, out)


class DistributedIBNet:
    """Distributed IB model where each feature is passed through its own probabilistic encoder MLP
    (models.py:26-123; ``dropout_rate``/``training`` from nb-radial cell 5).

    Custom-step variants of the same front end (keyword-only; SURVEY 8f3):
      ``feature_encoder_architecture='simple'`` -- nb-bool cell 4's SimpleEncoder for every feature (two trainable (1,1)
        constants mu_scaling = 1, logvar = -3; needs d_i == feature_embedding_dimension, no positional encoding);
      ``logvar_offset`` -- constant added to every encoder's log-variance (nb-particle cell 8, -3 there);
      ``kl_loss_exponent`` / ``kl_loss_scale`` -- nonlinear IB ``beta * scale * (sum_i KL_i) ** exponent`` (nb-chaos cell 10);
      ``model.encode`` / ``model.encoder_gradients`` -- encoder-only steps for a caller-owned downstream network
        (nb-particle's shared particle encoder + set transformer: see :class:`SharedParticleEncoder`).

    Extra keyword-only arguments (not in the reference): ``device``, ``seed`` (weight init + noise stream),
    ``precision`` ('fp32' exact-FMA parity path | 'tf32' kind::tf32 GEMMs | 'fp16' / 'bf16' fused 16-bit-operand
    tcgen05 kernels with fp32 accumulation; ``model.kernel_info()`` says what a handle actually runs), ``process_group``
    (data-parallel group; defaults to the WORLD group when torch.distributed is initialised), ``leaky_alpha``.
    """

    def __init__(self,
                 feature_dimensionalities: Sequence[int],
                 feature_encoder_architecture: Sequence[int],
                 integration_network_architecture: Sequence[int],
                 output_dimensionality: int,
                 use_positional_encoding: bool = True,
                 number_positional_encoding_frequencies: int = 5,
                 activation_fn: Optional[str] = 'relu',
                 feature_embedding_dimension: int = 32,
                 output_activation_fn: Optional[str] = None,
                 dropout_rate: float = 0.,
                 *, device=None, seed: int = 0, precision: str = 'fp32', process_group=None,
                 leaky_alpha: float = 0.2, logvar_offset: float = 0., kl_loss_exponent: float = 1.,
                 kl_loss_scale: float = 1.):
        _require_cuda()
        if not (0.0 <= float(dropout_rate) < 1.0):
            raise ValueError("dropout_rate must be in [0, 1)")
        self.dropout_rate = float(dropout_rate)       # nb-radial cell 5: Dropout after every hidden encoder Dense (train steps only)
        if activation_fn not in _lib.ACTIVATIONS or output_activation_fn not in _lib.ACTIVATIONS:
            raise ValueError(f"unsupported activation {activation_fn!r}/{output_activation_fn!r}")
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}, got {precision!r}")
        self.feature_dimensionalities = [int(d) for d in feature_dimensionalities]
        self.number_features = len(self.feature_dimensionalities)
        self.encoder_kind = "simple" if isinstance(feature_encoder_architecture, str) else "mlp"
        if self.encoder_kind == "simple":
            if feature_encoder_architecture != "simple":
                raise ValueError("feature_encoder_architecture must be a list of widths or 'simple'")
            feature_encoder_architecture, use_positional_encoding = [], False
        self.logvar_offset = float(logvar_offset)
        self.kl_loss_exponent = float(kl_loss_exponent)
        self.kl_loss_scale = float(kl_loss_scale)
        self.feature_encoder_architecture = [int(h) for h in feature_encoder_architecture]
        self.integration_network_architecture = [int(h) for h in integration_network_architecture]
        self.output_dimensionality = int(output_dimensionality)
        self.use_positional_encoding = bool(use_positional_encoding)
        self.number_positional_encoding_frequencies = int(number_positional_encoding_frequencies)
        self.activation_fn = activation_fn
        self.output_activation_fn = output_activation_fn
        self.feature_embedding_dimension = int(feature_embedding_dimension)
        self.leaky_alpha = float(leaky_alpha)
        self.precision = precision
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.seed = int(seed)
        self.noise_seed = int(seed)
        self.process_group = process_group
        self.stop_training = False

        self._lib = _lib.load()
        self._loss_kind = "bce_logits"
        self._handle = None
        self._handle_key = None
        self._workspace = None
        self._query_layout()

        with torch.cuda.device(self.device):
            self.beta = _Beta(self.device)                                   # models.py:86
            self._params = torch.zeros(self._P, dtype=torch.float32, device=self.device)
            self._init_glorot_uniform()
            self._gradstats = torch.zeros(self._P + self.number_features + 3, dtype=torch.float32, device=self.device)
            self._m = torch.zeros_like(self._params)
            self._v = torch.zeros_like(self._params)
            self._lr_dev = torch.full((1,), 1e-3, dtype=torch.float32, device=self.device)
            self._step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._epoch_acc = torch.zeros(self.number_features + 4, dtype=torch.float32, device=self.device)
        # the optimizer updates [model P | output encoder Q] as ONE flat buffer (one Adam iteration count per step, train.py:219);
        # without an output encoder these are the model's own buffers
        self._params_all, self._m_all, self._v_all = self._params, self._m, self._v
        self._Q = 0
        self.output_encoder = None         # InfoNCE: built from the first y batch's width (build_output_encoder)
        self._infonce = None               # the compiled keras_compat.InfoNCE
        self._nce_scratch = {}             # (n, kind) -> head scratch of the InfoNCE step
        self._train_step_count = 0
        # ---- CUDA-graph replay of the train step (launch-bound small batches; fewer host calls per step at any size)
        env = os.environ.get("DIB_CUDA_GRAPH", "auto").lower()
        self.use_cuda_graph = env not in ("0", "off", "false", "no")
        self._graphs = {}                  # (n, global_batch, sample_offset, world) -> captured step
        self._graph_seen = {}              # eager executions per key before capture (lazy one-time setup must be done)
        self._graph_failed = False
        self._noise_step_dev = None        # int32 device mirror of _train_step_count (Philox step word inside graphs)
        self._step_dev_active = False
        self._step_dev_dirty = False       # _train_step_count moved outside a graph replay: refill the device mirror
        self._replayed_launches = 0        # kernels launched by graph replays (dib_launch_count only sees eager launches)
        self._side_stream = None
        # two-bucket all-reduce overlapped with the encoder backward: measured SLOWER than one flat all-reduce on 2 B200s
        # (0.475 vs 0.444 ms/step strong, 0.758 vs 0.744 weak -- the second NCCL launch and the stream hand-offs cost more than
        # the 0.8 MB bucket hides), so it is opt-in (DIB_OVERLAP_ALLREDUCE=1)
        self.overlap_allreduce = os.environ.get("DIB_OVERLAP_ALLREDUCE", "0") in ("1", "on", "true", "yes")
        # (capturing the NCCL all-reduce inside the step's graph was tried on 2 B200s: no gain -- 0.611 vs 0.605 ms/step weak -- and
        #  the processes hung at teardown; the all-reduce stays an eager call between the backward graph and the optimizer graph)
        self._inference_calls = 0          # fresh noise per un-seeded inference call (tf.random.normal, models.py:108)
        self.optimizer = None
        self.compiled_metrics_names = []
        self.losses = []
        self.metrics_values = {}
        n_enc_vars = 2 if self.encoder_kind == "simple" else 2 * (len(self.feature_encoder_architecture) + 1)
        self.feature_encoders = [                                            # models.py:79
            _FeatureEncoder(self, i, range(i * n_enc_vars, (i + 1) * n_enc_vars)) for i in range(self.number_features)]
        self.integration_network = _IntegrationNetwork(                      # models.py:84
            self, range(self.number_features * n_enc_vars, len(self._var_off)))
        self._p_enc = int(self._var_off[self.number_features * n_enc_vars])  # first integration-network parameter

    # ------------------------------------------------------------------ library handle / buffers
    def _config(self, max_batch):
        F = self.number_features
        self._c_fd = (ctypes.c_int32 * F)(*self.feature_dimensionalities)
        L, Li = len(self.feature_encoder_architecture), len(self.integration_network_architecture)
        self._c_ea = (ctypes.c_int32 * max(L, 1))(*self.feature_encoder_architecture)
        self._c_ia = (ctypes.c_int32 * max(Li, 1))(*self.integration_network_architecture)
        return _lib.DibConfig(
            abi_version=_lib.ABI_VERSION, number_features=F, feature_dimensionalities=self._c_fd,
            number_encoder_layers=L, feature_encoder_architecture=self._c_ea,
            number_integration_layers=Li, integration_network_architecture=self._c_ia,
            output_dimensionality=self.output_dimensionality,
            use_positional_encoding=int(self.use_positional_encoding),
            number_positional_encoding_frequencies=self.number_positional_encoding_frequencies,
            activation_fn=_lib.ACTIVATIONS[self.activation_fn], leaky_relu_alpha=self.leaky_alpha,
            feature_embedding_dimension=self.feature_embedding_dimension,
            output_activation_fn=_lib.ACTIVATIONS[self.output_activation_fn],
            loss=_lib.LOSSES[self._loss_kind], precision=_lib.PRECISIONS[self.precision], max_batch=int(max_batch),
            logvar_offset=self.logvar_offset, kl_loss_exponent=self.kl_loss_exponent, kl_loss_scale=self.kl_loss_scale,
            encoder_kind=_lib.ENCODER_KINDS[self.encoder_kind], dropout_rate=self.dropout_rate)

    def _query_layout(self):
        with torch.cuda.device(self.device):
            h = ctypes.c_void_p()
            cfg = self._config(1)
            _lib.check(self._lib.dib_create(ctypes.byref(cfg), ctypes.byref(h)))
            try:
                self._P = int(self._lib.dib_param_count(h))
                nv = self._lib.dib_param_layout(h, None, None, None, 0)
                offs, rows, cols = (ctypes.c_int64 * nv)(), (ctypes.c_int32 * nv)(), (ctypes.c_int32 * nv)()
                assert self._lib.dib_param_layout(h, offs, rows, cols, nv) == nv
                self._var_off, self._var_rows, self._var_cols = list(offs), list(rows), list(cols)
            finally:
                self._lib.dib_destroy(h)

    @property
    def _PQ(self):
        return self._P + self._Q

    def _ensure_handle(self, n):
        oe = self.output_encoder
        key = (self._loss_kind, self.precision, None if oe is None else (oe.input_dimensionality, tuple(oe.architecture)))
        if self._handle is not None and self._handle_key == key and n <= self._max_batch:
            return
        self._release_handle()
        max_batch = max(int(n), 1)
        with torch.cuda.device(self.device):
            h = ctypes.c_void_p()
            cfg = self._config(max_batch)
            _lib.check(self._lib.dib_create(ctypes.byref(cfg), ctypes.byref(h)))
            self._handle, self._handle_key, self._max_batch = h, key, max_batch
            if oe is not None and self._loss_kind == "infonce":
                _lib.check(self._lib.dib_attach_output_encoder(h, ctypes.byref(oe._config())))
            self._graphs.clear(); self._graph_seen.clear()       # captured launches point into the old workspace
            self._step_dev_active = False
            if getattr(self, "_force_unfused", 0):
                _lib.check(self._lib.dib_debug_force_unfused(h, int(self._force_unfused)))
            nbytes = int(self._lib.dib_workspace_bytes(h))
            self._workspace = None
            self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            assert self._workspace.data_ptr() % 256 == 0

    def kernel_info(self, batch_hint=1):
        """What the library runs for this model: precision, kernel families, operand / accumulator types."""
        with torch.cuda.device(self.device):
            self._ensure_handle(max(int(batch_hint), 1))
            buf = ctypes.create_string_buffer(512)
            if self._lib.dib_model_info(self._handle, buf, len(buf)) < 0:
                raise _lib.DibError(self._lib.dib_last_error().decode())
        return buf.value.decode()

    def _release_handle(self):
        if getattr(self, "_handle", None) is not None:
            torch.cuda.synchronize(self.device)
            self._lib.dib_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release_handle()
        except Exception:
            pass

    def _var_view(self, i):
        off, r, c = self._var_off[i], self._var_rows[i], self._var_cols[i]
        v = self._params[off:off + max(r, 1) * c]
        return v.view(r, c) if r > 0 else v

    def _init_glorot_uniform(self):
        """Keras Dense defaults: kernel glorot_uniform, bias zeros (third-party behaviour; RNG stream is ours)."""
        g = torch.Generator(device="cpu")
        g.manual_seed(self.seed)
        flat = torch.zeros(self._P, dtype=torch.float32)
        n_simple = 2 * self.number_features if self.encoder_kind == "simple" else 0
        for k, (off, r, c) in enumerate(zip(self._var_off, self._var_rows, self._var_cols)):
            if k < n_simple:                 # nb-bool cell 4: mu_scaling = ones, logvar = -3 * ones
                flat[off] = 1.0 if k % 2 == 0 else -3.0
            elif r > 0:
                lim = math.sqrt(6.0 / (r + c))
                flat[off:off + r * c] = (torch.rand(r * c, generator=g) * 2 - 1) * lim
        self._params.copy_(flat)

    # ------------------------------------------------------------------ Keras-like variable access
    @property
    def trainable_variables(self):
        return [self._var_view(i) for i in range(len(self._var_off))]

    trainable_weights = trainable_variables
    weights = trainable_variables

    def get_weights(self):
        return [v.detach().cpu().numpy() for v in self.trainable_variables]

    def set_weights(self, weights):
        vs = self.trainable_variables
        if len(weights) != len(vs):
            raise ValueError(f"expected {len(vs)} arrays, got {len(weights)}")
        for v, w in zip(vs, weights):
            v.copy_(torch.as_tensor(np.asarray(w), dtype=torch.float32).view(v.shape))

    def get_flat_weights(self):
        return self._params.detach().cpu().numpy()

    def set_flat_weights(self, flat):
        self._params.copy_(torch.as_tensor(np.asarray(flat), dtype=torch.float32))

    def count_params(self):
        return self._P

    def build(self, input_shape):
        assert input_shape[-1] == sum(self.feature_dimensionalities)       # models.py:89

    # ------------------------------------------------------------------ data helpers
    def _to_device(self, a, cols=None):
        if a is None:
            return None
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        t = t.to(device=self.device, dtype=torch.float32, non_blocking=True)
        if cols is not None:
            t = t.reshape(t.shape[0], cols) if cols > 0 else t.reshape(t.shape[0])
        return t.contiguous()

    def _y_cols(self):
        if self._loss_kind == "infonce":
            if self.output_encoder is None:
                raise RuntimeError("the InfoNCE output encoder is not built: pass a batch or call build_output_encoder(dy)")
            return self.output_encoder.input_dimensionality
        return 0 if self._loss_kind == "sparse_ce_logits" else self.output_dimensionality

    # ------------------------------------------------------------------ InfoNCE output encoder (train.py:186-193)
    def build_output_encoder(self, input_dimensionality, architecture=None):
        """Build the trainable output encoder y [n, input_dimensionality] -> e2 [n, output_dimensionality] of the InfoNCE
        path (Keras builds it on its first call; fit / train_on_batch do this from the first y batch).  ``architecture``
        defaults to the compiled InfoNCE loss's ``output_encoder_architecture``.  Weights: glorot-uniform kernels and zero
        biases, drawn from a torch CPU generator seeded with ``seed + 0x5EED0E`` in flat order (a stream of its own, so the
        model's initial weights do not depend on whether an output encoder exists)."""
        if architecture is None:
            architecture = self._infonce.output_encoder_architecture if self._infonce is not None else (128, 128)
        dy, arch = int(input_dimensionality), [int(w) for w in architecture]
        if self.output_encoder is not None:
            if (self.output_encoder.input_dimensionality, self.output_encoder.architecture) == (dy, arch):
                return self.output_encoder
            raise ValueError("the output encoder is already built with a different shape")
        oe = OutputEncoder(self, dy, arch)
        with torch.cuda.device(self.device):
            h = ctypes.c_void_p()
            cfg = self._config(1)
            cfg.loss, cfg.output_activation_fn = _lib.LOSSES["infonce"], 0
            _lib.check(self._lib.dib_create(ctypes.byref(cfg), ctypes.byref(h)))
            try:
                _lib.check(self._lib.dib_attach_output_encoder(h, ctypes.byref(oe._config())))
                Q = int(self._lib.dib_output_encoder_param_count(h))
                nv = self._lib.dib_output_encoder_param_layout(h, None, None, None, 0)
                offs, rows, cols = (ctypes.c_int64 * nv)(), (ctypes.c_int32 * nv)(), (ctypes.c_int32 * nv)()
                assert self._lib.dib_output_encoder_param_layout(h, offs, rows, cols, nv) == nv
            finally:
                self._lib.dib_destroy(h)
            oe._layout = (list(offs), list(rows), list(cols))
            P = self._P
            g = torch.Generator(device="cpu")
            g.manual_seed(self.seed + 0x5EED0E)
            q = torch.zeros(Q, dtype=torch.float32)
            for off, r, c in zip(*oe._layout):
                if r > 0:
                    lim = math.sqrt(6.0 / (r + c))
                    q[off - P:off - P + r * c] = (torch.rand(r * c, generator=g) * 2 - 1) * lim
            self._release_handle()
            self._graphs.clear(); self._graph_seen.clear()
            new = []
            for old, tail in ((self._params_all, q.to(self.device)), (self._m_all, None), (self._v_all, None)):
                t = torch.zeros(P + Q, dtype=torch.float32, device=self.device)
                t[:P].copy_(old[:P])
                if tail is not None:
                    t[P:].copy_(tail)
                new.append(t)
            self._params_all, self._m_all, self._v_all = new
            self._params, self._m, self._v = (t[:P] for t in new)
            self._Q = Q
            self._gradstats = torch.zeros(P + Q + self.number_features + 3, dtype=torch.float32, device=self.device)
        self.output_encoder = oe
        return oe

    def _head_scratch(self, n):
        kind = _lib.SIMILARITIES[self._infonce.similarity_type]
        t = self._nce_scratch.get((n, kind))
        if t is None:
            nbytes = int(self._lib.dib_infonce_scratch_bytes(kind, n, self.output_dimensionality))
            # out of range (l1 / linf above 32768 rows): the step itself refuses with the reason
            t = torch.empty(max(nbytes, 128), dtype=torch.uint8, device=self.device)
            self._nce_scratch[(n, kind)] = t
        return kind, t

    def _infonce_call(self, x, y, step, sample_offset=0, eps=None, train=True, device_step=False, stats_out=None):
        """dib_infonce_train_step (gradients into self._gradstats = [grads (P+Q) || stats]) or dib_infonce_forward."""
        n = x.shape[0]
        self._ensure_handle(n)
        kind, scratch = self._head_scratch(n)
        PQ = self._PQ
        if train:
            self._set_device_step(device_step)
            _lib.check(self._lib.dib_infonce_train_step(
                self._handle, _lib.ptr(self._params_all), _lib.ptr(x), _lib.ptr(y), n, _lib.ptr(self.beta._dev), kind,
                self._infonce.temperature, _lib.ptr(eps), self.noise_seed, int(step) & 0xFFFFFFFF, int(sample_offset),
                _lib.ptr(scratch), _lib.ptr(self._gradstats), _lib.ptr(self._gradstats[PQ:]), _lib.ptr(self._workspace),
                _stream()))
            return self._gradstats[PQ:]
        stats = stats_out if stats_out is not None else torch.empty(self.number_features + 3, dtype=torch.float32,
                                                                    device=self.device)
        _lib.check(self._lib.dib_infonce_forward(
            self._handle, _lib.ptr(self._params_all), _lib.ptr(x), _lib.ptr(y), n, _lib.ptr(self.beta._dev), kind,
            self._infonce.temperature, _lib.ptr(eps), self.noise_seed, int(step) & 0xFFFFFFFF, int(sample_offset),
            _lib.ptr(scratch), _lib.ptr(stats), _lib.ptr(self._workspace), _stream()))
        return stats

    # ------------------------------------------------------------------ compute entry points
    def _forward(self, x, y, eps, step, sample_offset, want_pred=True, want_emb=False, stats_out=None):
        n = x.shape[0]
        self._ensure_handle(n)
        pred = torch.empty(n, self.output_dimensionality, dtype=torch.float32, device=self.device) if want_pred else None
        emb = torch.empty(n, self.number_features * self.feature_embedding_dimension, dtype=torch.float32,
                          device=self.device) if want_emb else None
        stats = stats_out if stats_out is not None else torch.empty(self.number_features + 3, dtype=torch.float32,
                                                                    device=self.device)
        _lib.check(self._lib.dib_forward(
            self._handle, _lib.ptr(self._params), _lib.ptr(x), _lib.ptr(y), n, _lib.ptr(self.beta._dev), _lib.ptr(eps),
            self.noise_seed, int(step) & 0xFFFFFFFF, int(sample_offset), _lib.ptr(pred), _lib.ptr(emb), _lib.ptr(stats),
            _lib.ptr(self._workspace), _stream()))
        return pred, emb, stats

    def _encode_feature(self, i, x_i):
        t = self._to_device(x_i, self.feature_dimensionalities[i])
        n = t.shape[0]
        self._ensure_handle(n)
        out = torch.empty(n, 2 * self.feature_embedding_dimension, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.dib_encode_feature(self._handle, _lib.ptr(self._params), i, _lib.ptr(t), n,
                                                    _lib.ptr(out), _lib.ptr(self._workspace), _stream()))
        return out

    def compression_matrices(self, x, row_index=None, want=("mu_logvar", "dist", "comp")):
        """All features at once (dib_compression_matrices; visualization.py:14-35 loops over features in Python):
        rows ``row_index[i]`` of ``x`` -> encoder i -> Bhattacharyya -> exp(-D).  ``row_index``: [F, n] integer array or
        None (= all rows of x for every feature).  Returns a dict of device tensors for the names in ``want``:
        mu_logvar [F, n, 2E], dist [F, n, n], comp [F, n, n]."""
        t = self._to_device(x, sum(self.feature_dimensionalities))
        F, E = self.number_features, self.feature_embedding_dimension
        if row_index is None:
            n, idx = t.shape[0], None
        else:
            idx = row_index if isinstance(row_index, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(row_index))
            idx = idx.to(device=self.device, dtype=torch.int32).contiguous()
            if idx.dim() != 2 or idx.shape[0] != F:
                raise ValueError("row_index must have shape [number_features, n]")
            n = idx.shape[1]
        self._ensure_handle(max(n, 1))
        out = {}
        if "mu_logvar" in want:
            out["mu_logvar"] = torch.empty(F, n, 2 * E, dtype=torch.float32, device=self.device)
        if "dist" in want:
            out["dist"] = torch.empty(F, n, n, dtype=torch.float32, device=self.device)
        if "comp" in want:
            out["comp"] = torch.empty(F, n, n, dtype=torch.float32, device=self.device)
        opt = lambda k: _lib.ptr(out[k]) if k in out else None
        with torch.cuda.device(self.device):
            _lib.check(self._lib.dib_compression_matrices(self._handle, _lib.ptr(self._params), _lib.ptr(t), t.shape[0],
                                                          _lib.ptr(idx) if idx is not None else None, n, opt("mu_logvar"),
                                                          opt("dist"), opt("comp"), _lib.ptr(self._workspace), _stream()))
        return out

    def _set_device_step(self, on):
        """Philox step word from the device mirror of _train_step_count (graph replay) or by value (everything else)."""
        if on == self._step_dev_active and self._handle is not None and not (on and self._step_dev_dirty):
            return
        if on:
            self._step_dev_dirty = False
            if self._noise_step_dev is None:
                self._noise_step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._noise_step_dev.fill_(int(self._train_step_count) & 0x7FFFFFFF)
        _lib.check(self._lib.dib_set_noise_step_device(self._handle, _lib.ptr(self._noise_step_dev) if on else None))
        self._step_dev_active = on

    def _backward(self, x, y, global_batch, eps=None, sample_offset=0, step=None, phases=3, device_step=False):
        """dib_train_step[_phased]: forward + reverse mode into self._gradstats = [grads (P) || stats (F+3)]."""
        if self._loss_kind == "infonce":
            st = 0 if device_step else (self._train_step_count if step is None else step)
            self._infonce_call(x, y, st, sample_offset, eps, device_step=device_step)
            return
        n = x.shape[0]
        self._ensure_handle(n)
        P = self._P
        self._set_device_step(device_step)
        st = 0 if device_step else (self._train_step_count if step is None else step)
        _lib.check(self._lib.dib_train_step_phased(
            self._handle, _lib.ptr(self._params), _lib.ptr(x), _lib.ptr(y), n, _lib.ptr(self.beta._dev),
            1.0 / float(global_batch), _lib.ptr(eps), self.noise_seed, int(st) & 0xFFFFFFFF,
            int(sample_offset), _lib.ptr(self._gradstats), _lib.ptr(self._gradstats[P:]), _lib.ptr(self._workspace),
            int(phases), _stream()))

    def apply_gradients(self, flat_grads):
        """optimizer.apply_gradients(zip(grads, model.trainable_variables)) of the custom loops (train.py:217-219,
        nb-bool cell 6): one Keras-Adam update of the flat parameter buffer with caller-supplied gradients."""
        g = torch.as_tensor(flat_grads, dtype=torch.float32).to(self.device).contiguous()
        if g.numel() != self._PQ:
            raise ValueError(f"expected {self._PQ} gradient values, got {g.numel()}")
        self._sync_lr()
        with torch.cuda.device(self.device):
            self._optimizer_update(g)
        self._train_step_count += 1
        self._step_dev_dirty = True

    def _optimizer_update(self, grads):
        """One dense update of the flat parameter buffer by the compiled optimizer (Adam: dib_adam_step; SGD / RMSprop:
        dib_optimizer_step); the two slot buffers are Adam's m / v, SGD's velocity, RMSprop's mean square / momentum."""
        opt = self.optimizer
        if isinstance(opt, Adam):
            _lib.check(self._lib.dib_adam_step(
                _lib.ptr(self._params_all), _lib.ptr(grads), _lib.ptr(self._m_all), _lib.ptr(self._v_all), self._PQ,
                _lib.ptr(self._lr_dev), _lib.ptr(self._step_dev), opt.beta_1, opt.beta_2, opt.epsilon, _stream()))
        else:
            h0, h1, h2 = opt.hyper()
            _lib.check(self._lib.dib_optimizer_step(
                opt.kind, _lib.ptr(self._params_all), _lib.ptr(grads), _lib.ptr(self._m_all), _lib.ptr(self._v_all), self._PQ,
                _lib.ptr(self._lr_dev), _lib.ptr(self._step_dev), h0, h1, h2, _stream()))

    def _adam(self):
        self._optimizer_update(self._gradstats)

    def _reduce_overlapped(self, world, run_phase1, run_phase2):
        """The data-parallel exchange in two buckets: [integration grads || stats] is all-reduced on a side stream while
        the encoder backward (phase 2) runs; [encoder grads] follows on the compute stream.  One process per GPU, NCCL."""
        pe = self._p_enc
        run_phase1()
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self.device)
        side, main = self._side_stream, torch.cuda.current_stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            work = parallel.allreduce_sum_async(self._gradstats[pe:], self.process_group)
        run_phase2()
        parallel.allreduce_sum_(self._gradstats[:pe], self.process_group)
        if work is not None:
            work.wait()                      # the compute stream waits for bucket 1 (no host sync)
        main.wait_stream(side)

    def _train_step(self, x, y, global_batch, eps=None, sample_offset=0):
        """backward, all-reduce over the data-parallel group, Keras-Adam.  Replayed from CUDA graphs once a
        (batch size, offset) combination has run eagerly twice; the all-reduce is split into two buckets so that the
        first overlaps the encoder backward."""
        P = self._PQ
        world, _ = parallel.world_and_rank(self.process_group)
        key = (int(x.shape[0]), int(global_batch), int(sample_offset), world)
        if self.use_cuda_graph and not self._graph_failed and eps is None and x.shape[0] > 0:
            g = self._graphs.get(key)
            if g is None and self._graph_seen.get(key, 0) >= 2:
                g = self._capture_step(key)
            if g is not None:
                return self._replay_step(g, x, y, world)
            self._graph_seen[key] = self._graph_seen.get(key, 0) + 1
        if world > 1 and self.overlap_allreduce:
            self._reduce_overlapped(world, lambda: self._backward(x, y, global_batch, eps, sample_offset, phases=1),
                                    lambda: self._backward(x, y, global_batch, eps, sample_offset, phases=2))
        else:
            self._backward(x, y, global_batch, eps, sample_offset)
            parallel.allreduce_sum_(self._gradstats, self.process_group)
        self._adam()
        self._train_step_count += 1
        self._step_dev_dirty = True
        return self._gradstats[P:]

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def _capture_step(self, key):
        """Capture the step for one (n, global_batch, sample_offset, world) into CUDA graphs.  Single GPU: ONE graph
        (forward + backward + Adam + noise-step increment).  Data parallel: two graphs (backward | Adam) with the NCCL all-reduce
        issued eagerly between them (three -- phase 1 | phase 2 | Adam -- for the opt-in two-bucket overlap).  Inputs are copied into static buffers before each replay; beta,
        learning rate, the Adam step and the Philox step are device scalars, so nothing by-value changes between replays."""
        n, global_batch, sample_offset, world = key
        D = sum(self.feature_dimensionalities)
        yc = self._y_cols()
        try:
            with torch.cuda.device(self.device):
                gx = torch.zeros(n, D, dtype=torch.float32, device=self.device)
                gy = torch.zeros((n, yc) if yc > 0 else (n,), dtype=torch.float32, device=self.device)
                self._ensure_handle(n)
                self._set_device_step(True)
                torch.cuda.synchronize(self.device)
                keep = [t.clone() for t in (self._params_all, self._m_all, self._v_all, self._step_dev, self._noise_step_dev)]
                graphs = []
                launches0 = int(self._lib.dib_launch_count())

                def cap(fn):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        fn()
                    graphs.append(g)

                def tail():
                    self._adam()
                    self._noise_step_dev.add_(1)

                if world == 1:
                    cap(lambda: (self._backward(gx, gy, global_batch, None, sample_offset, device_step=True), tail()))
                elif self.overlap_allreduce:
                    cap(lambda: self._backward(gx, gy, global_batch, None, sample_offset, phases=1, device_step=True))
                    cap(lambda: self._backward(gx, gy, global_batch, None, sample_offset, phases=2, device_step=True))
                    cap(tail)
                else:        # one all-reduce between backward and optimizer: two graphs
                    cap(lambda: self._backward(gx, gy, global_batch, None, sample_offset, device_step=True))
                    cap(tail)
                torch.cuda.synchronize(self.device)
                # capture does not execute, but be safe against any eager side effect: restore the optimizer state
                for t, k in zip((self._params_all, self._m_all, self._v_all, self._step_dev, self._noise_step_dev), keep):
                    t.copy_(k)
        except Exception as e:       # noqa: BLE001 -- an unsupported capture falls back to eager launches, loudly
            import warnings
            warnings.warn(f"CUDA-graph capture of the train step failed ({e!r}); continuing with eager launches")
            self._graph_failed = True
            self._set_device_step(False)
            return None
        g = dict(graphs=graphs, x=gx, y=gy, launches=int(self._lib.dib_launch_count()) - launches0)
        self._graphs[key] = g
        return g

    def _replay_step(self, g, x, y, world):
        P = self._PQ
        if not self._step_dev_active or self._step_dev_dirty:
            self._set_device_step(True)
        self._replayed_launches += g["launches"]
        g["x"].copy_(x.reshape(g["x"].shape), non_blocking=True)
        g["y"].copy_(y.reshape(g["y"].shape), non_blocking=True)
        if world == 1:
            g["graphs"][0].replay()
        elif self.overlap_allreduce:
            self._reduce_overlapped(world, g["graphs"][0].replay, g["graphs"][1].replay)
            g["graphs"][2].replay()
        else:
            g["graphs"][0].replay()
            parallel.allreduce_sum_(self._gradstats, self.process_group)
            g["graphs"][1].replay()
        self._train_step_count += 1
        return self._gradstats[P:]

    def compute_gradients(self, x, y, eps=None, global_batch=None, sample_offset=0, step=None):
        """GradientTape-style access (nb-bool cell 6 / train.py:201-220 custom loops): returns
        (flat gradient of task + beta*sum KL w.r.t. trainable_variables, statistics vector) as device tensors."""
        with torch.cuda.device(self.device):
            xd = self._to_device(x, sum(self.feature_dimensionalities))
            yd = self._to_device(y, self._y_cols())
            e = self._to_device(eps) if eps is not None else None
            self._backward(xd, yd, global_batch or max(xd.shape[0], 1), e, sample_offset, step)
            return self._gradstats[:self._PQ].clone(), self._gradstats[self._PQ:].clone()

    # ------------------------------------------------------------------ encoder-only custom steps (SURVEY 8f3)
    def encode(self, x, eps=None, step=None, sample_offset=0):
        """Every feature encoder + reparameterisation, without the integration network (nb-particle cell 8's
        ``particle_encoder`` front end): returns (emb [n, F*E] = mu + exp(logvar/2) eps, KL_i batch means [F]) as device
        tensors.  Noise as in ``__call__``: explicit ``eps``, Philox keyed by ``step``, or a fresh draw."""
        with torch.cuda.device(self.device):
            xd = self._to_device(x, sum(self.feature_dimensionalities))
            e = self._to_device(eps) if eps is not None else None
            n = xd.shape[0]
            self._ensure_handle(n)
            st = self._inference_step() if step is None else step
            emb = torch.empty(n, self.number_features * self.feature_embedding_dimension, dtype=torch.float32, device=self.device)
            stats = torch.empty(self.number_features + 3, dtype=torch.float32, device=self.device)
            _lib.check(self._lib.dib_encoders_forward(
                self._handle, _lib.ptr(self._params), _lib.ptr(xd), n, _lib.ptr(e), self.noise_seed, int(st) & 0xFFFFFFFF,
                int(sample_offset), _lib.ptr(emb), _lib.ptr(stats), _lib.ptr(self._workspace), _stream()))
            return emb, stats[:self.number_features] / max(n, 1)

    def encoder_gradients(self, x, d_emb, global_batch=None, eps=None, step=None, sample_offset=0):
        """Reverse mode of :meth:`encode` for a caller-owned downstream network: ``d_emb`` [n, F*E] is d(caller's loss)/d(emb)
        (already carrying the caller's batch scaling); the IB term beta * scale * (sum KL)^p, with KL means over
        ``global_batch`` rows (default n), is added here.  Returns (flat gradient [P] -- integration entries are zero --,
        statistics vector).  Pass the same ``eps`` / ``step`` as the ``encode`` call it differentiates."""
        with torch.cuda.device(self.device):
            xd = self._to_device(x, sum(self.feature_dimensionalities))
            gd = self._to_device(d_emb, self.number_features * self.feature_embedding_dimension)
            e = self._to_device(eps) if eps is not None else None
            n = xd.shape[0]
            self._ensure_handle(n)
            st = self._train_step_count if step is None else step
            P = self._P
            _lib.check(self._lib.dib_encoders_backward(
                self._handle, _lib.ptr(self._params), _lib.ptr(xd), _lib.ptr(gd), n, _lib.ptr(self.beta._dev),
                1.0 / float(global_batch or max(n, 1)), _lib.ptr(e), self.noise_seed, int(st) & 0xFFFFFFFF, int(sample_offset),
                _lib.ptr(self._gradstats), _lib.ptr(self._gradstats[P:]), _lib.ptr(self._workspace), _stream()))
            return self._gradstats[:P].clone(), self._gradstats[P:].clone()

    def debug_force_unfused(self, on=True, batch_hint=1):
        """Bring-up switch: keep the tensor-core mode on the unfused kernels (fused-vs-unfused comparisons)."""
        self._force_unfused = int(on)          # bit 0: unfused encoders, bit 1: fp32-storage integration network
        if self._handle is not None:
            _lib.check(self._lib.dib_debug_force_unfused(self._handle, int(on)))

    def epoch_permutation(self, epoch, n):
        """The shuffle Model.fit applies in ``epoch`` (our RNG stream; Keras' own is irreproducible)."""
        gen = torch.Generator(device=self.device)
        gen.manual_seed((self.seed << 20) + epoch)
        return torch.randperm(n, generator=gen, device=self.device)

    def _metrics_update(self, stats):
        _lib.check(self._lib.dib_metrics_update_ex(_lib.ptr(stats), _lib.ptr(self.beta._dev), _lib.ptr(self._epoch_acc),
                                                   self.number_features, self.kl_loss_exponent, self.kl_loss_scale, _stream()))

    def _read_epoch_logs(self, prefix=""):
        F = self.number_features
        a = self._epoch_acc.detach().cpu().numpy().astype(np.float64)       # one D2H per epoch
        n, nb = max(a[F + 2], 1.0), max(a[F + 3], 1.0)
        logs = {prefix + "loss": float(a[F] / n)}
        for m in self.compiled_metrics_names:
            logs[prefix + m] = float(a[F + 1] / n)
        for i in range(F):
            logs[f"{prefix}KL{i}"] = float(a[i] / nb)                        # add_metric mean over batches (models.py:115)
        logs[prefix + "beta"] = float(self.beta.value())                     # models.py:121
        return logs

    # ------------------------------------------------------------------ Keras-like public surface
    def _inference_step(self):
        """Philox 'step' word of an un-seeded inference call: bit 31 marks inference (training steps count from 0),
        bit 30 separates it from the validation passes of fit, the low bits count calls -- every call draws fresh
        noise like tf.random.normal at models.py:108 does."""
        self._inference_calls += 1
        return (3 << 30) | (self._inference_calls & 0x3FFFFFFF)

    def __call__(self, inputs, training=None, eps=None, step=None, sample_offset=0):
        """models.py:96-123.  Returns the prediction; ``model.losses`` then holds [beta * sum_i KL_i] and
        ``model.metrics_values`` the KL{i}/beta metrics, as add_loss/add_metric leave them in the reference.
        Noise: explicit ``eps`` [n, F, E], or Philox keyed by ``step`` (reproducible), or -- default -- a fresh draw
        on every call."""
        with torch.cuda.device(self.device):
            x = self._to_device(inputs, sum(self.feature_dimensionalities))
            e = self._to_device(eps) if eps is not None else None
            st = self._inference_step() if step is None else step
            pred, _, stats = self._forward(x, None, e, st, sample_offset)
            n = x.shape[0]
            kl = stats[:self.number_features] / max(n, 1)
            self.losses = [self.beta._dev[0] * self.kl_loss_scale * kl.sum() ** self.kl_loss_exponent]
            self._last_kl = kl
            self.metrics_values = {"beta": self.beta.value()}
        return _as_numpy_like(inputs, pred)

    call = __call__

    def compile(self, optimizer='adam', loss=None, metrics=None, **_):
        """train.py:138-142."""
        new_opt = optimizers.get(optimizer)
        kind = resolve_loss(loss)
        if kind == "infonce":
            nce = loss if isinstance(loss, InfoNCE) else InfoNCE()
            self._check_infonce(nce, metrics)
        elif self.output_encoder is not None:
            # the optimizer buffers and gradient/statistics layout now span [model P | output encoder Q]
            raise ValueError("this model has an InfoNCE output encoder: compile it with loss=InfoNCE")
        old_nce = self._infonce
        if kind == "infonce":
            self._infonce = nce
        # captured steps carry the loss (and the InfoNCE similarity / temperature) by value: re-capture after a change
        sig = lambda c: None if c is None else (c.similarity_type, c.temperature)
        if kind != self._loss_kind or (kind == "infonce" and sig(nce) != sig(old_nce)):
            self._graphs.clear(); self._graph_seen.clear()
        if new_opt is not self.optimizer:        # a fresh Keras optimizer has fresh slots and iteration count
            self._m_all.zero_(); self._v_all.zero_(); self._step_dev.zero_()
        self.optimizer = new_opt
        self._loss_kind = kind
        self.compiled_metrics_names = []
        for m in (metrics or []):
            if m not in ("accuracy", "acc"):
                raise ValueError(f"only metrics=['accuracy'] is implemented (reference data.py:67), got {m!r}")
            self.compiled_metrics_names.append("accuracy")
        self._lr_host = None
        self._sync_lr()

    def _check_infonce(self, loss, metrics):
        """compile(loss=InfoNCE(...)): what the InfoNCE step supports."""
        if metrics:
            raise ValueError(f"compile(loss=InfoNCE) takes no metrics (the InfoNCE path reports loss, KL{{i}} and beta), got {metrics!r}")
        if self.output_activation_fn not in (None, "linear"):
            raise ValueError("InfoNCE needs a linear output activation: the model output is the embedding e1 (train.py:117)")
        if loss.similarity_type in ("l2sq", "l2", "cosine") and self.output_dimensionality > 256:
            raise ValueError(f"InfoNCE with similarity {loss.similarity_type!r} needs output_dimensionality <= 256, "
                             f"got {self.output_dimensionality}")
        world, _ = parallel.world_and_rank(self.process_group)
        if world > 1:
            raise NotImplementedError("data-parallel InfoNCE training is not implemented: the loss couples every row of the "
                                      "global batch")
        if self.output_encoder is not None and self.output_encoder.architecture != loss.output_encoder_architecture:
            raise ValueError("the output encoder is already built with a different architecture")

    def _sync_lr(self):
        """Device copy of optimizer.learning_rate (the step kernels read it from memory so that a schedule needs no re-capture);
        refreshed only when the host value changed -- one fill kernel per step otherwise."""
        lr = float(self.optimizer.learning_rate)
        if lr != getattr(self, "_lr_host", None):
            self._lr_dev.fill_(lr)
            self._lr_host = lr

    def train_on_batch(self, x, y, return_dict=True, sync=True):
        """One optimizer step on a (host or device) batch.

        ``sync=True`` (Keras behaviour): returns the batch metrics (dict, or the scalar loss) -- forces the D2H read.
        ``sync=False``: returns a :class:`PendingBatchResult`; host batches are staged through a copy stream with two
        device slots and the metrics are copied to pinned memory asynchronously, so the H2D copy of call k+1 overlaps
        the compute of call k.  ``result.get()`` (or the next sync point) yields the same dict."""
        if self.optimizer is None:
            raise RuntimeError("call compile() first")
        with torch.cuda.device(self.device):
            self._sync_lr()
            D = sum(self.feature_dimensionalities)
            world, rank = parallel.world_and_rank(self.process_group)
            host_x = not (isinstance(x, torch.Tensor) and x.is_cuda)
            if self._loss_kind == "infonce" and self.output_encoder is None:
                self.build_output_encoder(int(np.shape(y)[-1]) if np.ndim(y) > 1 else 1)
            if sync or not host_x:
                xd, yd = self._to_device(x, D), self._to_device(y, self._y_cols())
                n = xd.shape[0]
                stats = self._train_step(xd, yd, global_batch=n * world, sample_offset=rank * n)
                res = PendingBatchResult(self, stats.detach().clone() if not sync else stats, None, None)
            else:
                xd, yd, slot = self._stage_async(x, y, D)
                n = xd.shape[0]
                stats = self._train_step(xd, yd, global_batch=n * world, sample_offset=rank * n)
                st = self._staging
                st["done"][slot].record(torch.cuda.current_stream())          # slot may be overwritten after this
                hi = (st["k"] - 1) % len(st["stats_host"])
                if st["pending"][hi] is not None:
                    st["pending"][hi].get()                                   # its pinned buffer is about to be reused
                host = st["stats_host"][hi]
                host.copy_(stats, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream())
                res = PendingBatchResult(self, None, host, ev)
                st["pending"][hi] = res
        if not sync:
            return res
        out = res.get()
        return out if return_dict else out["loss"]

    def _stage_async(self, x, y, D):
        """H2D of a host batch on the copy stream into one of two device slots; the compute stream waits on it."""
        xt = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        yt = y if isinstance(y, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(y, dtype=np.float32))
        n, yc = xt.shape[0], self._y_cols()
        st = getattr(self, "_staging", None)
        if st is None or st["n"] != n:
            st = dict(n=n, k=0, stream=torch.cuda.Stream(device=self.device),
                      x=[torch.empty(n, D, dtype=torch.float32, device=self.device) for _ in range(2)],
                      y=[torch.empty((n, yc) if yc > 0 else (n,), dtype=torch.float32, device=self.device) for _ in range(2)],
                      done=[torch.cuda.Event() for _ in range(2)], copied=[torch.cuda.Event() for _ in range(2)],
                      stats_host=[torch.empty(self.number_features + 3, dtype=torch.float32).pin_memory() for _ in range(8)],
                      pending=[None] * 8, used=[False, False])
            self._staging = st
        slot = st["k"] % 2
        st["k"] += 1
        cs = st["stream"]
        if st["used"][slot]:
            cs.wait_event(st["done"][slot])                   # the step that read this slot two calls ago has finished
        with torch.cuda.stream(cs):
            st["x"][slot].copy_(xt.reshape(n, D), non_blocking=True)
            st["y"][slot].copy_(yt.reshape(st["y"][slot].shape), non_blocking=True)
            st["copied"][slot].record(cs)
        torch.cuda.current_stream().wait_event(st["copied"][slot])
        st["used"][slot] = True
        return st["x"][slot], st["y"][slot], slot

    def fit(self, x=None, y=None, batch_size=None, epochs=1, verbose='auto', callbacks=None, validation_data=None,
            shuffle=True, initial_epoch=0, **_):
        """Keras ``Model.fit`` mechanics around the fused step (train.py:157-166, nb-radial cell 10): per epoch
        on_epoch_begin -> shuffled consecutive batches incl. a short last one -> running means -> validation pass
        (noise sampled, train.py:264-265) -> on_epoch_end; returns a History whose ``.history`` has the keys
        loss, accuracy, KL{i}, beta and their val_ twins.

        Data-parallel: with torch.distributed initialised every rank passes the SAME x, y; each global batch is
        split into contiguous row ranges per rank, so the result does not depend on the number of GPUs."""
        if self.optimizer is None:
            raise RuntimeError("call compile() first")
        batch_size = 32 if batch_size is None else int(batch_size)
        if self._loss_kind == "infonce":
            return self._fit_infonce(x, y, batch_size, epochs, verbose, callbacks, validation_data, shuffle, initial_epoch)
        world, rank = parallel.world_and_rank(self.process_group)
        D = sum(self.feature_dimensionalities)
        with torch.cuda.device(self.device):
            xd, yd = self._to_device(x, D), self._to_device(y, self._y_cols())
            N = xd.shape[0]
            xv = yv = None
            if validation_data is not None:
                xv, yv = self._to_device(validation_data[0], D), self._to_device(validation_data[1], self._y_cols())
            history = History()
            cbs = list(callbacks or []) + [history]
            for cb in cbs:
                cb.set_model(self) if hasattr(cb, "set_model") else setattr(cb, "model", self)
            self.history = history
            self.stop_training = False
            for cb in cbs:
                getattr(cb, "on_train_begin", lambda logs=None: None)()
            for epoch in range(initial_epoch, epochs):
                for cb in cbs:
                    cb.on_epoch_begin(epoch, logs=None)                      # beta annealing lives here
                self._sync_lr()
                if shuffle:
                    perm = self.epoch_permutation(epoch, N)
                self._epoch_acc.zero_()
                for b0 in range(0, N, batch_size):
                    b1 = min(b0 + batch_size, N)
                    lo, hi = parallel.shard_range(b1 - b0, rank, world)
                    if shuffle:
                        idx = perm[b0 + lo:b0 + hi]
                        xb, yb = xd.index_select(0, idx), yd.index_select(0, idx)
                    else:
                        xb, yb = xd[b0 + lo:b0 + hi], yd[b0 + lo:b0 + hi]
                    stats = self._train_step(xb, yb, global_batch=b1 - b0, sample_offset=lo)
                    self._metrics_update(stats)
                logs = self._read_epoch_logs()
                if xv is not None:
                    logs.update(self._evaluate_into_logs(xv, yv, batch_size, epoch, world, rank))
                if verbose not in (False, 0) and rank == 0:          # 'auto' -> 1 like Keras outside notebooks
                    print(f"Epoch {epoch + 1}/{epochs} - " + " - ".join(
                        f"{k}: {v:.4g}" for k, v in logs.items() if not k.removeprefix('val_').startswith('KL')))
                for cb in cbs:
                    cb.on_epoch_end(epoch, logs)
                if self.stop_training:
                    break
            for cb in cbs:
                getattr(cb, "on_train_end", lambda logs=None: None)()
        return history

    def _evaluate_into_logs(self, xv, yv, batch_size, epoch, world, rank):
        Nv = xv.shape[0]
        self._epoch_acc.zero_()
        stats = torch.empty(self.number_features + 3, dtype=torch.float32, device=self.device)
        for b0 in range(0, Nv, batch_size):
            b1 = min(b0 + batch_size, Nv)
            lo, hi = parallel.shard_range(b1 - b0, rank, world)
            self._forward(xv[b0 + lo:b0 + hi], yv[b0 + lo:b0 + hi], None, (2 ** 31 + epoch), b0 + lo,
                          want_pred=False, stats_out=stats)
            parallel.allreduce_sum_(stats, self.process_group)
            self._metrics_update(stats)
        return self._read_epoch_logs(prefix="val_")

    # ------------------------------------------------------------------ InfoNCE fit / evaluate (train.py:220-271)
    def _fit_infonce(self, x, y, batch_size, epochs, verbose, callbacks, validation_data, shuffle, initial_epoch):
        """fit for compile(loss=InfoNCE): full batches only.  Training step s reads rows [sB, (s+1)B) of the stream
        perm_0 || perm_1 || ... (perm_k = epoch_permutation(k, N), or arange(N) with shuffle=False: train.py:224's repeated
        dataset); epoch e runs steps [r(e), r(e+1)) with r(e) = np.round(e N / B) (train.py:236's epoch boundaries).  beta is
        set by the callbacks' on_epoch_begin as in the Keras path -- train.py:241-250 changes it after the first step of an
        epoch instead.  Validation: floor(Nv / B) + 1 full batches of consecutive rows of the repeated validation set
        (train.py:230-234), noise keyed (2**31 + epoch, position in that stream).  Training noise: (optimizer step, row)."""
        B = batch_size
        with torch.cuda.device(self.device):
            if self.output_encoder is None:
                self.build_output_encoder(int(np.shape(y)[-1]) if np.ndim(y) > 1 else 1)
            D = sum(self.feature_dimensionalities)
            xd, yd = self._to_device(x, D), self._to_device(y, self._y_cols())
            N = xd.shape[0]
            if N < 1:
                raise ValueError("fit needs at least one sample")
            xv = yv = None
            if validation_data is not None:
                xv, yv = self._to_device(validation_data[0], D), self._to_device(validation_data[1], self._y_cols())
            history = History()
            cbs = list(callbacks or []) + [history]
            for cb in cbs:
                cb.set_model(self) if hasattr(cb, "set_model") else setattr(cb, "model", self)
            self.history = history
            self.stop_training = False
            for cb in cbs:
                getattr(cb, "on_train_begin", lambda logs=None: None)()
            perms = {}

            def stream_rows(s):
                lo, hi = s * B, (s + 1) * B
                parts = []
                while lo < hi:
                    k, r0 = divmod(lo, N)
                    if k not in perms:
                        perms[k] = self.epoch_permutation(k, N) if shuffle else torch.arange(N, device=self.device)
                        for old in [j for j in perms if j < k - 1]:
                            del perms[old]
                    take = min(hi - lo, N - r0)
                    parts.append(perms[k][r0:r0 + take])
                    lo += take
                return parts[0] if len(parts) == 1 else torch.cat(parts)

            r = lambda e: int(np.round(e * N / B))
            for epoch in range(initial_epoch, epochs):
                for cb in cbs:
                    cb.on_epoch_begin(epoch, logs=None)
                self._sync_lr()
                self._epoch_acc.zero_()
                for s in range(r(epoch), r(epoch + 1)):
                    idx = stream_rows(s)
                    stats = self._train_step(xd.index_select(0, idx), yd.index_select(0, idx), global_batch=B)
                    self._metrics_update(stats)
                logs = self._read_epoch_logs()
                if xv is not None:
                    logs.update(self._evaluate_infonce(xv, yv, B, 2 ** 31 + epoch, prefix="val_"))
                if verbose not in (False, 0):
                    print(f"Epoch {epoch + 1}/{epochs} - " + " - ".join(
                        f"{k}: {v:.4g}" for k, v in logs.items() if not k.removeprefix('val_').startswith('KL')))
                for cb in cbs:
                    cb.on_epoch_end(epoch, logs)
                if self.stop_training:
                    break
            for cb in cbs:
                getattr(cb, "on_train_end", lambda logs=None: None)()
        return history

    def _evaluate_infonce(self, xv, yv, B, step, prefix=""):
        Nv = xv.shape[0]
        self._epoch_acc.zero_()
        stats = torch.empty(self.number_features + 3, dtype=torch.float32, device=self.device)
        for b in range(Nv // B + 1):
            idx = torch.arange(b * B, (b + 1) * B, device=self.device) % Nv
            self._infonce_call(xv.index_select(0, idx), yv.index_select(0, idx), step, b * B, train=False, stats_out=stats)
            self._metrics_update(stats)
        return self._read_epoch_logs(prefix=prefix)

    def evaluate(self, x, y, batch_size=32, return_dict=True, **_):
        if self._loss_kind == "infonce":
            with torch.cuda.device(self.device):
                if self.output_encoder is None:
                    self.build_output_encoder(int(np.shape(y)[-1]) if np.ndim(y) > 1 else 1)
                self._inference_calls += 1
                D = sum(self.feature_dimensionalities)
                logs = self._evaluate_infonce(self._to_device(x, D), self._to_device(y, self._y_cols()), int(batch_size),
                                              (1 << 29) | (self._inference_calls & 0x1FFFFFFF))
            return logs if return_dict else [logs["loss"]]
        with torch.cuda.device(self.device):
            world, rank = parallel.world_and_rank(self.process_group)
            D = sum(self.feature_dimensionalities)
            self._inference_calls += 1           # a fresh noise draw per evaluate() call
            logs = self._evaluate_into_logs(self._to_device(x, D), self._to_device(y, self._y_cols()), int(batch_size),
                                            (1 << 29) | (self._inference_calls & 0x1FFFFFFF), world, rank)
        logs = {k[len("val_"):]: v for k, v in logs.items()}
        return logs if return_dict else [logs["loss"]] + [logs[m] for m in self.compiled_metrics_names]

    def predict(self, x, batch_size=32, **_):
        outs = []
        n = len(x)
        st = self._inference_step()              # one noise stream per predict(); rows keyed by their global index
        for b0 in range(0, n, int(batch_size)):
            xb = x[b0:b0 + int(batch_size)]
            o = self(xb, training=False, step=st, sample_offset=b0)
            outs.append(o if isinstance(x, torch.Tensor) else np.asarray(o))
        return torch.cat(outs) if isinstance(x, torch.Tensor) else np.concatenate(outs)


class PendingBatchResult:
    """Metrics of one ``train_on_batch(..., sync=False)`` call; ``get()`` waits for the asynchronous D2H copy."""

    def __init__(self, model, stats_dev, stats_host, event):
        self._m, self._dev, self._host, self._ev = model, stats_dev, stats_host, event
        self._beta = float(model.beta.value())
        self._out = None

    def get(self):
        if self._out is None:
            if self._ev is not None:
                self._ev.synchronize()
                s = self._host.numpy().astype(np.float64)            # copy out of the pinned buffer
            else:
                s = self._dev.detach().cpu().numpy().astype(np.float64)
            F = self._m.number_features
            nn = max(s[F + 2], 1.0)
            m = self._m
            ib = self._beta * m.kl_loss_scale * (s[:F].sum() / nn) ** m.kl_loss_exponent      # models.py:118 / nb-chaos
            out = {"loss": float(s[F] / nn + ib)}
            if m._loss_kind != "infonce":                     # the InfoNCE path has no accuracy
                out["accuracy"] = float(s[F + 1] / nn)
            for i in range(F):
                out[f"KL{i}"] = float(s[i] / nn)
            self._out = out
        return self._out

    def __getitem__(self, k):
        return self.get()[k]


class OutputEncoder(_Network):
    """model.output_encoder of the InfoNCE path (train.py:186-193): y [n, input_dimensionality] -> [PositionalEncoding] ->
    Dense(w, activation_fn) per width -> Dense(output_dimensionality) -> e2.  Its variables are the [P, P+Q) tail of the
    buffer the optimizer updates; ``model.trainable_variables`` / ``get_flat_weights`` stay the model's own."""

    def __init__(self, model, input_dimensionality, architecture):
        super().__init__(model, [])
        self.input_dimensionality = int(input_dimensionality)
        self.architecture = [int(w) for w in architecture]
        self._layout = None

    def _config(self):
        self._c_arch = (ctypes.c_int32 * max(len(self.architecture), 1))(*self.architecture)
        return _lib.DibOutputEncoderConfig(input_dimensionality=self.input_dimensionality, number_layers=len(self.architecture),
                                           architecture=self._c_arch)

    @property
    def weights(self):
        m = self._model
        out = []
        for off, r, c in zip(*self._layout):
            v = m._params_all[off:off + max(r, 1) * c]
            out.append(v.view(r, c) if r > 0 else v)
        return out

    trainable_variables = weights

    def set_weights(self, weights):
        vs = self.weights
        if len(weights) != len(vs):
            raise ValueError(f"expected {len(vs)} arrays, got {len(weights)}")
        for v, w in zip(vs, weights):
            v.copy_(torch.as_tensor(np.asarray(w), dtype=torch.float32).view(v.shape))

    def get_flat_weights(self):
        m = self._model
        return m._params_all[m._P:].detach().cpu().numpy()

    def set_flat_weights(self, flat):
        m = self._model
        m._params_all[m._P:].copy_(torch.as_tensor(np.asarray(flat), dtype=torch.float32))

    def count_params(self):
        return self._model._Q

    def __call__(self, y, training=None):
        m = self._model
        with torch.cuda.device(m.device):
            t = m._to_device(y, self.input_dimensionality)
            n = t.shape[0]
            if m._loss_kind != "infonce":
                raise RuntimeError("the output encoder runs on a model compiled with loss=InfoNCE")
            m._ensure_handle(max(n, 1))
            out = torch.empty(n, m.output_dimensionality, dtype=torch.float32, device=m.device)
            _lib.check(m._lib.dib_output_encoder_forward(m._handle, _lib.ptr(m._params_all), _lib.ptr(t), n, _lib.ptr(out),
                                                         _lib.ptr(m._workspace), _stream()))
        return _as_numpy_like(y, out)

    call = __call__


class InfoBottleneckAnnealingCallback(Callback):
    """Callback to logarithmically increase beta during training (models.py:125-149).  The schedule is
    evaluated in float32 exactly like the tf ops there:
        beta = exp(log b0 + float32(max(epoch - n_pre, 0)) / n_anneal * (log b1 - log b0))."""

    def __init__(self, beta_start, beta_end, number_pretraining_epochs, number_annealing_epochs):
        super().__init__()
        self.beta_start = beta_start
        self.beta_end = beta_end
        self.number_pretraining_epochs = number_pretraining_epochs
        self.number_annealing_epochs = number_annealing_epochs

    def beta_at(self, epoch):
        f = np.float32
        frac = f(max(epoch - self.number_pretraining_epochs, 0)) / f(self.number_annealing_epochs)
        lo, hi = np.log(f(self.beta_start)), np.log(f(self.beta_end))
        return f(np.exp(lo + frac * (hi - lo)))

    def on_epoch_begin(self, epoch, logs=None):
        self.model.beta.assign(self.beta_at(epoch))


class SaveCompressionMatricesCallback(Callback):
    """Callback to save compression scheme matrices during training (models.py:152-186; the intended behaviour is
    the inline copy at train.py:251-261 -- the shipped on_epoch_end raises NameError).  For every feature: pick
    <=128 rows as visualization.py:17-28 does, encoder forward, Bhattacharyya matrix, exp(-D) (all features in one
    device call, dib_compression_matrices).  The reference renders a PNG with matplotlib, which is not available
    here; the numeric artefact is saved as ``feature_{i}_log10beta_{x:.3f}.npz`` (same stem) and kept in
    ``self.matrices``."""

    def __init__(self, save_frequency, x_processed, x_raw, outdir, max_number_to_display=128, seed=0):
        super().__init__()
        self.save_frequency = save_frequency
        self.x_processed = x_processed
        self.x_raw = x_raw
        self.outdir = outdir
        self.max_number_to_display = max_number_to_display
        self.rng = np.random.default_rng(seed)
        self.matrices = []

    def on_epoch_end(self, epoch, logs=None):
        if (epoch % self.save_frequency) != 0:
            return
        from . import utils
        model = self.model
        beta_value = float(model.beta.value())
        xp = np.asarray(self.x_processed.cpu() if isinstance(self.x_processed, torch.Tensor) else self.x_processed)
        xr = np.asarray(self.x_raw.cpu() if isinstance(self.x_raw, torch.Tensor) else self.x_raw)
        offs = np.cumsum([0] + list(model.feature_dimensionalities))
        if self.outdir:
            os.makedirs(self.outdir, exist_ok=True)
        # row selection per feature on the host (visualization.py:17-28), then ONE device call for all features
        picks = [utils.select_display_rows(xr[:, offs[i]:offs[i + 1]], self.max_number_to_display, self.rng)
                 for i in range(model.number_features)]
        n = max(len(inds) for inds, _ in picks)
        row_index = np.stack([np.concatenate([inds, np.full(n - len(inds), inds[-1])]) for inds, _ in picks])
        res = model.compression_matrices(xp, row_index, want=("dist", "comp"))
        comp_all, dist_all = res["comp"].cpu().numpy(), res["dist"].cpu().numpy()
        for i, (inds, sorted_raw) in enumerate(picks):
            k = len(inds)
            rec = dict(epoch=epoch, feature=i, beta=beta_value, compression_matrix=comp_all[i, :k, :k],
                       bhattacharyya=dist_all[i, :k, :k], raw_values=sorted_raw)
            self.matrices.append(rec)
            if self.outdir:
                np.savez(os.path.join(self.outdir, f'feature_{i}_log10beta_{np.log10(beta_value):.3f}.npz'), **rec)


class StashEmbeddingsCallback(Callback):
    """nb-radial cell 5: stash (mu, logvar) of every feature encoder on ``x_in`` every ``save_frequency`` epochs."""

    def __init__(self, save_frequency, x_in, save_start=0):
        super().__init__()
        self.save_frequency = save_frequency
        self.x_in = x_in
        self.mus_for_later = []
        self.logvars_for_later = []
        self.save_start = save_start

    def on_epoch_end(self, epoch, logs=None):
        if (epoch > self.save_start) and ((epoch % self.save_frequency) == 0):
            m = self.model
            E = m.feature_embedding_dimension
            o = m.compression_matrices(self.x_in, None, want=("mu_logvar",))["mu_logvar"].cpu().numpy()
            for i in range(m.number_features):
                self.mus_for_later.append(o[i, :, :E])
                self.logvars_for_later.append(o[i, :, E:])


class InfoPerFeatureCallback(Callback):
    """Callback to compute the information contained in each compression channel during training (models.py:188-223;
    the shipped version passes wrong keyword names to utils -- this follows the corrected copy in nb-radial cell 5).
    ``self.bounds`` collects [lower, upper] (nats) per feature each time it fires, feature-major like the reference."""

    def __init__(self, save_frequency, tf_dataset_validation, evaluation_batch_size=None, number_evaluation_batches=None,
                 info_bound_batch_size=1024, info_bound_number_batches=8, seed=0):
        super().__init__()
        self.save_frequency = save_frequency
        data = tf_dataset_validation[0] if isinstance(tf_dataset_validation, (tuple, list)) else tf_dataset_validation
        self.x_validation = data                                     # the reference maps (x, y) -> x
        self.bounds = []
        self.evaluation_batch_size = evaluation_batch_size or info_bound_batch_size
        self.number_evaluation_batches = number_evaluation_batches or info_bound_number_batches
        self.seed = seed

    def on_epoch_end(self, epoch, logs=None):
        if (epoch % self.save_frequency) != 0:
            return
        from . import utils
        m = self.model
        x = self.x_validation
        xt = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        # all features x all evaluation batches in one grouped encoder pass + one float64 sandwich launch
        lo_up = utils.estimate_mi_sandwich_bounds_all_features(m, xt, evaluation_batch_size=self.evaluation_batch_size,
                                                               number_evaluation_batches=self.number_evaluation_batches,
                                                               seed=self.seed + epoch)
        for i in range(m.number_features):
            self.bounds.append([float(lo_up[i, 0]), float(lo_up[i, 1])])


class SimpleEncoder:
    """nb-bool cell 4: "Simple encoder for a binary-valued variable.  With two trainable constants, mu and logvar, this
    encoder maps +1/-1 to a normal distribution with mean +mu/-mu and log variance of logvar."  Stand-alone callable with
    the reference's surface (``mu_scaling``, ``logvar``, ``call``); to TRAIN a bank of them with the fused step build
    ``DistributedIBNet(feature_dimensionalities, 'simple', integration_arch, out, feature_embedding_dimension=1)``."""

    def __init__(self):
        self.mu_scaling = np.ones((1, 1), np.float32)
        self.logvar = -3.0 * np.ones((1, 1), np.float32)

    def build(self, input_shape=None):
        return

    def __call__(self, inputs):
        t = torch.as_tensor(inputs, dtype=torch.float32)
        out = torch.cat([t * float(self.mu_scaling[0, 0]), torch.ones_like(t) * float(self.logvar[0, 0])], -1)
        return _as_numpy_like(inputs, out)

    call = __call__

    @property
    def trainable_variables(self):
        return [self.mu_scaling, self.logvar]


class SharedParticleEncoder:
    """nb-particle cell 8's front end: ONE encoder MLP (positional encoding -> Dense stack -> (mu, logvar)) applied with
    shared weights to every particle of every neighbourhood, logvar offset (-3 there), KL summed over embedding dims AND
    particles and averaged over the batch -- i.e. a one-feature DistributedIBNet on B*particles rows whose KL means are
    taken over B.  The downstream network (the notebook's set transformer) is the caller's: ``encode`` returns
    [B, particles, E] embeddings, ``gradients`` takes d(loss)/d(embeddings) back."""

    def __init__(self, particle_feature_dimensions, particle_encoder_arch_spec, bottleneck_dimension=32,
                 number_positional_encoding_frequencies=5, activation_fn='leaky_relu', leaky_alpha=0.1,
                 logvar_initialization=-3., **kw):
        self.net = DistributedIBNet([int(particle_feature_dimensions)], list(particle_encoder_arch_spec), [], 1,
                                    use_positional_encoding=number_positional_encoding_frequencies > 1,
                                    number_positional_encoding_frequencies=number_positional_encoding_frequencies,
                                    activation_fn=activation_fn, feature_embedding_dimension=bottleneck_dimension,
                                    leaky_alpha=leaky_alpha, logvar_offset=logvar_initialization, **kw)
        self.net.compile(optimizer='adam', loss='external')
        self.beta = self.net.beta
        self.d = int(particle_feature_dimensions)
        self.E = int(bottleneck_dimension)

    def encode(self, batch_inp, eps=None, step=None):
        """batch_inp [B, particles, d] -> (embs_reparam [B, particles, E], kl = mean_B sum_{particles, E})."""
        t = torch.as_tensor(batch_inp, dtype=torch.float32)
        B, Np = t.shape[0], t.shape[1]
        e = None if eps is None else torch.as_tensor(eps, dtype=torch.float32).reshape(B * Np, 1, self.E)
        emb, kl_rows = self.net.encode(t.reshape(B * Np, self.d), eps=e, step=step)
        return emb.reshape(B, Np, self.E), kl_rows[0] * Np

    def gradients(self, batch_inp, d_embs, eps=None, step=None):
        """Flat encoder gradient of (caller's loss + beta * kl) given d(caller's loss)/d(embs_reparam) [B, particles, E]."""
        t = torch.as_tensor(batch_inp, dtype=torch.float32)
        B, Np = t.shape[0], t.shape[1]
        e = None if eps is None else torch.as_tensor(eps, dtype=torch.float32).reshape(B * Np, 1, self.E)
        g, _ = self.net.encoder_gradients(t.reshape(B * Np, self.d), torch.as_tensor(d_embs).reshape(B * Np, self.E),
                                          global_batch=B, eps=e, step=step)
        return g

    def apply_gradients(self, flat_grads):
        self.net.apply_gradients(flat_grads)
