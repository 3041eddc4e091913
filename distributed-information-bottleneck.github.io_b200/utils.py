"""Host-side mirror of the parts of the reference's ``utils.py`` / ``visualization.py`` that sit on the
compression-matrix path of SaveCompressionMatricesCallback (SURVEY.md section 8 a14)."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib


def _dev(a, device):
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device=device, dtype=torch.float32).contiguous()


def _pairwise(kind, mus1, logvars1, mus2, logvars2, device):
    if not torch.cuda.is_available():
        raise _lib.DibError("dib_b200 needs a CUDA device; there is no CPU path")
    lib = _lib.load()
    device = device or (mus1.device if isinstance(mus1, torch.Tensor) and mus1.is_cuda
                        else torch.device("cuda", torch.cuda.current_device()))
    ml1 = torch.cat([_dev(mus1, device), _dev(logvars1, device)], dim=1).contiguous()
    same = mus2 is None or (mus2 is mus1 and logvars2 is logvars1)
    ml2 = ml1 if same else torch.cat([_dev(mus2, device), _dev(logvars2, device)], dim=1).contiguous()
    if ml1.shape[1] != ml2.shape[1]:
        raise ValueError("embedding dimensions differ")
    n, m, E = ml1.shape[0], ml2.shape[0], ml1.shape[1] // 2
    out = torch.empty(n, m, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.dib_pairwise_gaussian(kind, _lib.ptr(ml1), n, _lib.ptr(ml2), m, E, _lib.ptr(out), None,
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out if isinstance(mus1, torch.Tensor) else out.cpu().numpy()


def bhattacharyya_dist_mat(mus1, logvars1, mus2=None, logvars2=None, device=None):
    """utils.py:177-212 (Bhattacharyya distances between diagonal Gaussians, [N, M]) on the GPU in the O(N*M*E)
    closed form (dib_pairwise_gaussian kind 0)."""
    return _pairwise(0, mus1, logvars1, mus2, logvars2, device)


def kl_divergence_mat(mus1, logvars1, mus2=None, logvars2=None, device=None):
    """utils.py:213-247: KL(N(mus1_i, e^logvars1_i) || N(mus2_j, e^logvars2_j)), [N, M] (dib_pairwise_gaussian kind 1)."""
    return _pairwise(1, mus1, logvars1, mus2, logvars2, device)


def select_display_rows(inp_features_raw, max_number_to_display=128, rng=None):
    """visualization.py:17-28: unique values if fewer than 10 distinct, else ``max_number_to_display`` random rows,
    sorted by raw value.  Returns (row indices into the input, sorted raw values)."""
    raw = np.asarray(inp_features_raw)
    flat = raw.reshape(raw.shape[0], -1)[:, 0]
    unique_vals, unique_inds = np.unique(flat, return_index=True)
    if len(unique_vals) < 10:
        return unique_inds[np.argsort(unique_vals)], np.sort(unique_vals)
    rng = rng or np.random.default_rng()
    sel = rng.choice(flat.shape[0], max_number_to_display)
    order = np.argsort(flat[sel])
    return sel[order], flat[sel][order]


def compression_matrix(feature_encoder, feature_inps):
    """visualization.py:30-34: encoder forward -> (mu, logvar) -> Bhattacharyya -> exp(-D).
    Returns (compression_matrix, bhattacharyya_distance_matrix) as numpy arrays."""
    lib = _lib.load()
    model = feature_encoder._model
    o = model._encode_feature(feature_encoder.index, feature_inps)            # [n, 2E] on the device
    n, E = o.shape[0], model.feature_embedding_dimension
    dist = torch.empty(n, n, dtype=torch.float32, device=o.device)
    comp = torch.empty(n, n, dtype=torch.float32, device=o.device)
    with torch.cuda.device(o.device):
        _lib.check(lib.dib_bhattacharyya(_lib.ptr(o), n, E, _lib.ptr(dist), _lib.ptr(comp),
                                         ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return comp.cpu().numpy(), dist.cpu().numpy()


def mi_sandwich_batch(mu_logvar, eps=None, seed=0, step=0):
    """One batch of utils.py:36-65 on the GPU (dib_mi_sandwich_bounds): (InfoNCE lower, leave-one-out upper) in nats.
    ``mu_logvar`` [n, 2E] on the device; ``eps`` [n, E] or None (Philox)."""
    lib = _lib.load()
    n, E = mu_logvar.shape[0], mu_logvar.shape[1] // 2
    dev = mu_logvar.device
    scratch = torch.empty(2 * n, dtype=torch.float32, device=dev)
    out = torch.empty(2, dtype=torch.float32, device=dev)
    e = None if eps is None else _dev(eps, dev)
    with torch.cuda.device(dev):
        _lib.check(lib.dib_mi_sandwich_bounds(_lib.ptr(mu_logvar.contiguous()), n, E, _lib.ptr(e), int(seed), int(step) & 0xFFFFFFFF,
                                              _lib.ptr(scratch), _lib.ptr(out),
                                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


def estimate_mi_sandwich_bounds(encoder, dataset, evaluation_batch_size=1024, number_evaluation_batches=8, seed=0):
    """utils.py:10-73: upper and lower bounds of the information transmitted by one feature encoder.

    ``encoder`` is ``model.feature_encoders[i]``; ``dataset`` the rows of that feature ([N, d_i] array or tensor; a
    ``(x, y)`` tuple is accepted and y dropped, as the reference's callback does).  Batches are drawn like the
    reference's ``repeat().shuffle().batch().take()``: ``number_evaluation_batches`` batches of
    ``evaluation_batch_size`` rows sampled (with our seeded RNG; the reference's shuffle is unseeded) from the
    repeated data.  Returns np.array([lower, upper]) in nats, the mean over batches."""
    if isinstance(dataset, (tuple, list)):
        dataset = dataset[0]
    model = encoder._model
    x = _dev(dataset, model.device)
    if x.dim() == 1:
        x = x[:, None]
    N = x.shape[0]
    gen = torch.Generator(device=model.device)
    gen.manual_seed(int(seed))
    outs = []
    for b in range(int(number_evaluation_batches)):
        idx = torch.randint(0, N, (int(evaluation_batch_size),), generator=gen, device=model.device)
        o = model._encode_feature(encoder.index, x.index_select(0, idx))
        outs.append(mi_sandwich_batch(o, None, seed=(int(seed) << 8) + encoder.index, step=b))
    return torch.stack(outs).mean(0).double().cpu().numpy()


def estimate_mi_sandwich_bounds_all_features(model, x, evaluation_batch_size=1024, number_evaluation_batches=8, seed=0):
    """utils.py:10-73 for EVERY feature encoder of ``model`` at once (what InfoPerFeatureCallback, models.py:188-223, loops
    over in Python): one grouped encoder forward on the gathered rows (dib_compression_matrices) and ONE launch of the
    batched float64 sandwich kernel (dib_mi_sandwich_bounds_batched) over features x batches groups.  Row draws and noise
    streams are those of the per-feature ``estimate_mi_sandwich_bounds`` calls with the same ``seed``.
    ``x``: [N, sum d_i] rows (a ``(x, y)`` tuple is accepted).  Returns a float64 array [F, 2] = (lower, upper) in nats."""
    if isinstance(x, (tuple, list)):
        x = x[0]
    lib = _lib.load()
    xd = _dev(x, model.device)
    N, F, E = xd.shape[0], model.number_features, model.feature_embedding_dimension
    bs, nb = int(evaluation_batch_size), int(number_evaluation_batches)
    gen = torch.Generator(device=model.device)
    gen.manual_seed(int(seed))
    idx = torch.cat([torch.randint(0, N, (bs,), generator=gen, device=model.device) for _ in range(nb)])
    row_index = idx.to(torch.int32).unsqueeze(0).expand(F, -1).contiguous()
    ml = model.compression_matrices(xd, row_index, want=("mu_logvar",))["mu_logvar"]          # [F, nb * bs, 2E]
    scratch = torch.empty(F * nb * bs * 2, dtype=torch.float64, device=model.device)
    out = torch.empty(F * nb, 2, dtype=torch.float64, device=model.device)
    with torch.cuda.device(model.device):
        _lib.check(lib.dib_mi_sandwich_bounds_batched(_lib.ptr(ml), F * nb, bs, E, None, int(seed), nb, _lib.ptr(scratch),
                                                      _lib.ptr(out), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.view(F, nb, 2).mean(1).cpu().numpy()


SIMILARITY_TYPES = {"l2sq": 0, "l2": 1, "l1": 2, "linf": 3, "cosine": 4}


def _similarity_kind(similarity_type):
    if similarity_type not in SIMILARITY_TYPES:
        raise ValueError(f"Similarity type not implemented: {similarity_type}")      # utils.py:172
    return SIMILARITY_TYPES[similarity_type]


def get_scaled_similarity(embeddings1, embeddings2, similarity_type, temperature):
    """utils.py:127-175 on the GPU (dib_scaled_similarity): [N, d], [M, d] -> [N, M] similarities / temperature."""
    kind = _similarity_kind(similarity_type)
    if not torch.cuda.is_available():
        raise _lib.DibError("dib_b200 needs a CUDA device; there is no CPU path")
    lib = _lib.load()
    device = (embeddings1.device if isinstance(embeddings1, torch.Tensor) and embeddings1.is_cuda
              else torch.device("cuda", torch.cuda.current_device()))
    e1, e2 = _dev(embeddings1, device), _dev(embeddings2, device)
    if e1.shape[1] != e2.shape[1]:
        raise ValueError("embedding dimensions differ")
    out = torch.empty(e1.shape[0], e2.shape[0], dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.dib_scaled_similarity(kind, _lib.ptr(e1), e1.shape[0], _lib.ptr(e2), e2.shape[0], e1.shape[1],
                                             float(temperature), _lib.ptr(out),
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out if isinstance(embeddings1, torch.Tensor) else out.cpu().numpy()


# the exact head (dib_infonce_head) keeps the n x n similarity matrix in scratch and stops here
_EXACT_HEAD_MAX_N = 32768
# similarities with a Gram form, which the streaming tensor-core head (dib_infonce_head_tc) computes
_GRAM_KINDS = (SIMILARITY_TYPES["l2sq"], SIMILARITY_TYPES["l2"], SIMILARITY_TYPES["cosine"])


def _infonce_inputs(embeddings1, embeddings2):
    device = (embeddings1.device if isinstance(embeddings1, torch.Tensor) and embeddings1.is_cuda
              else torch.device("cuda", torch.cuda.current_device()))
    e1, e2 = _dev(embeddings1, device), _dev(embeddings2, device)
    if e1.shape != e2.shape:
        raise ValueError("the InfoNCE loss needs two [n, d] batches of equal shape (train.py:222-223)")
    loss = torch.empty(1, dtype=torch.float32, device=device)
    return device, e1, e2, loss


def infonce_loss_and_grads(embeddings1, embeddings2, similarity_type, temperature, want_grads=True):
    """The InfoNCE head of the custom loop (train.py:203-213) with its reverse mode (dib_infonce_head).
    Returns (loss [1], d loss/d embeddings1, d loss/d embeddings2) as device tensors (grads None if not wanted).
    Batches above 32768 rows, where the exact head's n x n scratch no longer fits, run on the streaming tensor-core head
    (dib_infonce_head_tc) for 'l2sq', 'l2' and 'cosine'; 'l1' and 'linf' have no such path and raise there."""
    kind = _similarity_kind(similarity_type)
    lib = _lib.load()
    device, e1, e2, loss = _infonce_inputs(embeddings1, embeddings2)
    n, d = e1.shape
    if n > _EXACT_HEAD_MAX_N and kind in _GRAM_KINDS:
        return _infonce_head_tc(e1, e2, kind, temperature, want_grads)
    scratch = torch.empty(n * n + 4 * n, dtype=torch.float32, device=device)
    d1 = torch.empty_like(e1) if want_grads else None
    d2 = torch.empty_like(e2) if want_grads else None
    with torch.cuda.device(device):
        _lib.check(lib.dib_infonce_head(kind, _lib.ptr(e1), _lib.ptr(e2), n, d, float(temperature), _lib.ptr(scratch),
                                        _lib.ptr(loss), _lib.ptr(d1), _lib.ptr(d2),
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return loss, d1, d2


def _infonce_head_tc(embeddings1, embeddings2, kind, temperature, want_grads=True):
    """dib_infonce_head_tc at any n: the same (loss, d_e1, d_e2) as dib_infonce_head, streamed on the tensor cores."""
    lib = _lib.load()
    device, e1, e2, loss = _infonce_inputs(embeddings1, embeddings2)
    n, d = e1.shape
    nbytes = lib.dib_infonce_head_tc_scratch_bytes(n, d)
    if nbytes < 0:
        raise ValueError(f"the tensor-core InfoNCE head takes 1 <= n <= 2^26 rows of d <= 256 (got n={n}, d={d})")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=device)
    d1 = torch.empty_like(e1) if want_grads else None
    d2 = torch.empty_like(e2) if want_grads else None
    with torch.cuda.device(device):
        _lib.check(lib.dib_infonce_head_tc(kind, _lib.ptr(e1), _lib.ptr(e2), n, d, float(temperature), _lib.ptr(scratch),
                                           _lib.ptr(loss), _lib.ptr(d1), _lib.ptr(d2),
                                           ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return loss, d1, d2
