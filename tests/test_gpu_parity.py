"""GPU (B200): the CUDA path, called through the C ABI (ctypes) by the dib_b200 host shim, against
 (a) the committed golden vectors produced by the reference's own code (tests/golden/),
 (b) the float64 CPU oracle on the same seeded inputs,
 (c) size-independent properties at the BASELINE batch (65 536): shard additivity, determinism.
Tolerances are fp32-vs-float64 reduction-order tolerances and are written next to each check."""
import os

import numpy as np
import pytest
import torch

from oracle import dib_oracle as O
from oracle import philox

pytestmark = pytest.mark.gpu

CASES = ["c0_small", "pendulum_like", "radial_like", "odd_shapes"]
LOSS_OF = {"c0_small": ("bce_logits", O.LOSS_BCE_LOGITS), "pendulum_like": ("mse", O.LOSS_MSE),
           "radial_like": ("bce_logits", O.LOSS_BCE_LOGITS), "odd_shapes": ("sparse_ce_logits", O.LOSS_SPARSE_CE_LOGITS)}


def build_model(cfg, precision="fp32", loss="bce_logits", lr=1e-3, seed=0):
    import dib_b200
    m = dib_b200.DistributedIBNet(
        cfg.feature_dimensionalities, cfg.feature_encoder_architecture, cfg.integration_network_architecture,
        cfg.output_dimensionality, use_positional_encoding=cfg.use_positional_encoding,
        number_positional_encoding_frequencies=cfg.number_positional_encoding_frequencies,
        activation_fn=cfg.activation_fn, feature_embedding_dimension=cfg.feature_embedding_dimension,
        output_activation_fn=cfg.output_activation_fn, precision=precision, seed=seed, leaky_alpha=cfg.leaky_alpha)
    m.compile(optimizer=dib_b200.Adam(lr), loss=loss, metrics=["accuracy"])
    return m


def load_case(golden_dir, name):
    return O.load_forward_golden(os.path.join(golden_dir, f"ref_forward_{name}.npz"))


def make_labels(rng, loss, B, out):
    if loss == O.LOSS_SPARSE_CE_LOGITS:
        return rng.integers(0, out, size=B).astype(np.float32)
    if loss == O.LOSS_BCE_LOGITS:
        return rng.integers(0, 2, size=(B, out)).astype(np.float32)
    return rng.standard_normal((B, out)).astype(np.float32)


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize("name", CASES)
def test_forward_matches_reference_goldens(golden_dir, name):
    cfg, z = load_case(golden_dir, name)
    m = build_model(cfg, loss=LOSS_OF[name][0])
    m.set_flat_weights(z["params"])
    m.beta.assign(float(z["beta"]))
    pred = m(z["x"], eps=z["eps"])
    assert rel_err(pred, z["pred"]) < 2e-5                       # fp32 FMA vs float64
    kl = (m._last_kl).cpu().numpy()
    np.testing.assert_allclose(kl, z["kl"], rtol=2e-5)
    np.testing.assert_allclose(float(m.losses[0]), float(z["ib_loss"]), rtol=2e-5)
    offs = np.cumsum([0] + list(cfg.feature_dimensionalities))
    for i in range(cfg.number_features):
        o = m.feature_encoders[i](z["x"][:, offs[i]:offs[i + 1]])
        assert rel_err(o, z[f"enc{i}"]) < 2e-5, i


@pytest.mark.parametrize("name", CASES)
def test_train_step_gradients_match_oracle(golden_dir, name):
    cfg, z = load_case(golden_dir, name)
    loss_name, loss = LOSS_OF[name]
    m = build_model(cfg, loss=loss_name)
    m.set_flat_weights(z["params"])
    beta = float(z["beta"])
    m.beta.assign(beta)
    rng = np.random.default_rng(5)
    y = make_labels(rng, loss, z["x"].shape[0], cfg.output_dimensionality)
    g, stats = m.compute_gradients(z["x"], y, eps=z["eps"])
    g_ref, fr = O.train_grads(cfg, z["params"], z["x"], y, z["eps"], beta, loss)
    assert rel_err(g.cpu().numpy(), g_ref) < 5e-5
    # per-variable check so that small-magnitude layers are not hidden by large ones
    off = 0
    for s in cfg.param_shapes():
        n = int(np.prod(s))
        assert rel_err(g.cpu().numpy()[off:off + n], g_ref[off:off + n]) < 2e-4, (off, s)
        off += n
    st = stats.cpu().numpy()
    B, F = z["x"].shape[0], cfg.number_features
    np.testing.assert_allclose(st[:F] / B, fr.kl_per_feature, rtol=2e-5)
    np.testing.assert_allclose(st[F] / B, fr.task_loss, rtol=2e-5)
    np.testing.assert_allclose(st[F + 1], fr.acc_sum, rtol=1e-6)
    assert st[F + 2] == B


def test_in_kernel_philox_matches_oracle_generator():
    cfg = O.DIBConfig([1] * 4, [32], [32], 1, feature_embedding_dimension=8)
    m = build_model(cfg)
    rng = np.random.default_rng(0)
    p = O.glorot_uniform_params(cfg, rng)
    m.set_flat_weights(p)
    x = rng.standard_normal((300, 4)).astype(np.float32)
    m.noise_seed = 0x1234567887654321
    with torch.cuda.device(m.device):
        xd = m._to_device(x, 4)
        _, emb, _ = m._forward(xd, None, None, step=17, sample_offset=1000, want_emb=True)
    eps = philox.normal_noise(0x1234567887654321, 17, np.arange(300) + 1000, 4, 8, dtype=np.float64)
    fr = O.forward(cfg, p, x, eps, 1.0)
    assert rel_err(emb.cpu().numpy(), fr.emb) < 2e-5
    # and the noise alone: u - mu over sigma
    fr0 = O.forward(cfg, p, x, np.zeros_like(eps), 1.0)
    encs, _ = O.unflatten(cfg, p.astype(np.float64))


def test_adam_matches_keras_semantics_oracle():
    import ctypes
    from dib_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(3)
    n = 10007
    w = rng.standard_normal(n).astype(np.float32)
    st = O.AdamState(np.zeros(n, np.float32), np.zeros(n, np.float32))
    w_ref = w.copy()
    dev = torch.device("cuda")
    wd, md, vd = torch.from_numpy(w).to(dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    lr = torch.full((1,), 3e-4, device=dev)
    step = torch.zeros(1, dtype=torch.int32, device=dev)
    for t in range(5):
        g = (rng.standard_normal(n) * 10.0 ** rng.integers(-6, 1, n)).astype(np.float32)
        O.adam_step(w_ref, g, st, 3e-4)
        gd = torch.from_numpy(g).to(dev)
        _lib.check(lib.dib_adam_step(_lib.ptr(wd), _lib.ptr(gd), _lib.ptr(md), _lib.ptr(vd), n, _lib.ptr(lr),
                                     _lib.ptr(step), 0.9, 0.999, 1e-7,
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert int(step.item()) == 5
    np.testing.assert_allclose(wd.cpu().numpy(), w_ref, rtol=1e-6, atol=1e-7)
    # m is a sum of terms of mixed sign: compare against its scale (cancellation leaves ~1 ulp of the largest term)
    np.testing.assert_allclose(md.cpu().numpy(), st.m, rtol=1e-5, atol=1e-6 * np.abs(st.m).max())
    np.testing.assert_allclose(vd.cpu().numpy(), st.v, rtol=1e-5, atol=1e-20)


def test_bhattacharyya_matches_reference_golden(golden_dir):
    import dib_b200
    z = np.load(os.path.join(golden_dir, "ref_bhattacharyya.npz"))
    D = dib_b200.utils.bhattacharyya_dist_mat(z["mu"], z["lv"], z["mu"], z["lv"])
    np.testing.assert_allclose(D, z["D"], rtol=2e-5, atol=2e-5)
    D34 = dib_b200.utils.bhattacharyya_dist_mat(z["mu3"], z["lv3"], z["mu4"], z["lv4"])
    np.testing.assert_allclose(D34, z["D34"], rtol=2e-5, atol=2e-5)
    D2 = dib_b200.utils.bhattacharyya_dist_mat(z["mu2"], z["lv2"])
    np.testing.assert_allclose(D2[0, 1], 0.48466528, rtol=1e-5)       # SURVEY.md section 4 KAT
    np.testing.assert_allclose(np.diag(D2), 0, atol=1e-6)


def test_fit_history_matches_oracle_fit():
    """Keras fit mechanics (shuffle, short last batch, weighted/unweighted means, validation pass with noise,
    beta callback) end to end on the paper's Boolean circuit, against the float64 oracle with the same
    permutations, noise and initial weights."""
    import dib_b200
    x, y = O.boolean_circuit_truth_table()
    cfg = O.DIBConfig([1] * 10, [32, 32], [64], 1, feature_embedding_dimension=8)
    m = build_model(cfg, lr=2e-3, seed=4)
    m.noise_seed = 99
    p0 = m.get_flat_weights().copy()
    cb = dib_b200.InfoBottleneckAnnealingCallback(1e-3, 1e-1, 1, 3)
    hist = m.fit(x, y, epochs=4, batch_size=100, shuffle=True, callbacks=[cb], verbose=False,
                 validation_data=(x[:250], y[:250])).history
    perms = {e: m.epoch_permutation(e, 1024).cpu().numpy() for e in range(4)}
    eps_fn = lambda step, ids: philox.normal_noise(99, step, ids, 10, 8, dtype=np.float64)
    p_ref, h_ref = O.fit(cfg, p0, x.astype(np.float64), y.astype(np.float64), loss=O.LOSS_BCE_LOGITS, epochs=4,
                         batch_size=100, lr=2e-3, eps_fn=eps_fn, perm_fn=lambda e, n: perms[e],
                         beta_fn=lambda e: O.beta_schedule(e, 1e-3, 1e-1, 1, 3),
                         validation_data=(x[:250].astype(np.float64), y[:250].astype(np.float64)))
    assert set(hist) == set(h_ref)
    for k in h_ref:
        # 44 Adam steps of fp32-vs-float64 drift; accuracy can flip single samples -> looser
        tol = 2e-2 if "accuracy" in k else 2e-3
        np.testing.assert_allclose(hist[k], h_ref[k], rtol=tol, atol=1e-6, err_msg=k)
    assert rel_err(m.get_flat_weights(), p_ref) < 2e-3


@pytest.mark.parametrize("n", [1, 2, 127, 129, 257, 1000])
def test_ragged_batch_sizes(n):
    cfg = O.DIBConfig([1, 3], [16, 12], [20], 2, feature_embedding_dimension=5, activation_fn="tanh",
                      number_positional_encoding_frequencies=2)
    m = build_model(cfg, loss="mse")
    rng = np.random.default_rng(n)
    p = O.glorot_uniform_params(cfg, rng)
    m.set_flat_weights(p)
    m.beta.assign(0.1)
    x = rng.standard_normal((n, 4)).astype(np.float32)
    eps = rng.standard_normal((n, 2, 5)).astype(np.float32)
    y = rng.standard_normal((n, 2)).astype(np.float32)
    g, stats = m.compute_gradients(x, y, eps=eps)
    g_ref, fr = O.train_grads(cfg, p, x, y, eps, 0.1, O.LOSS_MSE)
    assert rel_err(g.cpu().numpy(), g_ref) < 5e-5
    np.testing.assert_allclose(stats.cpu().numpy()[2] / n, fr.task_loss, rtol=5e-5)


def test_empty_batch_is_a_no_op():
    cfg = O.DIBConfig([1, 1], [8], [8], 1, feature_embedding_dimension=4)
    m = build_model(cfg)
    g, stats = m.compute_gradients(np.zeros((0, 2), np.float32), np.zeros((0, 1), np.float32))
    assert float(g.abs().sum()) == 0 and float(stats.abs().sum()) == 0


def test_full_size_properties_c0():
    """BASELINE config C0 at the full batch (65 536 x 16): (i) bit-reproducible, (ii) data-parallel shards are
    additive: grads(full) == grads(rows 0..B/2) + grads(rows B/2..B) with global sample offsets, (iii) gradient of
    a random direction agrees with a finite difference of the loss reported by the forward entry point."""
    cfg = O.DIBConfig([1] * 16, [128, 128], [256, 256], 1)
    m = build_model(cfg, seed=1)
    B = 65536
    rng = np.random.default_rng(0)
    x = rng.standard_normal((B, 16)).astype(np.float32)
    y = (x[:, 0] * x[:, 1] + np.sin(2 * x[:, 2]) + 0.5 * x[:, 3] > 0).astype(np.float32)[:, None]
    m.beta.assign(1e-2)
    g1, s1 = m.compute_gradients(x, y, step=3)
    g2, s2 = m.compute_gradients(x, y, step=3)
    assert torch.equal(g1, g2) and torch.equal(s1, s2)                       # (i)
    h = B // 2
    ga, sa = m.compute_gradients(x[:h], y[:h], global_batch=B, sample_offset=0, step=3)
    gb, sb = m.compute_gradients(x[h:], y[h:], global_batch=B, sample_offset=h, step=3)
    assert rel_err((ga + gb).cpu().numpy(), g1.cpu().numpy()) < 1e-5         # (ii)
    np.testing.assert_allclose((sa + sb).cpu().numpy(), s1.cpu().numpy(), rtol=1e-5)
    # (iii) directional derivative
    F = 16
    def loss_at(flat):
        m.set_flat_weights(flat)
        with torch.cuda.device(m.device):
            _, _, st = m._forward(m._to_device(x, 16), m._to_device(y, 1), None, 3, 0, want_pred=False)
        st = st.cpu().numpy().astype(np.float64)
        return (st[F] + 1e-2 * st[:F].sum()) / B
    p = m.get_flat_weights().astype(np.float64)
    gv = g1.cpu().numpy().astype(np.float64)
    d = gv / np.linalg.norm(gv)                       # steepest direction: derivative = |g|, well above fp32 loss noise
    hh = 0.05
    fd = (loss_at((p + hh * d).astype(np.float32)) - loss_at((p - hh * d).astype(np.float32))) / (2 * hh)
    m.set_flat_weights(p.astype(np.float32))
    an = float(gv @ d)
    assert abs(fd - an) < 5e-2 * abs(an), (fd, an)


def test_compression_matrix_callback(tmp_path):
    import dib_b200
    x, y = O.boolean_circuit_truth_table()
    cfg = O.DIBConfig([1] * 10, [16], [16], 1, feature_embedding_dimension=4)
    m = build_model(cfg)
    cb = dib_b200.SaveCompressionMatricesCallback(1, x, x, str(tmp_path))
    stash = dib_b200.StashEmbeddingsCallback(1, x[:32], save_start=-1)
    m.fit(x, y, epochs=1, batch_size=256, callbacks=[dib_b200.InfoBottleneckAnnealingCallback(1e-3, 1, 0, 2), cb, stash])
    assert len(cb.matrices) == 10
    rec = cb.matrices[3]
    assert rec["compression_matrix"].shape == (2, 2)                         # binary feature: 2 unique values
    ref = O.compression_matrix(cfg, m.get_flat_weights(), 3, np.array([[-1.0], [1.0]]))
    np.testing.assert_allclose(rec["compression_matrix"], ref, rtol=1e-4, atol=1e-5)
    assert os.path.exists(os.path.join(str(tmp_path), f"feature_3_log10beta_{np.log10(1e-3):.3f}.npz"))
    assert len(stash.mus_for_later) == 10 and stash.mus_for_later[0].shape == (32, 4)


def test_kl_divergence_mat_matches_reference_golden(golden_dir):
    """next row f2: utils.kl_divergence_mat (utils.py:213-247) through dib_pairwise_gaussian."""
    from dib_b200 import utils
    z = np.load(os.path.join(golden_dir, "ref_kl_divergence.npz"))
    np.testing.assert_allclose(utils.kl_divergence_mat(z["mu1"], z["lv1"], z["mu2"], z["lv2"]), z["KL12"], rtol=3e-5, atol=3e-5)
    K11 = utils.kl_divergence_mat(z["mu1"], z["lv1"])
    np.testing.assert_allclose(K11, z["KL11"], rtol=3e-5, atol=3e-5)
    np.testing.assert_allclose(np.diag(K11), 0, atol=1e-5)


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("tf32", 5e-3), ("fp16", 5e-3)])
def test_compression_matrices_all_features_in_one_call(precision, tol):
    """next row f2: dib_compression_matrices (all encoders as one grouped problem + batched Bhattacharyya) against the
    oracle's per-feature loop (visualization.py:14-35), with per-feature row gathers and without."""
    rng = np.random.default_rng(5)
    cfg = O.DIBConfig([2, 1, 3, 1], [64, 32], [32], 1, feature_embedding_dimension=8)
    m = build_model(cfg, precision=precision, seed=3)
    x = rng.standard_normal((300, 7)).astype(np.float32)
    row_index = np.stack([rng.choice(300, 96) for _ in range(4)])
    got = m.compression_matrices(x, row_index)
    ml, dist, comp = O.compression_matrices(cfg, m.get_flat_weights(), x, row_index)
    assert rel_err(got["mu_logvar"].cpu().numpy(), ml) < tol
    np.testing.assert_allclose(got["comp"].cpu().numpy(), comp, atol=10 * tol)
    if precision == "fp32":
        np.testing.assert_allclose(got["dist"].cpu().numpy(), dist, rtol=1e-4, atol=1e-4)
    got = m.compression_matrices(x[:50], None, want=("mu_logvar",))
    assert set(got) == {"mu_logvar"}
    assert rel_err(got["mu_logvar"].cpu().numpy(), O.compression_matrices(cfg, m.get_flat_weights(), x[:50])[0]) < tol
    for i in range(4):                                                   # same numbers as the per-feature a15 contract
        o = m.feature_encoders[i](x[:50, sum(cfg.feature_dimensionalities[:i]):sum(cfg.feature_dimensionalities[:i + 1])])
        np.testing.assert_allclose(np.asarray(o), got["mu_logvar"][i].cpu().numpy(), rtol=1e-6, atol=1e-6)


def test_mi_sandwich_bounds_kernel_and_callback(golden_dir):
    """next row f1: dib_mi_sandwich_bounds against the reference-code golden, the oracle with explicit and with Philox
    noise, and InfoPerFeatureCallback end to end on the Boolean circuit (binary features carry <= 1 bit each)."""
    import dib_b200
    from dib_b200 import utils
    z = np.load(os.path.join(golden_dir, "ref_mi_sandwich.npz"))
    bs, nb = int(z["bs"]), int(z["nb"])
    dev = torch.device("cuda")
    outs = []
    for b in range(nb):
        ml = torch.from_numpy(np.concatenate([z["mu"][b * bs:(b + 1) * bs], z["lv"][b * bs:(b + 1) * bs]], -1)).float().to(dev)
        outs.append(utils.mi_sandwich_batch(ml, z["eps"][b]).cpu().numpy())
    np.testing.assert_allclose(np.mean(outs, 0), z["bounds"], rtol=2e-5)
    rng = np.random.default_rng(1)
    n, E = 700, 32
    mu, lv = rng.standard_normal((n, E)), rng.standard_normal((n, E)) * 0.5 - 1.0
    ml = torch.from_numpy(np.concatenate([mu, lv], -1)).float().to(dev)
    got = utils.mi_sandwich_batch(ml, None, seed=77, step=3).cpu().numpy()
    eps = philox.normal_noise(77, 3, np.arange(n), 1, E, dtype=np.float64)[:, 0, :]
    np.testing.assert_allclose(got, O.mi_sandwich_batch(mu.astype(np.float32), lv.astype(np.float32), eps), rtol=1e-4, atol=1e-4)
    x, y = O.boolean_circuit_truth_table()
    cfg = O.DIBConfig([1] * 10, [32], [32], 1, feature_embedding_dimension=8)
    m = build_model(cfg, lr=3e-3)
    cb = dib_b200.InfoPerFeatureCallback(1, (x, y), evaluation_batch_size=256, number_evaluation_batches=2)
    m.fit(x, y, epochs=2, batch_size=256, callbacks=[dib_b200.InfoBottleneckAnnealingCallback(1e-4, 1e-3, 0, 2), cb])
    bounds = np.asarray(cb.bounds).reshape(2, 10, 2) / np.log(2)
    assert np.all(bounds[..., 0] <= bounds[..., 1] + 1e-4) and np.all(bounds[..., 0] < 1.0 + 1e-3) and np.all(bounds > -1e-3)


# ---------------------------------------------------------------------------------------------------------
# next row f3: custom training steps -- caller-owned loss (DIB_LOSS_EXTERNAL) and the InfoNCE head
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-3), ("tf32", 5e-3), ("fp16", 5e-3)])    # fp32 sums over 4160 rows vs float64
def test_external_loss_gradients_match_oracle(precision, tol):
    """dib_train_step with loss = external: y carries d(task)/d(pred).  The upstream gradient is the MSE gradient against
    random targets, so the step must equal (a) the oracle fed the same upstream gradient and (b) the compiled-MSE step
    of the same model.  4160 rows: in tensor-core mode single activation-sign flips under 11-bit operands are only
    invisible against a coherent gradient over a few thousand samples (cf. test_gpu_tf32)."""
    rng = np.random.default_rng(11)
    cfg = O.DIBConfig([1] * 4, [128, 128], [256, 256], 8, feature_embedding_dimension=32, output_activation_fn="tanh")
    B = 4096 + 64
    x = rng.standard_normal((B, 4)).astype(np.float32)
    y = rng.standard_normal((B, 8)).astype(np.float32)
    eps = rng.standard_normal((B, 4, 32)).astype(np.float32)
    m = build_model(cfg, precision=precision, loss="external", seed=2)
    m.beta.assign(0.05)
    p = m.get_flat_weights()
    fr = O.forward(cfg, p, x, eps, 0.05)
    pred = np.asarray(m(x, eps=eps))
    assert rel_err(pred, fr.pred) < tol
    d_pred = (O.task_loss_grad("mse", fr.pred, y) / B).astype(np.float32)
    g, stats = m.compute_gradients(x, d_pred, eps=eps)
    g_ref, _ = O.train_grads(cfg, p, x, d_pred, eps, 0.05, "external")
    assert rel_err(g.cpu().numpy(), g_ref) < tol
    st = stats.cpu().numpy()
    np.testing.assert_allclose(st[:4] / B, fr.kl_per_feature, rtol=10 * tol)
    assert st[4] == 0 and st[5] == 0 and st[6] == B
    m2 = build_model(cfg, precision=precision, loss="mse", seed=2)
    m2.beta.assign(0.05)
    g_mse, _ = m2.compute_gradients(x, y, eps=eps)
    # same kernels, same summation order: the caller-owned and the compiled loss agree far tighter than either with float64
    assert rel_err(g.cpu().numpy(), g_mse.cpu().numpy()) < (2e-5 if precision == "fp32" else 2 * tol)


def test_scaled_similarity_and_infonce_head(golden_dir):
    from dib_b200 import utils
    z = np.load(os.path.join(golden_dir, "ref_scaled_similarity.npz"))
    for kind in O.SIMILARITY_TYPES:
        got = utils.get_scaled_similarity(z["e1"], z["e2"], kind, float(z["temperature"]))
        np.testing.assert_allclose(got, z[kind], rtol=2e-5, atol=2e-5)
    with pytest.raises(ValueError):
        utils.get_scaled_similarity(z["e1"], z["e2"], "hamming", 1.0)
    rng = np.random.default_rng(8)
    for n, d in ((300, 32), (129, 200), (5, 3)):
        a, b = rng.standard_normal((n, d)).astype(np.float32), rng.standard_normal((n, d)).astype(np.float32)
        for kind in O.SIMILARITY_TYPES:
            T = 0.3 if kind == "cosine" else 2.0 * np.sqrt(d)
            loss, da, db = utils.infonce_loss_and_grads(a, b, kind, T)
            l_ref, da_ref, db_ref, _ = O.infonce_loss_and_grads(a, b, kind, T)
            np.testing.assert_allclose(loss.item(), l_ref, rtol=2e-5)
            assert rel_err(da.cpu().numpy(), da_ref) < 1e-4, (kind, n, d)
            assert rel_err(db.cpu().numpy(), db_ref) < 1e-4, (kind, n, d)


def test_infonce_custom_loop_trains():
    """train.py:201-220 end to end: model(x) -> InfoNCE head against an output encoder -> d_pred -> dib_train_step
    (external loss) -> apply_gradients.  The output encoder here is a fixed linear map (the reference trains an MLP;
    any torch module can own that side).  The loss must fall well below its chance level 2 ln(n)."""
    import dib_b200
    from dib_b200 import utils
    rng = np.random.default_rng(0)
    n, F, d = 256, 4, 16
    x = rng.standard_normal((n * 8, F)).astype(np.float32)
    y = np.stack([x[:, 0] * x[:, 1], np.sin(2 * x[:, 2]), x[:, 3]], -1).astype(np.float32)
    Wy = (rng.standard_normal((3, d)) * 0.8).astype(np.float32)
    cfg = O.DIBConfig([1] * F, [64, 64], [128], d, feature_embedding_dimension=8)
    m = build_model(cfg, loss="external", lr=2e-3, seed=1)
    m.beta.assign(1e-4)
    losses = []
    for step in range(60):
        sl = slice((step % 8) * n, (step % 8 + 1) * n)
        e1 = m(torch.from_numpy(x[sl]).cuda(), step=step)                       # forward with this step's noise
        e2 = torch.from_numpy(y[sl] @ Wy).cuda()
        loss, d_e1, _ = utils.infonce_loss_and_grads(e1, e2, "l2sq", 4.0)
        g, _ = m.compute_gradients(x[sl], d_e1, step=step)                      # same (seed, step) -> same noise
        m.apply_gradients(g)
        losses.append(loss.item())
    assert losses[0] > 0.9 * 2 * np.log(n) * 0.5 and np.mean(losses[-5:]) < 0.8 * np.mean(losses[:5])


# ---------------------------------------------------------------------------------------------------------
# next row f3 (continued): SimpleEncoder bank, shared particle encoder with logvar offset, nonlinear IB
# ---------------------------------------------------------------------------------------------------------
def test_simple_encoder_bank_matches_notebook_golden_and_oracle(golden_dir):
    """nb-bool cell 4/6: 10 SimpleEncoders (2 constants each, E = 1) + [256]*3 leaky-relu predictor.  Forward against the
    golden produced by executing the notebook's own SimpleEncoder class; one train step against the oracle."""
    import dib_b200
    z = np.load(os.path.join(golden_dir, "ref_simple_encoder.npz"))
    cfg = O.DIBConfig([1] * 10, [], [256, 256, 256], 1, use_positional_encoding=False, feature_embedding_dimension=1,
                      activation_fn="leaky_relu", encoder_kind="simple")
    m = dib_b200.DistributedIBNet([1] * 10, "simple", [256, 256, 256], 1, activation_fn="leaky_relu",
                                  feature_embedding_dimension=1, seed=3)
    m.compile(optimizer=dib_b200.Adam(1e-3), loss=dib_b200.losses.BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
    p0 = m.get_flat_weights()
    assert np.all(p0[0:20:2] == 1.0) and np.all(p0[1:20:2] == -3.0) and m.count_params() == cfg.param_count()
    p = p0.copy()
    p[:20] = z["enc_params"]
    m.set_flat_weights(p)
    for i in range(10):                                                       # a15 contract on the notebook's own class output
        np.testing.assert_allclose(np.asarray(m.feature_encoders[i](z["x"][:, i:i + 1])), z[f"enc{i}"], rtol=1e-6, atol=1e-7)
    emb, kl = m.encode(z["x"], eps=z["eps"])
    np.testing.assert_allclose(emb.cpu().numpy(), z["emb"], rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(kl.cpu().numpy(), z["kl"], rtol=2e-6)
    y = (z["x"][:, :1] * z["x"][:, 1:2] > 0).astype(np.float32)
    m.beta.assign(0.05)
    g, st = m.compute_gradients(z["x"], y, eps=z["eps"])
    g_ref, fr = O.train_grads(cfg, p, z["x"], y, z["eps"], 0.05, O.LOSS_BCE_LOGITS)
    assert rel_err(g.cpu().numpy(), g_ref) < 5e-5
    assert rel_err(g.cpu().numpy()[:20], g_ref[:20]) < 1e-4                   # the 20 encoder constants themselves
    out = m.train_on_batch(z["x"], y)                                         # per-step beta + Adam on the flat buffer
    assert np.isfinite(out["loss"])


@pytest.mark.parametrize("precision,tol", [("fp32", 5e-5), ("tf32", 5e-3)])
def test_shared_particle_encoder_with_logvar_offset(precision, tol):
    """nb-particle cell 8: one encoder shared by 50 particles (12 -> PE(60) -> 128 -> 128 -> 64, LeakyReLU(0.1)),
    logvar offset -3, KL summed over particles and dims, averaged over the batch; the downstream network is the caller's
    (a fixed random readout here).  Embeddings, KL and encoder gradients against the oracle."""
    import dib_b200
    rng = np.random.default_rng(2)
    B, Np, d, E = 8, 50, 12, 32
    enc = dib_b200.SharedParticleEncoder(d, [128, 128], E, seed=5, precision=precision)
    cfg = O.DIBConfig([d], [128, 128], [], 1, activation_fn="leaky_relu", leaky_alpha=0.1, feature_embedding_dimension=E,
                      logvar_offset=-3.0)
    p = enc.net.get_flat_weights()
    x = rng.standard_normal((B, Np, d)).astype(np.float32)
    eps = rng.standard_normal((B, Np, E)).astype(np.float32)
    enc.beta.assign(2e-1)
    embs, kl = enc.encode(x, eps=eps)
    fr = O.forward(cfg, p, x.reshape(B * Np, d), eps.reshape(B * Np, 1, E), 0.2)
    assert rel_err(embs.cpu().numpy().reshape(B * Np, E), fr.emb) < tol
    np.testing.assert_allclose(float(kl), fr.kl_per_feature[0] * Np, rtol=10 * tol)
    R = rng.standard_normal((B, Np, E)).astype(np.float32) / (B * Np)          # d loss / d embs of loss = sum(embs * R)
    g = enc.gradients(x, R, eps=eps).cpu().numpy()
    g_ref, _ = O.train_grads(cfg, p, x.reshape(B * Np, d), None, eps.reshape(B * Np, 1, E), 0.2, "external",
                             batch_for_mean=B, d_emb=R.reshape(B * Np, E))
    nenc = g_ref.size - (E * 1 + 1)
    assert rel_err(g[:nenc], g_ref[:nenc]) < (tol if precision == "fp32" else 4 * tol)      # 400 rows only in the tc mode
    assert np.all(g[nenc:] == 0)
    enc.apply_gradients(g)


def test_nonlinear_ib_weighting_matches_oracle():
    """nb-chaos cell 10: loss_IB = beta * number_states * KL ** 2 through the fused train step: gradients, reported loss."""
    import dib_b200
    rng = np.random.default_rng(4)
    cfg = O.DIBConfig([2], [128, 128], [64], 3, number_positional_encoding_frequencies=4, activation_fn="leaky_relu",
                      feature_embedding_dimension=8, kl_loss_exponent=2.0, kl_loss_scale=12.0)
    m = dib_b200.DistributedIBNet([2], [128, 128], [64], 3, number_positional_encoding_frequencies=4, activation_fn="leaky_relu",
                                  feature_embedding_dimension=8, kl_loss_exponent=2.0, kl_loss_scale=12.0, seed=6)
    m.compile(optimizer=dib_b200.Adam(3e-4), loss="mse")
    B = 300
    x = rng.standard_normal((B, 2)).astype(np.float32)
    y = rng.standard_normal((B, 3)).astype(np.float32)
    eps = rng.standard_normal((B, 1, 8)).astype(np.float32)
    p = m.get_flat_weights()
    m.beta.assign(0.7)
    g, st = m.compute_gradients(x, y, eps=eps)
    g_ref, fr = O.train_grads(cfg, p, x, y, eps, 0.7, O.LOSS_MSE)
    assert rel_err(g.cpu().numpy(), g_ref) < 5e-5
    pred = m(x, eps=eps)
    np.testing.assert_allclose(float(m.losses[0]), O.ib_loss(cfg, 0.7, fr.kl_per_feature), rtol=2e-5)
    out = m.train_on_batch(x, y)
    assert np.isfinite(out["loss"])


def test_mi_bounds_all_features_in_one_launch_matches_per_feature_loop_and_float64_oracle():
    """next row f1, batched (dib_mi_sandwich_bounds_batched): all features x all evaluation batches in one launch against
    (a) the per-feature / per-batch loop with the same row draws and noise streams, (b) the float64 oracle on the batched
    kernel's own inputs with explicit noise."""
    from dib_b200 import _lib, utils
    import ctypes
    cfg = O.DIBConfig([1, 2, 1], [64, 32], [32], 1, feature_embedding_dimension=8)
    m = build_model(cfg, seed=3)
    rng = np.random.default_rng(2)
    x = rng.standard_normal((3000, 4)).astype(np.float32)
    got = utils.estimate_mi_sandwich_bounds_all_features(m, x, evaluation_batch_size=256, number_evaluation_batches=3, seed=11)
    offs = [0, 1, 3, 4]
    for i in range(3):
        ref = utils.estimate_mi_sandwich_bounds(m.feature_encoders[i], x[:, offs[i]:offs[i + 1]], 256, 3, seed=11)
        np.testing.assert_allclose(got[i], ref, rtol=2e-5, atol=2e-6)           # the looped path accumulates in fp32
    assert got.dtype == np.float64 and np.all(got[:, 0] <= got[:, 1] + 1e-9)
    # (b) explicit noise, float64 oracle
    lib = _lib.load()
    G, n, E = 5, 300, 8
    mu, lv = rng.standard_normal((G, n, E)), rng.standard_normal((G, n, E)) * 0.5 - 1.0
    eps = rng.standard_normal((G, n, E)).astype(np.float32)
    dev = torch.device("cuda")
    ml = torch.from_numpy(np.concatenate([mu, lv], -1)).float().to(dev).contiguous()
    scratch = torch.empty(G * n * 2, dtype=torch.float64, device=dev)
    out = torch.empty(G, 2, dtype=torch.float64, device=dev)
    _lib.check(lib.dib_mi_sandwich_bounds_batched(_lib.ptr(ml), G, n, E, _lib.ptr(torch.from_numpy(eps).to(dev)), 0, 1,
                                                  _lib.ptr(scratch), _lib.ptr(out),
                                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    for g in range(G):
        ref = O.mi_sandwich_batch(mu[g].astype(np.float32), lv[g].astype(np.float32), eps[g].astype(np.float64))
        np.testing.assert_allclose(out[g].cpu().numpy(), ref, rtol=1e-9, atol=1e-9)     # float64 on both sides


@pytest.mark.parametrize("opt_name", ["sgd", "sgd_nesterov", "rmsprop", "rmsprop_momentum"])
def test_other_keras_optimizers_match_oracle(opt_name):
    """tf.keras.optimizers.get(name) beyond Adam (train.py:41,128): three steps through the public API against the
    oracle's restatement of the Keras / TensorFlow update rules."""
    import dib_b200
    cfg = O.DIBConfig([1, 2], [16], [12], 1, feature_embedding_dimension=4)
    rng = np.random.default_rng(9)
    opt = {"sgd": dib_b200.SGD(0.05), "sgd_nesterov": dib_b200.SGD(0.05, momentum=0.9, nesterov=True),
           "rmsprop": dib_b200.RMSprop(1e-2), "rmsprop_momentum": dib_b200.RMSprop(1e-2, rho=0.8, momentum=0.5)}[opt_name]
    m = build_model(cfg, seed=1)
    m.compile(optimizer=opt, loss="bce_logits", metrics=["accuracy"])
    p = m.get_flat_weights().copy()
    s1, s2 = np.zeros_like(p), np.zeros_like(p)
    m.beta.assign(0.1)
    for t in range(3):
        x = rng.standard_normal((50, 3)).astype(np.float32)
        y = (x[:, :1] > 0).astype(np.float32)
        eps = philox.normal_noise(m.noise_seed, t, np.arange(50), 2, 4, dtype=np.float64)
        g, _ = O.train_grads(cfg, p, x, y, eps, 0.1, O.LOSS_BCE_LOGITS)
        g = g.astype(np.float32)
        if opt_name.startswith("sgd"):
            O.sgd_step(p, g, s1, 0.05, opt.momentum, opt.nesterov)
        else:
            O.rmsprop_step(p, g, s1, s2, 1e-2, opt.rho, opt.momentum, opt.epsilon)
        m.train_on_batch(x, y)
    assert rel_err(m.get_flat_weights(), p) < 2e-5


def test_bce_on_probabilities_and_library_entry_points():
    """BinaryCrossentropy() with the Keras default from_logits=False on a sigmoid-output model; and the stand-alone
    model.integration_network(emb) / PositionalEncoding(freqs)(x) calls, which run in the library (no torch math)."""
    import dib_b200
    cfg = O.DIBConfig([1, 1, 2], [16, 8], [12, 10], 2, feature_embedding_dimension=4, output_activation_fn="sigmoid")
    rng = np.random.default_rng(10)
    m = build_model(cfg, seed=2)
    m.compile(optimizer="adam", loss=dib_b200.losses.BinaryCrossentropy(), metrics=["accuracy"])
    p = m.get_flat_weights()
    B = 70
    x = rng.standard_normal((B, 4)).astype(np.float32)
    y = rng.integers(0, 2, size=(B, 2)).astype(np.float32)
    eps = rng.standard_normal((B, 3, 4)).astype(np.float32)
    m.beta.assign(0.2)
    g, st = m.compute_gradients(x, y, eps=eps)
    g_ref, fr = O.train_grads(cfg, p, x, y, eps, 0.2, O.LOSS_BCE_PROBS)
    assert rel_err(g.cpu().numpy(), g_ref) < 5e-5
    np.testing.assert_allclose(st.cpu().numpy()[3] / B, fr.task_loss, rtol=2e-5)
    np.testing.assert_allclose(st.cpu().numpy()[4], fr.acc_sum, rtol=1e-6)
    # integration network as a callable
    emb = rng.standard_normal((33, 12)).astype(np.float32)
    got = m.integration_network(emb)
    _, integ = O.unflatten(cfg, p.astype(np.float64))
    h = emb.astype(np.float64)
    for k, (W, b) in enumerate(integ):
        h = O.act_fwd(cfg.activation_fn if k < len(integ) - 1 else cfg.output_activation_fn, h @ W + b)
    assert rel_err(got, h) < 2e-5
    # positional encoding as a callable (models.py:12-23)
    xs = rng.standard_normal((17, 3)).astype(np.float32)
    pe = dib_b200.PositionalEncoding(2 ** np.arange(1, 5))(xs)
    np.testing.assert_allclose(pe, O.positional_encoding(xs.astype(np.float64), [2, 4, 8, 16]), rtol=0, atol=2e-6)


@pytest.mark.parametrize("precision,tol", [("fp32", 5e-5), ("tf32", 5e-3)])
def test_dropout_in_feature_encoders_matches_oracle(precision, tol):
    """nb-radial cell 5: `dropout_rate` puts a Keras Dropout after every hidden Dense of the feature encoders.  Train-step
    gradients with the Philox-keyed masks against the oracle; inference (validation, model(x)) ignores dropout; `fit` runs."""
    import dib_b200
    cfg = O.DIBConfig([1] * 6, [128, 128], [256, 256, 256], 1, use_positional_encoding=False, activation_fn="tanh",
                      dropout_rate=0.25)
    rng = np.random.default_rng(12)
    B = 640
    x = rng.standard_normal((B, 6)).astype(np.float32)
    y = (x[:, :1] * x[:, 1:2] > 0).astype(np.float32)
    m = dib_b200.DistributedIBNet([1] * 6, [128, 128], [256, 256, 256], 1, use_positional_encoding=False, activation_fn="tanh",
                                  dropout_rate=0.25, precision=precision, seed=5)
    m.compile(optimizer=dib_b200.Adam(1e-4), loss=dib_b200.losses.BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
    m.noise_seed = 31
    p = m.get_flat_weights()
    m.beta.assign(0.01)
    eps = philox.normal_noise(31, 4, np.arange(B), 6, 32, dtype=np.float64)
    g, st = m.compute_gradients(x, y, step=4)
    g_ref, fr = O.train_grads(cfg, p, x, y, eps, 0.01, O.LOSS_BCE_LOGITS, dropout=(31, 4, np.arange(B)))
    assert rel_err(g.cpu().numpy(), g_ref) < tol
    g_nodrop, _ = O.train_grads(cfg, p, x, y, eps, 0.01, O.LOSS_BCE_LOGITS)
    assert rel_err(g_ref, g_nodrop) > 0.05                                   # the masks really change the step
    pred = np.asarray(m(x, step=4))                                          # inference: Dropout is the identity
    assert rel_err(pred, O.forward(cfg, p, x, eps, 0.01).pred) < tol
    h = m.fit(x, y, epochs=2, batch_size=128, verbose=False, validation_data=(x[:128], y[:128])).history
    assert np.isfinite(h["loss"]).all() and np.isfinite(h["val_loss"]).all()
