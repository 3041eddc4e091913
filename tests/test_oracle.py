"""CPU: the oracle against (i) golden vectors produced by the reference's own code (tests/golden/
make_golden.py), (ii) the closed-form known answers of SURVEY.md section 4, (iii) itself (finite differences,
torch-autograd twin, data-parallel shard additivity)."""
import os

import numpy as np
import pytest

from oracle import dib_oracle as O
from oracle import philox

CASES = ["c0_small", "pendulum_like", "radial_like", "odd_shapes"]


def load_case(golden_dir, name):
    return O.load_forward_golden(os.path.join(golden_dir, f"ref_forward_{name}.npz"))


@pytest.mark.parametrize("name", CASES)
def test_forward_matches_reference_code(golden_dir, name):
    cfg, z = load_case(golden_dir, name)
    fr = O.forward(cfg, z["params"], z["x"], z["eps"], float(z["beta"]))
    np.testing.assert_allclose(fr.pred, z["pred"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(fr.kl_per_feature, z["kl"], rtol=1e-12)
    np.testing.assert_allclose(float(z["beta"]) * fr.kl_per_feature.sum(), z["ib_loss"], rtol=1e-12)
    encs, _ = O.unflatten(cfg, z["params"].astype(np.float64))
    xs = O.split_features(cfg, z["x"].astype(np.float64))
    for i in range(cfg.number_features):
        np.testing.assert_allclose(O.encoder_forward(cfg, encs[i], xs[i]), z[f"enc{i}"], rtol=1e-12, atol=1e-12)


def test_beta_schedule_golden_and_kat(golden_dir):
    z = np.load(os.path.join(golden_dir, "ref_beta_schedule.npz"))
    for tag in ["train_py_defaults", "nb_radial", "bench"]:
        b0, b1, npre, nann = z[tag + "_args"]
        got = [O.beta_schedule(int(e), b0, b1, int(npre), int(nann)) for e in z[tag + "_epochs"]]
        np.testing.assert_array_equal(np.array(got, dtype=np.float32), z[tag + "_beta"])
    # SURVEY.md section 4 KAT values (evaluated from models.py:147-149)
    f = lambda e: O.beta_schedule(e, 1e-4, 3.0, 1000, 10000)
    assert f(0) == f(1000) == np.float32(9.999999e-05)
    np.testing.assert_allclose(f(1001), 1.0010313e-04, rtol=2e-7)
    np.testing.assert_allclose(f(6000), 1.7320503e-02, rtol=2e-6)
    np.testing.assert_allclose(f(10999), 2.9969075, rtol=2e-6)
    np.testing.assert_allclose(O.beta_schedule(249, 1e-6, 1.0, 0, 250), 0.94623667, rtol=2e-6)


def test_kl_closed_form_kat():
    mu = np.array([[1., -2.], [0., .5]])
    lv = np.array([[0., np.log(4.)], [-1., 1.]])
    per_row = (0.5 * (mu ** 2 + np.exp(lv) - lv - 1)).sum(-1)
    np.testing.assert_allclose(per_row, [3.30685282, 0.66808063], rtol=1e-8)
    np.testing.assert_allclose(per_row.mean(), 1.98746673, rtol=1e-8)


def test_kl_divergence_mat_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "ref_kl_divergence.npz"))
    np.testing.assert_allclose(O.kl_divergence_mat(z["mu1"], z["lv1"], z["mu2"], z["lv2"]), z["KL12"], rtol=1e-10, atol=1e-11)
    np.testing.assert_allclose(O.kl_divergence_mat(z["mu1"], z["lv1"], z["mu1"], z["lv1"]), z["KL11"], rtol=1e-10, atol=1e-11)


def test_compression_matrices_agree_with_single_feature_path():
    rng = np.random.default_rng(2)
    cfg = O.DIBConfig([2, 1], [8], [8], 1, feature_embedding_dimension=4)
    p = O.glorot_uniform_params(cfg, np.random.default_rng(0))
    x = rng.standard_normal((20, 3))
    idx = np.stack([rng.choice(20, 6), rng.choice(20, 6)])
    _, _, comp = O.compression_matrices(cfg, p, x, idx)
    np.testing.assert_allclose(comp[1], O.compression_matrix(cfg, p, 1, x[idx[1], 2:3]), rtol=1e-12)


def test_scaled_similarity_golden_and_infonce_grads_vs_autograd(golden_dir):
    """next row f3: similarity matrices against the reference's utils.get_scaled_similarity; the analytic InfoNCE
    gradients against torch autograd of the same loss (train.py:203-213)."""
    import torch
    z = np.load(os.path.join(golden_dir, "ref_scaled_similarity.npz"))
    for kind in O.SIMILARITY_TYPES:
        np.testing.assert_allclose(O.get_scaled_similarity(z["e1"], z["e2"], kind, float(z["temperature"])), z[kind],
                                   rtol=1e-9, atol=1e-9)
    rng = np.random.default_rng(0)
    a, b = rng.standard_normal((9, 5)), rng.standard_normal((9, 5))
    for kind in O.SIMILARITY_TYPES:
        loss, da, db, _ = O.infonce_loss_and_grads(a, b, kind, 0.5)
        ta, tb = torch.tensor(a, requires_grad=True), torch.tensor(b, requires_grad=True)
        diff = ta[:, None, :] - tb[None, :, :]
        if kind == "l2sq": S = -(diff ** 2).sum(-1)
        elif kind == "l2": S = -torch.sqrt((diff ** 2).sum(-1) + 1e-9)
        elif kind == "l1": S = -diff.abs().sum(-1)
        elif kind == "linf": S = -diff.abs().amax(-1)
        else: S = torch.nn.functional.normalize(ta, dim=-1, eps=0) @ torch.nn.functional.normalize(tb, dim=-1, eps=0).T
        S = S / 0.5
        lab = torch.arange(9)
        tl = torch.nn.functional.cross_entropy(S, lab) + torch.nn.functional.cross_entropy(S.T, lab)
        tl.backward()
        np.testing.assert_allclose(loss, tl.item(), rtol=1e-10)
        np.testing.assert_allclose(da, ta.grad.numpy(), rtol=1e-8, atol=1e-10)
        np.testing.assert_allclose(db, tb.grad.numpy(), rtol=1e-8, atol=1e-10)


def test_external_loss_gradients_equal_compiled_loss_gradients():
    """next row f3: handing the oracle d(task)/d(pred) of the compiled loss reproduces the compiled-loss gradients."""
    rng = np.random.default_rng(3)
    cfg = O.DIBConfig([1, 2], [8], [8], 2, feature_embedding_dimension=4, output_activation_fn="tanh")
    p = O.glorot_uniform_params(cfg, np.random.default_rng(1)).astype(np.float64)
    x, y = rng.standard_normal((12, 3)), rng.standard_normal((12, 2))
    eps = rng.standard_normal((12, 2, 4))
    g_ref, fr = O.train_grads(cfg, p, x, y, eps, 0.3, "mse")
    d_pred = O.task_loss_grad("mse", fr.pred, y) / 12
    g_ext, _ = O.train_grads(cfg, p, x, d_pred, eps, 0.3, "external")
    np.testing.assert_allclose(g_ext, g_ref, rtol=1e-12, atol=1e-14)


def test_bhattacharyya_golden_and_kat(golden_dir):
    z = np.load(os.path.join(golden_dir, "ref_bhattacharyya.npz"))
    np.testing.assert_allclose(O.bhattacharyya_dist_mat(z["mu"], z["lv"], z["mu"], z["lv"]), z["D"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(O.bhattacharyya_dist_mat(z["mu3"], z["lv3"], z["mu4"], z["lv4"]), z["D34"], rtol=1e-9, atol=1e-10)
    D2 = O.bhattacharyya_dist_mat(z["mu2"], z["lv2"], z["mu2"], z["lv2"])
    np.testing.assert_allclose(D2[0, 1], 0.48466528, rtol=1e-7)
    np.testing.assert_allclose(np.exp(-D2[0, 1]), 0.61590331, rtol=1e-7)
    np.testing.assert_allclose(np.diag(D2), 0, atol=1e-12)


def test_positional_encoding_layout():
    cfg = O.DIBConfig([2], [4], [4], 1)
    assert cfg.frequencies == [2, 4, 8, 16]
    x = np.array([[0.1, -0.3]])
    pe = O.positional_encoding(x, cfg.frequencies)
    assert pe.shape == (1, 10)
    np.testing.assert_allclose(pe[0], [0.1, -0.3, np.sin(.2), np.sin(-.6), np.sin(.4), np.sin(-1.2),
                                       np.sin(.8), np.sin(-2.4), np.sin(1.6), np.sin(-4.8)])


def test_boolean_circuit_truth_table_kat():
    x, y = O.boolean_circuit_truth_table()
    assert x.shape == (1024, 10) and set(np.unique(x)) == {-1.0, 1.0}
    assert y.sum() == 224
    p = y.mean()
    H = -(p * np.log2(p) + (1 - p) * np.log2(1 - p))
    np.testing.assert_allclose(H, 0.757878, atol=1e-6)
    # single-input mutual informations (bits), SURVEY.md section 4
    mi = []
    for j in range(10):
        m = 0.0
        for xv in (-1, 1):
            for yv in (0, 1):
                pxy = np.mean((x[:, j] == xv) & (y == yv))
                if pxy > 0:
                    m += pxy * np.log2(pxy / (np.mean(x[:, j] == xv) * np.mean(y == yv)))
        mi.append(m)
    np.testing.assert_allclose(mi, [0.0041, 0.0041, 0.2635, 0, 0, 0, 0.0010, 0, 0, 0.0524], atol=6e-5)


def test_param_count_c0():
    cfg = O.DIBConfig([1] * 16, [128, 128], [256, 256], 1)
    assert cfg.param_count() == 605953          # SURVEY.md section 8(a10)
    cfg = O.DIBConfig([1] * 100, [128, 128], [256] * 3, 1, use_positional_encoding=False)
    assert cfg.param_count() == 3453697         # nb-radial shape, SURVEY.md section 8(d)


def test_philox_known_answers():
    # Random123 kat_vectors for philox4x32-10
    r = philox.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(v) for v in r] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    r = philox.philox4x32_10(0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff)
    assert [int(v) for v in r] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    r = philox.philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0)
    assert [int(v) for v in r] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_philox_normal_moments_and_sharding():
    ids = np.arange(4096)
    e = philox.normal_noise(7, 3, ids, 4, 32)
    assert e.shape == (4096, 4, 32)
    assert abs(e.mean()) < 0.01 and abs(e.std() - 1) < 0.01
    # indexed by GLOBAL sample id: a shard sees exactly its rows
    e2 = philox.normal_noise(7, 3, ids[1000:1100], 4, 32)
    np.testing.assert_array_equal(e[1000:1100], e2)
    assert not np.allclose(e, philox.normal_noise(7, 4, ids, 4, 32))


@pytest.mark.parametrize("loss,out,act", [(O.LOSS_BCE_LOGITS, 1, "relu"), (O.LOSS_MSE, 3, "tanh"),
                                          (O.LOSS_SPARSE_CE_LOGITS, 4, "leaky_relu")])
def test_gradients_finite_difference(loss, out, act):
    rng = np.random.default_rng(0)
    cfg = O.DIBConfig([1, 2, 1], [8, 6], [10], out, activation_fn=act, feature_embedding_dimension=3,
                      number_positional_encoding_frequencies=3)
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64)
    p += 0.1 * rng.standard_normal(p.size)
    B = 5
    x = rng.standard_normal((B, 4))
    eps = rng.standard_normal((B, 3, 3))
    y = rng.integers(0, out, size=B).astype(np.float64) if loss == O.LOSS_SPARSE_CE_LOGITS else \
        (rng.integers(0, 2, size=(B, out)).astype(np.float64) if loss == O.LOSS_BCE_LOGITS else rng.standard_normal((B, out)))
    beta = 0.37
    g, fr = O.train_grads(cfg, p, x, y, eps, beta, loss)
    idx = rng.choice(p.size, size=40, replace=False)
    for j in idx:
        d = np.zeros_like(p)
        d[j] = 1e-6
        lp = O.forward(cfg, p + d, x, eps, beta, y=y, loss=loss).loss
        lm = O.forward(cfg, p - d, x, eps, beta, y=y, loss=loss).loss
        np.testing.assert_allclose(g[j], (lp - lm) / 2e-6, rtol=2e-4, atol=1e-8)


def test_data_parallel_shards_are_additive():
    rng = np.random.default_rng(1)
    cfg = O.DIBConfig([1] * 3, [8], [8], 1, feature_embedding_dimension=4)
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64)
    B = 12
    x, y = rng.standard_normal((B, 3)), rng.integers(0, 2, size=B).astype(np.float64)
    eps = rng.standard_normal((B, 3, 4))
    g, _ = O.train_grads(cfg, p, x, y, eps, 0.2, O.LOSS_BCE_LOGITS)
    parts = [O.train_grads(cfg, p, x[s], y[s], eps[s], 0.2, O.LOSS_BCE_LOGITS, batch_for_mean=B)[0]
             for s in (slice(0, 6), slice(6, 12))]
    np.testing.assert_allclose(parts[0] + parts[1], g, rtol=1e-10, atol=1e-14)


def test_fit_history_keys_and_learning():
    x, y = O.boolean_circuit_truth_table()
    cfg = O.DIBConfig([1] * 10, [16], [32], 1, feature_embedding_dimension=4)
    rng = np.random.default_rng(2)
    p0 = O.glorot_uniform_params(cfg, rng)
    eps_fn = lambda step, ids: philox.normal_noise(5, step, ids, 10, 4, dtype=np.float64)
    perm_fn = lambda e, n: np.random.default_rng(100 + e).permutation(n)
    _, h = O.fit(cfg, p0, x.astype(np.float64), y.astype(np.float64), loss=O.LOSS_BCE_LOGITS, epochs=3,
                 batch_size=100, lr=3e-3, eps_fn=eps_fn, perm_fn=perm_fn,
                 beta_fn=lambda e: O.beta_schedule(e, 1e-4, 1e-2, 1, 2), validation_data=(x.astype(np.float64), y.astype(np.float64)))
    for k in ["loss", "accuracy", "beta", "val_loss", "val_accuracy"] + [f"KL{i}" for i in range(10)] + [f"val_KL{i}" for i in range(10)]:
        assert len(h[k]) == 3
    assert h["loss"][-1] < h["loss"][0]
    assert h["beta"][0] == h["beta"][1] == float(np.float32(9.999999e-05))


def test_numpy_backward_matches_torch_autograd_twin():
    import torch
    from oracle.torch_twin import TwinDIB
    rng = np.random.default_rng(7)
    cfg = O.DIBConfig([1, 2, 1, 1], [16, 16], [24, 24], 1, feature_embedding_dimension=6)
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64) + 0.05 * rng.standard_normal(cfg.param_count())
    B = 33
    x, eps = rng.standard_normal((B, 5)), rng.standard_normal((B, 4, 6))
    y = rng.integers(0, 2, size=(B, 1)).astype(np.float64)
    g, fr = O.train_grads(cfg, p, x, y, eps, 0.3, O.LOSS_BCE_LOGITS)
    twin = TwinDIB(cfg, p).double()
    twin.load_flat(p)
    twin.beta = 0.3
    total, task, kls, pred = twin.loss(torch.from_numpy(x), torch.from_numpy(y), O.LOSS_BCE_LOGITS, torch.from_numpy(eps))
    total.backward()
    np.testing.assert_allclose(twin.flat_grads().numpy(), g, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(float(total), fr.loss, rtol=1e-12)
    np.testing.assert_allclose(kls.detach().numpy(), fr.kl_per_feature, rtol=1e-12)


def test_mi_sandwich_matches_reference_code_and_closed_forms(golden_dir):
    """next row f1: the oracle against utils.estimate_mi_sandwich_bounds executed from the reference (golden) and two
    closed forms: identical conditionals -> lower 0, upper log(bs/(bs-1)); k well separated clusters -> ~log k."""
    z = np.load(os.path.join(golden_dir, "ref_mi_sandwich.npz"))
    bs, nb = int(z["bs"]), int(z["nb"])
    out = [O.mi_sandwich_batch(z["mu"][b * bs:(b + 1) * bs], z["lv"][b * bs:(b + 1) * bs], z["eps"][b]) for b in range(nb)]
    np.testing.assert_allclose(np.mean(out, 0), z["bounds"], rtol=1e-10)
    rng = np.random.default_rng(0)
    bs, E = 32, 4
    lo, up = O.mi_sandwich_batch(np.zeros((bs, E)), np.zeros((bs, E)), rng.standard_normal((bs, E)))
    np.testing.assert_allclose([lo, up], [0.0, np.log(bs / (bs - 1))], atol=1e-12)
    k, bs = 4, 512
    lab = np.arange(bs) % k
    mu = np.stack([np.cos(2 * np.pi * lab / k), np.sin(2 * np.pi * lab / k)], -1) * 50.0
    lo, up = O.mi_sandwich_batch(mu, np.zeros((bs, 2)), rng.standard_normal((bs, 2)))
    np.testing.assert_allclose(lo, np.log(k), atol=1e-6)
    assert up >= lo - 1e-9


# ------------------------------------------------------------------------------------------------
# custom-step variants (SURVEY 8f3): SimpleEncoder bank, logvar offset, nonlinear IB, encoder-only reverse mode
# ------------------------------------------------------------------------------------------------
def test_simple_encoder_oracle_matches_notebook_golden(golden_dir):
    """tests/golden/ref_simple_encoder.npz comes from exec'ing nb-bool cell 4 (class SimpleEncoder) and the per-gate forward
    lines of its cell 6 verbatim (tests/golden/make_f3_golden.py)."""
    z = np.load(os.path.join(golden_dir, "ref_simple_encoder.npz"))
    cfg = O.DIBConfig([1] * 10, [], [256, 256, 256], 1, use_positional_encoding=False, feature_embedding_dimension=1,
                      activation_fn="leaky_relu", encoder_kind="simple")
    assert cfg.param_count() == 20 + (10 * 256 + 256) + 2 * (256 * 256 + 256) + 256 + 1
    p = O.glorot_uniform_params(cfg, np.random.default_rng(0), dtype=np.float64)
    assert np.all(p[0:20:2] == 1.0) and np.all(p[1:20:2] == -3.0)            # nb-bool cell 4 initial values
    p[:20] = z["enc_params"]
    fr = O.forward(cfg, p, z["x"], z["eps"], 0.1)
    np.testing.assert_allclose(fr.emb, z["emb"], rtol=1e-12)
    np.testing.assert_allclose(fr.kl_per_feature, z["kl"], rtol=1e-12)


@pytest.mark.parametrize("variant", ["simple", "offset_nonlinear", "encoder_only"])
def test_variant_gradients_match_finite_differences(variant):
    rng = np.random.default_rng(0)
    d_emb = None
    if variant == "simple":
        cfg = O.DIBConfig([1] * 3, [], [8], 1, use_positional_encoding=False, feature_embedding_dimension=1,
                          encoder_kind="simple", activation_fn="leaky_relu")
    else:
        cfg = O.DIBConfig([2, 1], [6], [5], 2, feature_embedding_dimension=3, logvar_offset=-3.0, kl_loss_exponent=2.0,
                          kl_loss_scale=12.0, activation_fn="tanh")
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64)
    p = p + 0.01 * rng.standard_normal(p.size)
    B, D = 7, sum(cfg.feature_dimensionalities)
    x = rng.standard_normal((B, D))
    y = rng.standard_normal((B, cfg.output_dimensionality))
    eps = rng.standard_normal((B, cfg.number_features, cfg.feature_embedding_dimension))
    if variant == "encoder_only":                                             # caller's loss = sum(emb * R)
        R = rng.standard_normal((B, cfg.number_features * cfg.feature_embedding_dimension))
        d_emb = R
        f = lambda q: float((O.forward(cfg, q, x, eps, 0.3).emb * R).sum()) + O.ib_loss(cfg, 0.3, O.forward(cfg, q, x, eps, 0.3).kl_per_feature)
        g, _ = O.train_grads(cfg, p, x, None, eps, 0.3, "external", d_emb=d_emb)
    else:
        f = lambda q: O.forward(cfg, q, x, eps, 0.3, y=y, loss=O.LOSS_MSE).loss
        g, _ = O.train_grads(cfg, p, x, y, eps, 0.3, O.LOSS_MSE)
    num = np.zeros_like(p)
    for i in range(p.size):
        dlt = np.zeros_like(p)
        dlt[i] = 1e-6
        num[i] = (f(p + dlt) - f(p - dlt)) / 2e-6
    n_enc = sum(int(np.prod(s)) for s in cfg.param_shapes()[:-2 * (len(cfg.integration_network_architecture) + 1)])
    if variant == "encoder_only":
        assert np.all(g[n_enc:] == 0)
        np.testing.assert_allclose(g[:n_enc], num[:n_enc], rtol=1e-5, atol=1e-7)
    else:
        np.testing.assert_allclose(g, num, rtol=1e-5, atol=1e-7)


def test_dropout_oracle_gradients_and_mask_statistics():
    """nb-radial cell 5 Dropout after every hidden encoder Dense: Philox-keyed masks keep a 1 - rate fraction, the
    backward applies the same scale mask (finite differences), inference ignores it."""
    rng = np.random.default_rng(0)
    cfg = O.DIBConfig([2, 1], [6, 5], [5], 2, feature_embedding_dimension=3, activation_fn="tanh", dropout_rate=0.3)
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64)
    p = p + 0.01 * rng.standard_normal(p.size)
    B = 9
    x, y, eps = rng.standard_normal((B, 3)), rng.standard_normal((B, 2)), rng.standard_normal((B, 2, 3))
    dr = (7, 3, np.arange(B) + 100)
    g, _ = O.train_grads(cfg, p, x, y, eps, 0.3, O.LOSS_MSE, dropout=dr)
    f = lambda q: O.forward(cfg, q, x, eps, 0.3, y=y, loss=O.LOSS_MSE, dropout=dr).loss
    num = np.zeros_like(p)
    for i in range(p.size):
        d = np.zeros_like(p)
        d[i] = 1e-6
        num[i] = (f(p + d) - f(p - d)) / 2e-6
    np.testing.assert_allclose(g, num, rtol=1e-5, atol=1e-7)
    keep = philox.dropout_keep(7, 3, np.arange(20000), 1, 2, 8, 0.3)
    assert abs(keep.mean() - 0.7) < 5e-3
    assert not np.array_equal(keep, philox.dropout_keep(7, 4, np.arange(20000), 1, 2, 8, 0.3))      # a new mask every step
    cfg0 = O.DIBConfig([2, 1], [6, 5], [5], 2, feature_embedding_dimension=3, activation_fn="tanh")
    np.testing.assert_array_equal(O.forward(cfg, p, x, eps, 0.3).pred, O.forward(cfg0, p, x, eps, 0.3).pred)
