"""GPU (B200): compile(loss=InfoNCE) training -- the one-call step (dib_infonce_train_step) against the float64 oracle
(tests/infonce_oracle.py) and against the composition dib_forward -> head -> dib_train_step, fit against the oracle's
fit, CUDA-graph replay, determinism, learning, and the refusals of compile."""
import numpy as np
import pytest
import torch

from oracle import dib_oracle as O
from oracle import philox
from tests import infonce_oracle as NO

pytestmark = pytest.mark.gpu

KINDS = ["l2sq", "l2", "l1", "linf", "cosine"]
CFG = O.DIBConfig([2, 1, 2, 1], [32, 32], [32], 16, feature_embedding_dimension=8)
OCFG = NO.OutputEncoderConfig(6, [16, 12])
# fused-kernel-eligible shape for the 16-bit modes (C0-like features, E = 32), D = 64
CFG_TC = O.DIBConfig([1] * 4, [128, 128], [128], 64, feature_embedding_dimension=32)
OCFG_TC = NO.OutputEncoderConfig(1, [128, 128])


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def build(cfg, ocfg, kind="l2", T=1.0, precision="fp32", seed=0, lr=1e-3):
    import dib_b200
    m = dib_b200.DistributedIBNet(
        cfg.feature_dimensionalities, cfg.feature_encoder_architecture, cfg.integration_network_architecture,
        cfg.output_dimensionality, use_positional_encoding=cfg.use_positional_encoding,
        number_positional_encoding_frequencies=cfg.number_positional_encoding_frequencies,
        activation_fn=cfg.activation_fn, feature_embedding_dimension=cfg.feature_embedding_dimension,
        precision=precision, seed=seed)
    m.compile(optimizer=dib_b200.Adam(lr), loss=dib_b200.losses.InfoNCE(kind, T, ocfg.architecture))
    m.build_output_encoder(ocfg.input_dimensionality)
    return m


def inputs(cfg, ocfg, n, seed):
    rng = np.random.default_rng(seed)
    p = O.glorot_uniform_params(cfg, rng)
    q = NO.output_encoder_glorot(cfg, ocfg, rng)
    x = rng.standard_normal((n, sum(cfg.feature_dimensionalities))).astype(np.float32)
    y = rng.standard_normal((n, ocfg.input_dimensionality)).astype(np.float32)
    eps = rng.standard_normal((n, cfg.number_features, cfg.feature_embedding_dimension)).astype(np.float32)
    return p, q, x, y, eps


def gram_head(e1, e2, kind, T):
    """float64 InfoNCE head for 'l2' / 'cosine' in matrix form (O(n^2) memory; the oracle's is O(n^2 d))."""
    a, b = np.asarray(e1, np.float64), np.asarray(e2, np.float64)
    n = a.shape[0]
    if kind == "l2":
        dist = np.sqrt(np.maximum((a * a).sum(1)[:, None] + (b * b).sum(1)[None, :] - 2 * a @ b.T, 0) + 1e-9)
        S = -dist / T
    else:
        na, nb = np.linalg.norm(a, axis=1), np.linalg.norm(b, axis=1)
        ah, bh = a / na[:, None], b / nb[:, None]
        c = ah @ bh.T
        S = c / T
    row, col = O._logsumexp(S, 1), O._logsumexp(S, 0)
    loss = float((row - np.diag(S)).mean() + (col - np.diag(S)).mean())
    dS = (np.exp(S - row[:, None]) + np.exp(S - col[None, :]) - 2 * np.eye(n)) / n
    if kind == "l2":
        W = dS / dist / T
        da = -(W.sum(1)[:, None] * a - W @ b)
        db = W.T @ a - W.sum(0)[:, None] * b
    else:
        da = (dS @ bh - (dS * c).sum(1)[:, None] * ah) / na[:, None] / T
        db = (dS.T @ ah - (dS * c).sum(0)[:, None] * bh) / nb[:, None] / T
    return loss, da, db, S


def oracle_step(cfg, ocfg, p, q, x, y, eps, beta, kind, T, gram=False):
    if not gram:
        return NO.infonce_train_grads(cfg, ocfg, p, q, x, y, eps, beta, kind, T)
    e1 = O.forward(cfg, p, x, eps, beta).pred
    e2, acts = NO.output_encoder_forward(cfg, ocfg, q, y, keep=True)
    loss, d1, d2, _ = gram_head(e1, e2, kind, T)
    gp, fr = O.train_grads(cfg, p, x, d1, eps, beta, "external")
    return gp, NO.output_encoder_backward(cfg, ocfg, q, acts, d2), loss, fr


def step(m, p, q, x, y, eps, beta):
    m.set_flat_weights(p)
    m.output_encoder.set_flat_weights(q)
    m.beta.assign(beta)
    g, st = m.compute_gradients(x, y, eps=eps)
    return g.cpu().numpy(), st.cpu().numpy()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [5, 129, 300])
def test_fp32_step_matches_oracle(kind, n):
    m = build(CFG, OCFG, kind, T=0.5)
    p, q, x, y, eps = inputs(CFG, OCFG, n, seed=n)
    g, st = step(m, p, q, x, y, eps, 0.05)
    gp, gq, loss, fr = NO.infonce_train_grads(CFG, OCFG, p, q, x, y, eps, 0.05, kind, 0.5)
    P, F = len(p), CFG.number_features
    assert g.size == P + len(q)
    assert rel_err(g[:P], gp) < 1e-4, rel_err(g[:P], gp)
    assert rel_err(g[P:], gq) < 1e-4, rel_err(g[P:], gq)
    np.testing.assert_allclose(st[F], n * loss, rtol=2e-5)
    np.testing.assert_allclose(st[:F] / n, fr.kl_per_feature, rtol=2e-5)
    assert st[F + 1] == 0 and st[F + 2] == n
    # the output encoder alone, and the model's e1 through the plain forward
    e2 = m.output_encoder(y)
    assert rel_err(e2, NO.output_encoder_forward(CFG, OCFG, q, y)) < 2e-5


def test_fp32_matches_the_reference_golden(golden_dir):
    """tests/golden/ref_infonce_step.npz (train.py's own output encoder and eval_batch_infonce): e1, e2, loss_infonce and
    the KL sum of dib_forward / dib_output_encoder_forward / dib_infonce_forward."""
    import os
    for name, (cfg, ocfg, z) in NO.load_infonce_golden(os.path.join(golden_dir, "ref_infonce_step.npz")).items():
        kind, T, n = str(z["kind"]), float(z["temperature"]), z["x"].shape[0]
        m = build(cfg, ocfg, kind, T=T)
        m.set_flat_weights(z["p"])
        m.output_encoder.set_flat_weights(z["q"])
        m.beta.assign(float(z["beta"]))
        e1 = m(z["x"], eps=z["eps"])
        assert rel_err(e1, z["e1"]) < 2e-5, name
        assert rel_err(m.output_encoder(z["y"]), z["e2"]) < 2e-5, name
        with torch.cuda.device(m.device):
            st = m._infonce_call(m._to_device(z["x"], 6), m._to_device(z["y"], ocfg.input_dimensionality), 0,
                                 eps=m._to_device(z["eps"]), train=False).cpu().numpy()
        F = cfg.number_features
        np.testing.assert_allclose(st[F] / n, float(z["loss_infonce"]), rtol=2e-5, err_msg=name)
        np.testing.assert_allclose(st[:F].sum() / n, z["kl"].sum(), rtol=2e-5, err_msg=name)


def test_fp32_step_with_padded_embedding_rows():
    """D = 3: e1 / e2 rows are padded to 4 floats in the workspace; the heads get unpadded copies (all five kinds)."""
    cfg = O.DIBConfig([2, 1, 2, 1], [16], [12], 3, feature_embedding_dimension=4)
    ocfg = NO.OutputEncoderConfig(2, [8])
    for kind in KINDS:
        m = build(cfg, ocfg, kind, T=0.7)
        p, q, x, y, eps = inputs(cfg, ocfg, 77, seed=13)
        g, st = step(m, p, q, x, y, eps, 0.05)
        gp, gq, loss, _ = NO.infonce_train_grads(cfg, ocfg, p, q, x, y, eps, 0.05, kind, 0.7)
        P, F = len(p), cfg.number_features
        assert rel_err(g[:P], gp) < 1e-4, (kind, rel_err(g[:P], gp))
        assert rel_err(g[P:], gq) < 1e-4, (kind, rel_err(g[P:], gq))
        np.testing.assert_allclose(st[F], 77 * loss, rtol=2e-5, err_msg=kind)


# End to end, the InfoNCE gradient amplifies the 10-bit (7-bit for bf16) operand rounding of e1 / e2: the softmax over n
# columns turns a relative error of e1 into errors of every dS entry.  The bounds are per mode; the observed values are
# printed.  test_tensor_core_step_decomposed isolates the parts: each matches at the bound of its own kernels.
@pytest.mark.parametrize("precision,tol", [("tf32", 5e-2), ("fp16", 5e-2), ("bf16", 8e-2)])
@pytest.mark.parametrize("kind", ["l2", "cosine"])
def test_tensor_core_step_matches_oracle(precision, tol, kind):
    n = 4160
    m = build(CFG_TC, OCFG_TC, kind, T=0.5, precision=precision)
    p, q, x, y, eps = inputs(CFG_TC, OCFG_TC, n, seed=7)
    g, st = step(m, p, q, x, y, eps, 0.01)
    gp, gq, loss, fr = oracle_step(CFG_TC, OCFG_TC, p, q, x, y, eps, 0.01, kind, 0.5, gram=True)
    P, F = len(p), CFG_TC.number_features
    ep, eq, el = rel_err(g[:P], gp), rel_err(g[P:], gq), abs(st[F] / n - loss) / loss
    print(f"{precision} {kind} n={n}: step vs float64 oracle: model grads {ep:.3g}, encoder grads {eq:.3g}, loss {el:.3g}")
    assert ep < tol and eq < tol and el < tol
    info = m.kernel_info(n)
    assert "output_encoder=" in info and "tcgen05" in info.split("output_encoder=")[1], info


@pytest.mark.parametrize("precision,tol,model_tol", [("tf32", 5e-3, 5e-2), ("fp16", 5e-3, 5e-2), ("bf16", 4e-2, 8e-2)])
@pytest.mark.parametrize("kind", ["l2", "cosine"])
def test_tensor_core_step_decomposed(precision, tol, model_tol, kind):
    """Where the end-to-end difference of the tensor-core step comes from.  (b) The head on the GPU's own e1 / e2 against
    float64: its 1e-4 bound (observed 1.0-1.7e-5).  (a) The output-encoder backward given the head's d e2: the external-loss
    bounds of the mode (observed 0.8-4.9e-3).  The model backward given the head's d e1 carries the whole end-to-end
    difference (observed 1.2e-2 l2, 3.0-3.7e-2 cosine / bf16): that part is the existing external-loss step
    (dib_train_step), which the one-call step reproduces bit for bit (test_large_batch_step...)."""
    from dib_b200 import utils
    n = 4160
    m = build(CFG_TC, OCFG_TC, kind, T=0.5, precision=precision)
    p, q, x, y, eps = inputs(CFG_TC, OCFG_TC, n, seed=7)
    g, st = step(m, p, q, x, y, eps, 0.01)
    e1 = m(torch.from_numpy(x).cuda(), eps=eps, step=0)                 # the forward the step runs (bit-identical)
    e2 = m.output_encoder(torch.from_numpy(y).cuda())
    loss, d1, d2 = utils._infonce_head_tc(e1, e2, utils._similarity_kind(kind), 0.5)
    l64, d1_64, d2_64, _ = gram_head(e1.cpu().numpy(), e2.cpu().numpy(), kind, 0.5)
    d1, d2 = d1.cpu().numpy(), d2.cpu().numpy()
    eh = max(rel_err(d1, d1_64), rel_err(d2, d2_64))
    assert eh < 1e-4 and abs(float(loss) - l64) < 1e-5 * l64, eh
    gp, _ = O.train_grads(CFG_TC, p, x, d1, eps, 0.01, "external")
    _, acts = NO.output_encoder_forward(CFG_TC, OCFG_TC, q, y, keep=True)
    gq = NO.output_encoder_backward(CFG_TC, OCFG_TC, q, acts, d2)
    P = len(p)
    ep, eq = rel_err(g[:P], gp), rel_err(g[P:], gq)
    print(f"{precision} {kind} n={n}: head {eh:.3g}; backward from the head's d e1 / d e2: model {ep:.3g}, encoder {eq:.3g}")
    assert eq < tol and ep < model_tol


def _composition(m, kind, p, q, x, y, eps, beta, precision):
    """dib_forward -> the selected head -> dib_train_step of an external-loss model with the same weights."""
    import dib_b200
    from dib_b200 import utils
    cfg = CFG if precision == "fp32" and x.shape[1] == 6 else CFG_TC
    ext = dib_b200.DistributedIBNet(
        cfg.feature_dimensionalities, cfg.feature_encoder_architecture, cfg.integration_network_architecture,
        cfg.output_dimensionality, feature_embedding_dimension=cfg.feature_embedding_dimension, precision=precision)
    ext.compile(optimizer="adam", loss="external")
    ext.set_flat_weights(p)
    ext.beta.assign(beta)
    e1 = ext(torch.from_numpy(x).cuda(), eps=eps, step=0)
    e2 = m.output_encoder(torch.from_numpy(y).cuda())
    loss, d1, d2 = utils._infonce_head_tc(e1, e2, utils._similarity_kind(kind), 0.5)
    g, st = ext.compute_gradients(x, d1, eps=eps)
    return float(loss), g.cpu().numpy(), st.cpu().numpy(), d2.cpu().numpy()


@pytest.mark.parametrize("kind", ["l2", "cosine"])
def test_one_call_step_equals_the_composition_fp32(kind):
    n = 300
    m = build(CFG, OCFG, kind, T=0.5)
    p, q, x, y, eps = inputs(CFG, OCFG, n, seed=3)
    g, st = step(m, p, q, x, y, eps, 0.05)
    loss, gc, stc, d2 = _composition(m, kind, p, q, x, y, eps, 0.05, "fp32")
    P, F = len(p), CFG.number_features
    err = rel_err(g[:P], gc)
    # the output-encoder half: float64 reverse mode of the encoder from the head's d e2 (fp32 step vs float64: 1e-5)
    _, acts = NO.output_encoder_forward(CFG, OCFG, q, y, keep=True)
    eq = rel_err(g[P:], NO.output_encoder_backward(CFG, OCFG, q, acts, d2))
    print(f"fp32 {kind}: one-call step vs composition, model grads {err:.3g}, encoder grads vs float64 backward {eq:.3g}")
    assert err < 1e-6
    assert eq < 1e-5
    np.testing.assert_allclose(st[F] / n, loss, rtol=1e-6)
    np.testing.assert_allclose(st[:F], stc[:F], rtol=1e-6)


@pytest.mark.parametrize("n", [40000, 65536])
@pytest.mark.parametrize("kind", ["l2", "cosine"])
def test_large_batch_step_runs_with_linear_scratch(kind, n):
    m = build(CFG_TC, OCFG_TC, kind, T=0.5, precision="fp16")
    p, q, x, y, eps = inputs(CFG_TC, OCFG_TC, n, seed=11)
    g, st = step(m, p, q, x, y, eps, 0.01)
    scratch = sum(t.numel() for t in m._nce_scratch.values())
    assert scratch < 64 * n * CFG_TC.output_dimensionality * 4, scratch           # O(n d), not n^2
    loss, gc, _, _ = _composition(m, kind, p, q, x, y, eps, 0.01, "fp16")
    P, F = len(p), CFG_TC.number_features
    assert np.isfinite(g).all()
    err = rel_err(g[:P], gc)
    print(f"fp16 {kind} n={n}: one-call step vs composition, relative max-norm difference {err:.3g}")
    assert err < 1e-6
    np.testing.assert_allclose(st[F] / n, loss, rtol=1e-6)


def test_l1_above_32768_rows_is_refused():
    import dib_b200
    m = build(CFG_TC, OCFG_TC, "l1", precision="fp16")
    p, q, x, y, eps = inputs(CFG_TC, OCFG_TC, 40000, seed=1)
    with pytest.raises(dib_b200.DibError, match="32768"):
        step(m, p, q, x, y, eps, 0.01)


def _fit_pair(precision, shuffle=True):
    import dib_b200
    N, B, Nv, E, lr = 1000, 128, 300, 4, 2e-3
    rng = np.random.default_rng(21)
    x = rng.standard_normal((N + Nv, 6)).astype(np.float32)
    y = np.concatenate([np.sin(x[:, :3]), x[:, 3:] ** 2], 1).astype(np.float32)
    m = build(CFG, OCFG, "l2", T=1.0, precision=precision, seed=5, lr=lr)
    m.noise_seed = 77
    p0, q0 = m.get_flat_weights().copy(), m.output_encoder.get_flat_weights().copy()
    cb = dib_b200.InfoBottleneckAnnealingCallback(1e-3, 1e-1, 1, 2)
    hist = m.fit(x[:N], y[:N], batch_size=B, epochs=E, callbacks=[cb], verbose=False, shuffle=shuffle,
                 validation_data=(x[N:], y[N:])).history
    return m, hist, (x, y, N, B, E, lr, p0, q0)


# fp16: the history series stay within 3e-2; the final weights of 31 Adam steps drift further (3.7e-2 measured)
@pytest.mark.parametrize("precision,tol,wtol", [("fp32", 2e-3, 2e-3), ("fp16", 3e-2, 5e-2)])
def test_fit_matches_oracle_fit(precision, tol, wtol):
    m, hist, (x, y, N, B, E, lr, p0, q0) = _fit_pair(precision)
    r = NO.epoch_boundaries(N, B, E)
    assert m._train_step_count == r[E] == int(m._step_dev.item())
    perms = {k: m.epoch_permutation(k, N).cpu().numpy() for k in range(r[E] * B // N + 2)}
    F, Ef = CFG.number_features, CFG.feature_embedding_dimension
    eps_fn = lambda s, ids: philox.normal_noise(77, s, ids, F, Ef, dtype=np.float64)
    p_ref, q_ref, h_ref, steps = NO.fit_infonce(
        CFG, OCFG, p0, q0, x[:N].astype(np.float64), y[:N].astype(np.float64), kind="l2", T=1.0, epochs=E, batch_size=B,
        lr=lr, eps_fn=eps_fn, perm_fn=lambda k, n: perms[k], beta_fn=lambda e: O.beta_schedule(e, 1e-3, 1e-1, 1, 2),
        validation_data=(x[N:].astype(np.float64), y[N:].astype(np.float64)))
    assert steps == r[E]
    assert set(hist) == set(h_ref)
    for k in h_ref:
        np.testing.assert_allclose(hist[k], h_ref[k], rtol=tol, atol=1e-6, err_msg=k)
    assert rel_err(m.get_flat_weights(), p_ref) < wtol
    assert rel_err(m.output_encoder.get_flat_weights(), q_ref) < wtol


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_graph_replayed_steps_are_bit_identical_to_eager_steps(precision):
    cfg, ocfg = (CFG, OCFG) if precision == "fp32" else (CFG_TC, OCFG_TC)
    rng = np.random.default_rng(2)
    n = 256
    xs = [torch.from_numpy(rng.standard_normal((n, sum(cfg.feature_dimensionalities))).astype(np.float32)).cuda() for _ in range(6)]
    ys = [torch.from_numpy(rng.standard_normal((n, ocfg.input_dimensionality)).astype(np.float32)).cuda() for _ in range(6)]
    out = []
    for graphs in (True, False):
        m = build(cfg, ocfg, "cosine", T=0.3, precision=precision, seed=9)
        m.use_cuda_graph = graphs
        res = [m.train_on_batch(xb, yb) for xb, yb in zip(xs, ys)]
        assert (len(m._graphs) == 1) == graphs
        out.append((m.get_flat_weights(), m.output_encoder.get_flat_weights(), res))
    (pa, qa, ra), (pb, qb, rb) = out
    assert np.array_equal(pa, pb) and np.array_equal(qa, qb)
    assert ra == rb and "accuracy" not in ra[0]


def test_identically_seeded_fits_are_identical():
    a, ha, _ = _fit_pair("fp32")
    b, hb, _ = _fit_pair("fp32")
    assert ha == hb
    assert np.array_equal(a.get_flat_weights(), b.get_flat_weights())
    assert np.array_equal(a.output_encoder.get_flat_weights(), b.output_encoder.get_flat_weights())


def test_infonce_training_learns():
    import dib_b200
    rng = np.random.default_rng(4)
    B = 256
    m = dib_b200.DistributedIBNet([1] * 4, [64, 64], [64], 16, feature_embedding_dimension=8, seed=1)
    m.compile(optimizer=dib_b200.Adam(1e-3), loss=dib_b200.losses.InfoNCE("l2", 1.0, (64, 64)))
    m.beta.assign(1e-4)
    losses = []
    for _ in range(120):
        x = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
        y = np.stack([np.sin(3 * x[:, 0]) + x[:, 1], x[:, 2] * x[:, 3]], 1).astype(np.float32)
        r = m.train_on_batch(x, y)
        losses.append(r["loss"])
    first, last = np.mean(losses[:10]), np.mean(losses[-10:])
    print(f"InfoNCE + IB: first 10 steps {first:.4f}, last 10 steps {last:.4f} (chance 2 ln B = {2 * np.log(B):.4f})")
    assert last <= 0.8 * first


def test_recompile_recaptures_and_keeps_the_layout():
    """A captured step carries similarity and temperature by value: recompiling with other ones re-captures; a non-InfoNCE
    loss on a model with an output encoder is refused."""
    import dib_b200
    m = build(CFG, OCFG, "l2", T=1.0)
    rng = np.random.default_rng(0)
    x = torch.from_numpy(rng.standard_normal((64, 6)).astype(np.float32)).cuda()
    y = torch.from_numpy(rng.standard_normal((64, 6)).astype(np.float32)).cuda()
    for _ in range(4):
        m.train_on_batch(x, y)
    assert len(m._graphs) == 1, m._graph_seen
    m.compile(optimizer=m.optimizer, loss=dib_b200.losses.InfoNCE("cosine", 0.3, OCFG.architecture))
    assert not m._graphs
    ref = build(CFG, OCFG, "cosine", T=0.3)
    ref.set_flat_weights(m.get_flat_weights())
    ref.output_encoder.set_flat_weights(m.output_encoder.get_flat_weights())
    step_now = m._train_step_count
    rs = [m.train_on_batch(x, y)["loss"] for _ in range(4)]        # eager, eager, then a fresh capture
    _, st = ref.compute_gradients(x, y, step=step_now)
    st = st.cpu().numpy()
    F = CFG.number_features
    np.testing.assert_allclose(rs[0], st[F] / 64 + float(ref.beta) * st[:F].sum() / 64, rtol=1e-6)
    assert len(m._graphs) == 1
    with pytest.raises(ValueError, match="output encoder"):
        m.compile(optimizer="adam", loss="mse")


def test_compile_refusals(monkeypatch):
    import dib_b200
    from dib_b200 import parallel
    m = dib_b200.DistributedIBNet([1, 1], [8], [8], 4, feature_embedding_dimension=2)
    with pytest.raises(ValueError, match="metrics"):
        m.compile(loss=dib_b200.losses.InfoNCE(), metrics=["accuracy"])
    with pytest.raises(ValueError, match="Similarity type not implemented"):
        m.compile(loss=dib_b200.losses.InfoNCE("dot"))
    s = dib_b200.DistributedIBNet([1, 1], [8], [8], 4, feature_embedding_dimension=2, output_activation_fn="sigmoid")
    with pytest.raises(ValueError, match="linear output activation"):
        s.compile(loss="infonce")
    w = dib_b200.DistributedIBNet([1, 1], [8], [8], 300, feature_embedding_dimension=2)
    with pytest.raises(ValueError, match="256"):
        w.compile(loss=dib_b200.losses.InfoNCE("cosine"))
    w.compile(loss=dib_b200.losses.InfoNCE("l1"))                  # the exact head has no such limit
    monkeypatch.setattr(parallel, "world_and_rank", lambda group=None: (2, 0))
    with pytest.raises(NotImplementedError):
        m.compile(loss="infonce")
