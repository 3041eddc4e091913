"""CPU: the float64 InfoNCE training oracle (tests/infonce_oracle.py) -- its step gradients against central finite
differences for every similarity, and the fit mechanics' step count."""
import numpy as np
import pytest

from oracle import dib_oracle as O
from tests import infonce_oracle as NO

CFG = O.DIBConfig([2, 1, 2, 1], [7, 5], [6], 4, feature_embedding_dimension=3, number_positional_encoding_frequencies=3,
                  activation_fn="tanh")
OCFG = NO.OutputEncoderConfig(2, [5, 4])


def _setup(kind, seed=0):
    rng = np.random.default_rng(seed)
    p = O.glorot_uniform_params(CFG, rng, dtype=np.float64) + rng.standard_normal(CFG.param_count()) * 0.05
    q = NO.output_encoder_glorot(CFG, OCFG, rng, dtype=np.float64)
    q = q + rng.standard_normal(q.size) * 0.05
    n = 6
    x = rng.standard_normal((n, 6))
    y = rng.standard_normal((n, 2))
    eps = rng.standard_normal((n, 4, 3))
    return p, q, x, y, eps


def _total(p, q, x, y, eps, beta, kind, T):
    loss, fr = NO.infonce_forward(CFG, OCFG, p, q, x, y, eps, beta, kind, T)
    return loss + beta * float(np.sum(fr.kl_per_feature))


@pytest.mark.parametrize("kind", O.SIMILARITY_TYPES)
def test_step_gradients_match_finite_differences(kind):
    p, q, x, y, eps = _setup(kind)
    beta, T = 0.3, 0.7
    gp, gq, loss, fr = NO.infonce_train_grads(CFG, OCFG, p, q, x, y, eps, beta, kind, T)
    assert np.isfinite(loss) and loss > 0
    h = 1e-6
    for g, vec, is_q in ((gp, p, False), (gq, q, True)):
        fd = np.empty_like(vec)
        for i in range(vec.size):
            a, b = vec.copy(), vec.copy()
            a[i] += h
            b[i] -= h
            fa = _total(p, a, x, y, eps, beta, kind, T) if is_q else _total(a, q, x, y, eps, beta, kind, T)
            fb = _total(p, b, x, y, eps, beta, kind, T) if is_q else _total(b, q, x, y, eps, beta, kind, T)
            fd[i] = (fa - fb) / (2 * h)
        # l1 / linf are piecewise linear: random inputs keep |differences| and the argmax away from ties
        assert np.abs(g - fd).max() <= 1e-6 * max(np.abs(fd).max(), 1.0), (kind, is_q)


def test_fit_runs_the_epoch_boundaries_of_the_repeated_stream():
    rng = np.random.default_rng(1)
    cfg = O.DIBConfig([1, 1], [4], [4], 3, feature_embedding_dimension=2, number_positional_encoding_frequencies=2)
    ocfg = NO.OutputEncoderConfig(1, [3])
    p = O.glorot_uniform_params(cfg, rng, dtype=np.float64)
    q = NO.output_encoder_glorot(cfg, ocfg, rng, dtype=np.float64)
    N, B, E = 50, 8, 3
    x, y = rng.standard_normal((N, 2)), rng.standard_normal((N, 1))
    r = NO.epoch_boundaries(N, B, E)
    assert r == [0, 6, 12, 19]                          # np.round(6.25 e): 6.25, 12.5 -> 12 (half to even), 18.75
    eps_fn = lambda s, ids: np.zeros((len(ids), 2, 2))
    _, _, hist, steps = NO.fit_infonce(cfg, ocfg, p, q, x, y, kind="l2", T=1.0, epochs=E, batch_size=B, lr=1e-3,
                                       eps_fn=eps_fn, validation_data=(x[:20], y[:20]))
    assert steps == r[E]
    assert set(hist) == {"loss", "beta", "KL0", "KL1", "val_loss", "val_beta", "val_KL0", "val_KL1"}
    assert all(len(v) == E for v in hist.values())


def test_oracle_matches_the_reference_infonce_golden(golden_dir):
    """tests/golden/ref_infonce_step.npz: train.py's own output encoder and eval_batch_infonce on the numpy stand-in."""
    import os
    cases = NO.load_infonce_golden(os.path.join(golden_dir, "ref_infonce_step.npz"))
    assert len(cases) == 4
    for name, (cfg, ocfg, z) in cases.items():
        kind, T, beta = str(z["kind"]), float(z["temperature"]), float(z["beta"])
        e2 = NO.output_encoder_forward(cfg, ocfg, z["q"], z["y"])
        loss, fr = NO.infonce_forward(cfg, ocfg, z["p"], z["q"], z["x"], z["y"], z["eps"], beta, kind, T)
        np.testing.assert_allclose(fr.pred, z["e1"], rtol=1e-12, atol=1e-14, err_msg=name)
        np.testing.assert_allclose(e2, z["e2"], rtol=1e-12, atol=1e-14, err_msg=name)
        np.testing.assert_allclose(loss, float(z["loss_infonce"]), rtol=1e-12, err_msg=name)
        # kl_loss / model.beta of train.py:220 is model.losses / beta = [sum_i KL_i]
        np.testing.assert_allclose(fr.kl_per_feature.sum(), z["kl"].sum(), rtol=1e-12, err_msg=name)
