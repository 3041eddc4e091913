"""GPU (B200): the streaming tensor-core InfoNCE head (dib_infonce_head_tc) against
 (a) the float64 oracle (oracle.dib_oracle.infonce_loss_and_grads) at small n,
 (b) the exact GPU head (dib_infonce_head, S in scratch) at n = 8209,
 (c) a blockwise float64 reference (row blocks of S on the GPU) at n = 40000 and 65536, where the exact head refuses.
Bounds: loss relative error <= 1e-5, gradient rel_err (max abs error over max abs value) <= 1e-4; measured on one B200 at
most 1.3e-6 and 1.8e-5 (n = 65536, cosine).  The logit-range test keeps 5e-4 (measured 2.6e-4 for cosine at T = 0.003,
where a cosine error of 1e-7 is 3e-5 nats).  The products use bf16 hi + lo split operands (~2^-17 relative) with fp32
accumulation; the positive pairs s_ii are exact fp32."""
import numpy as np
import pytest
import torch

from oracle import dib_oracle as O

pytestmark = pytest.mark.gpu

KINDS = ["l2sq", "l2", "cosine"]
LOSS_TOL, GRAD_TOL = 1e-5, 1e-4


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def head_tc(a, b, kind, T):
    from dib_b200 import utils
    return utils._infonce_head_tc(a, b, utils.SIMILARITY_TYPES[kind], T)


def temperature(kind, d):
    return 0.3 if kind == "cosine" else 2.0 * np.sqrt(d)      # as in test_scaled_similarity_and_infonce_head


def check(loss, da, db, l_ref, da_ref, db_ref, what, grad_tol=GRAD_TOL):
    loss, da, db = float(loss.item()), da.cpu().numpy(), db.cpu().numpy()
    assert np.isfinite(loss) and np.isfinite(da).all() and np.isfinite(db).all(), what
    assert abs(loss - l_ref) <= LOSS_TOL * max(abs(l_ref), 1.0), (what, loss, l_ref)
    scale_a, scale_b = max(np.abs(da_ref).max(), 1e-6), max(np.abs(db_ref).max(), 1e-6)
    assert np.abs(da - da_ref).max() / scale_a <= grad_tol, (what, np.abs(da - da_ref).max() / scale_a)
    assert np.abs(db - db_ref).max() / scale_b <= grad_tol, (what, np.abs(db - db_ref).max() / scale_b)


def blockwise_reference(a, b, kind, T, block=2048):
    """float64 InfoNCE loss and gradients from row blocks of S (never the whole n x n matrix at once)."""
    a, b = a.double(), b.double()
    n = a.shape[0]
    na, nb = a.norm(dim=1), b.norm(dim=1)
    an, bn = a / na[:, None], b / nb[:, None]
    a2, b2 = (a * a).sum(1), (b * b).sum(1)

    def rows(i0, i1):
        if kind == "cosine":
            g = an[i0:i1] @ bn.T
            return g / T, g
        d2 = (a2[i0:i1, None] + b2[None, :] - 2.0 * (a[i0:i1] @ b.T)).clamp_min(0.0)
        if kind == "l2sq":
            return -d2 / T, None
        q = torch.sqrt(d2 + 1e-9)
        return -q / T, q

    r = torch.empty(n, dtype=torch.float64, device=a.device)
    c = torch.full((n,), -float("inf"), dtype=torch.float64, device=a.device)
    diag = torch.empty(n, dtype=torch.float64, device=a.device)
    for i0 in range(0, n, block):
        i1 = min(n, i0 + block)
        s, _ = rows(i0, i1)
        r[i0:i1] = torch.logsumexp(s, 1)
        c = torch.logaddexp(c, torch.logsumexp(s, 0))
        diag[i0:i1] = s[torch.arange(i1 - i0), torch.arange(i0, i1)]
    loss = (r + c - 2.0 * diag).mean().item()
    da, db = torch.zeros_like(a), torch.zeros_like(b)
    for i0 in range(0, n, block):
        i1 = min(n, i0 + block)
        s, extra = rows(i0, i1)
        p = torch.exp(s - r[i0:i1, None]) + torch.exp(s - c[None, :])
        p[torch.arange(i1 - i0), torch.arange(i0, i1)] -= 2.0
        p /= n
        if kind == "cosine":
            pc = p * extra
            da[i0:i1] = (p @ bn - an[i0:i1] * pc.sum(1)[:, None]) / (T * na[i0:i1, None])
            db += (p.T @ an[i0:i1] - bn * pc.sum(0)[:, None]) / (T * nb[:, None])
        else:
            w, f = (p, 2.0 / T) if kind == "l2sq" else (p / extra, 1.0 / T)
            da[i0:i1] = f * (w @ b - a[i0:i1] * w.sum(1)[:, None])
            db += f * (w.T @ a[i0:i1] - b * w.sum(0)[:, None])
    return loss, da.cpu().numpy(), db.cpu().numpy()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 2, 5, 129, 300])
@pytest.mark.parametrize("d", [3, 64, 100, 130, 200])     # 1, 1, 2, 3 and 4 panels of 64 columns
def test_head_matches_float64_oracle(kind, n, d):
    rng = np.random.default_rng(1000 * n + d)
    a, b = rng.standard_normal((n, d)).astype(np.float32), rng.standard_normal((n, d)).astype(np.float32)
    T = temperature(kind, d)
    loss, da, db = head_tc(a, b, kind, T)
    l_ref, da_ref, db_ref, _ = O.infonce_loss_and_grads(a, b, kind, T)
    check(loss, da, db, l_ref, da_ref, db_ref, (kind, n, d))


@pytest.mark.parametrize("kind", KINDS)
def test_blockwise_reference_matches_oracle(kind):
    """The large-n reference below is itself checked against the oracle."""
    rng = np.random.default_rng(5)
    a, b = rng.standard_normal((300, 24)), rng.standard_normal((300, 24))
    T = temperature(kind, 24)
    loss, da, db = blockwise_reference(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda(), kind, T, block=128)
    l_ref, da_ref, db_ref, _ = O.infonce_loss_and_grads(a, b, kind, T)
    assert abs(loss - l_ref) < 1e-12 * abs(l_ref) + 1e-12
    assert rel_err(da, da_ref) < 1e-10 and rel_err(db, db_ref) < 1e-10


def correlated_batch(n, d, seed, noise=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randn(n, d, device="cuda", generator=g)
    b = a + noise * torch.randn(n, d, device="cuda", generator=g)
    return a, b


@pytest.mark.parametrize("kind", KINDS)
def test_head_matches_exact_gpu_head_at_8209(kind):
    from dib_b200 import utils
    a, b = correlated_batch(8209, 64, 11)
    T = temperature(kind, 64)
    l_ex, da_ex, db_ex = utils.infonce_loss_and_grads(a, b, kind, T)
    loss, da, db = head_tc(a, b, kind, T)
    check(loss, da, db, l_ex.item(), da_ex.cpu().numpy(), db_ex.cpu().numpy(), kind)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [40000, 65536])
def test_head_beyond_the_exact_head(kind, n):
    """utils.infonce_loss_and_grads takes the tensor-core head where the exact head refuses (n > 32768)."""
    from dib_b200 import utils
    a, b = correlated_batch(n, 64, n)
    T = temperature(kind, 64)
    loss, da, db = utils.infonce_loss_and_grads(a, b, kind, T)
    l_ref, da_ref, db_ref = blockwise_reference(a, b, kind, T)
    check(loss, da, db, l_ref, da_ref, db_ref, (kind, n))


def test_gram_free_kinds_still_refuse_beyond_32768():
    from dib_b200 import DibError, utils
    a, b = correlated_batch(32769, 8, 3)
    with pytest.raises(DibError):
        utils.infonce_loss_and_grads(a, b, "l1", 1.0)


@pytest.mark.parametrize("kind", KINDS)
def test_logits_spanning_hundreds_inside_one_tile(kind):
    """A few pairs moved far away and a small temperature: logits inside one 64 x 128 tile span > 300, and no row or
    column may lose its sum to underflow."""
    n, d = 1000, 64
    a, b = correlated_batch(n, d, 21, noise=0.3)
    moved = torch.tensor([0, 3, 64, 700], device="cuda")
    shift = 10.0 * torch.ones(d, device="cuda")
    a[moved] += shift
    b[moved] += shift
    T = {"l2sq": 0.5, "l2": 0.2, "cosine": 0.003}[kind]
    l_ref, da_ref, db_ref = blockwise_reference(a, b, kind, T)
    from dib_b200 import utils
    s_tile = utils.get_scaled_similarity(a[:128], b[:64], kind, T)
    assert (s_tile.max() - s_tile.min()).item() > 300
    loss, da, db = head_tc(a, b, kind, T)
    check(loss, da, db, l_ref, da_ref, db_ref, kind, grad_tol=5e-4)


@pytest.mark.parametrize("kind", KINDS)
def test_near_duplicate_pairs_off_the_diagonal(kind):
    """Rows of e2 that nearly repeat rows of e1 at other indices (duplicate samples on the Y side).  For l2 the weight
    dS / |a_i - b_j| is large there, and the Gram expansion cannot resolve |a_i - b_j|: those pairs are recomputed from the
    fp32 rows, like the diagonal."""
    n, d = 700, 64
    a, b = correlated_batch(n, d, 31)
    g = torch.Generator(device="cuda").manual_seed(32)
    src, dst = torch.tensor([5, 64, 300, 301, 699], device="cuda"), torch.tensor([9, 63, 301, 0, 128], device="cuda")
    for scale in (1e-3, 1e-5, 0.0):
        b2 = b.clone()
        b2[dst] = a[src] + scale * torch.randn(len(src), d, device="cuda", generator=g)
        T = temperature(kind, d)
        l_ref, da_ref, db_ref = blockwise_reference(a, b2, kind, T)
        loss, da, db = head_tc(a, b2, kind, T)
        check(loss, da, db, l_ref, da_ref, db_ref, (kind, scale))


@pytest.mark.parametrize("kind", KINDS)
def test_identical_calls_are_bit_identical(kind):
    a, b = correlated_batch(5000, 64, 9)
    T = temperature(kind, 64)
    first = [t.cpu().numpy().tobytes() for t in head_tc(a, b, kind, T)]
    second = [t.cpu().numpy().tobytes() for t in head_tc(a, b, kind, T)]
    assert first == second


def test_loss_only_call_matches_full_call():
    from dib_b200 import utils
    a, b = correlated_batch(777, 64, 4)
    full = head_tc(a, b, "l2", 8.0)
    loss, d1, d2 = utils._infonce_head_tc(a, b, utils.SIMILARITY_TYPES["l2"], 8.0, want_grads=False)
    assert d1 is None and d2 is None and loss.item() == full[0].item()
