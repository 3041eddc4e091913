"""Next row f4: the CTW entropy-rate estimator.  Host code (no GPU): the C-ABI functions are compared BIT-EXACTLY with
 (a) goldens produced by the reference's own chaos/cppctw.cpp (tests/golden/ref_ctw.npz, make_ctw_golden.py),
 (b) the reference build's results on seeded sweeps of fresh sequences (tests/golden/ref_ctw_sweeps.npz, same script),
 (c) the Python restatement oracle/ctw_oracle.py on small sequences."""
import os

import numpy as np
import pytest

from oracle import ctw_oracle


@pytest.fixture(scope="module")
def ctw():
    from dib_b200 import ctw as mod
    return mod


def _cases(golden_dir):
    z = np.load(os.path.join(golden_dir, "ref_ctw.npz"))
    names = sorted(k[:-4] for k in z.files if k.endswith("_seq"))
    return [(n, z[n + "_seq"], int(z[n + "_A"]), float(z[n + "_H"])) for n in names]


def test_oracle_restatement_matches_reference_goldens(golden_dir):
    for name, seq, A, H in _cases(golden_dir):
        if len(seq) <= 2500:
            assert ctw_oracle.estimate_entropy(seq, A) == H, name
    assert ctw_oracle.estimate_entropy([1, 0, 0, 1], 2) == 1.0232774019241333          # SURVEY section 4 KAT


def test_library_matches_reference_goldens_bit_exactly(ctw, golden_dir):
    cases = _cases(golden_dir)
    for name, seq, A, H in cases:
        assert ctw.estimate_entropy(seq, A) == H, name
    for A in sorted({c[2] for c in cases}):
        group = [c for c in cases if c[2] == A]
        got = ctw.estimate_entropy_batch([c[1] for c in group], A, num_threads=3)
        np.testing.assert_array_equal(got, [c[3] for c in group])


def fresh_sequences():
    """(sequence, alphabet size) pairs of the fresh-sequence comparison; make_ctw_golden.py stores the reference's results."""
    rng = np.random.default_rng(123)
    out = []
    for n, A in ((1, 3), (33, 2), (1000, 3), (6000, 4), (3000, 27)):
        seq = rng.integers(0, A, n)
        seq[n // 3: n // 3 + min(n // 4, 900)] = seq[0]                       # a long run: deep tails, depth > 512
        out.append((seq, A))
    return out


def small_sequences():
    """(sequence, alphabet size) pairs of the small-sequence sweep: short sequences over small alphabets, incl. long runs
    and periodic pieces that exercise the lazy tail extension; make_ctw_golden.py stores the reference's results."""
    rng = np.random.default_rng(2024)
    out = []
    for trial in range(300):
        A = int(rng.integers(1, 6))
        n = int(rng.integers(1, 90))
        kind = trial % 3
        if kind == 0:
            seq = rng.integers(0, A, n)
        elif kind == 1:                                                       # runs
            seq = np.repeat(rng.integers(0, A, max(n // 7, 1)), 7)[:n]
        else:                                                                 # periodic with a defect
            seq = np.tile(rng.integers(0, A, int(rng.integers(1, 5))), n)[:n]
            seq[int(rng.integers(0, n))] = int(rng.integers(0, A))
        out.append((seq, A))
    return out


def _sweep_goldens(golden_dir, key, cases):
    want = np.load(os.path.join(golden_dir, "ref_ctw_sweeps.npz"))[key]
    assert len(want) == len(cases)
    return want


def test_library_matches_reference_build_on_fresh_sequences(ctw, golden_dir):
    assert np.isnan(ctw.estimate_entropy([], 2))
    cases = fresh_sequences()
    for (seq, A), H in zip(cases, _sweep_goldens(golden_dir, "fresh_H", cases)):
        assert ctw.estimate_entropy(seq, A) == H, (len(seq), A)


def test_edge_cases_and_errors(ctw):
    from dib_b200._lib import DibError
    assert np.isnan(ctw.estimate_entropy([], 2))
    assert ctw.estimate_entropy([0], 2) == 1.0
    with pytest.raises(DibError):
        ctw.estimate_entropy([0, 2], 2)                                        # symbol outside the alphabet
    with pytest.raises(ValueError):
        ctw.estimate_entropy([[0, 1]], 2)
    assert ctw.estimate_entropy_batch([], 2).shape == (0,)
    h = ctw.estimate_entropy_batch([[0, 1, 1], [], [1] * 50], 2, num_threads=8)
    assert h[0] == ctw.estimate_entropy([0, 1, 1], 2) and np.isnan(h[1]) and h[2] == ctw.estimate_entropy([1] * 50, 2)


def test_entropy_rate_properties(ctw):
    rng = np.random.default_rng(5)
    fair = ctw.estimate_entropy(rng.integers(0, 2, 50000), 2)
    biased = ctw.estimate_entropy((rng.random(50000) < 0.1).astype(np.int8), 2)
    h_biased = -(0.1 * np.log2(0.1) + 0.9 * np.log2(0.9))
    assert abs(fair - 1.0) < 0.01 and abs(biased - h_biased) < 0.02
    markov = [0]
    for _ in range(50000):                                                    # sticky two-state chain, H = h(0.05)
        markov.append(markov[-1] ^ int(rng.random() < 0.05))
    assert abs(ctw.estimate_entropy(markov, 2) - (-(0.05 * np.log2(0.05) + 0.95 * np.log2(0.95)))) < 0.02


def test_random_small_sequences_against_python_restatement(ctw, golden_dir):
    """hypothesis-style sweep (seeded): library == Python restatement == the reference, bit for bit."""
    cases = small_sequences()
    for trial, ((seq, A), H) in enumerate(zip(cases, _sweep_goldens(golden_dir, "small_H", cases))):
        got = ctw.estimate_entropy(seq, A)
        assert got == ctw_oracle.estimate_entropy(seq, A), (trial, A, seq.tolist())
        assert got == H, (trial, A, seq.tolist())
