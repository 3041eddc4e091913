"""Generates tests/golden/ref_ctw.npz and ref_ctw_sweeps.npz from the REFERENCE'S OWN native code: chaos/cppctw.cpp
compiled where it lies in a checkout of the reference (oracle/Makefile -> oracle/_ref/libctw_ref.so):
    make -C oracle REF=<reference checkout> && python tests/golden/make_ctw_golden.py
ref_ctw_sweeps.npz holds the reference's entropy for each sequence of the seeded sweeps in tests/test_ctw.py."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import ctw_oracle  # noqa: E402
from tests.test_ctw import fresh_sequences, small_sequences  # noqa: E402


def sequences():
    rng = np.random.default_rng(7)
    out = {"kat_1001": (np.array([1, 0, 0, 1]), 2),                     # chaos/setup.py:26-28 smoke call
           "zeros_1000": (np.zeros(1000, dtype=np.int64), 2),
           "alternating_1000": (np.arange(1000) % 2, 2),
           "single": (np.array([0]), 2)}
    lcg, v = [], 12345                                                   # SURVEY section 4: 20 000 LCG symbols, A = 4
    for _ in range(20000):
        v = (1103515245 * v + 12345) % (1 << 31)
        lcg.append((v >> 16) & 3)
    out["lcg_20000"] = (np.array(lcg), 4)
    x, sym = 0.3, []
    for _ in range(6000):                                                # a chaotic source (logistic map, r = 3.9)
        x = 3.9 * x * (1 - x)
        sym.append(int(x > 0.5))
    out["logistic_6000"] = (np.array(sym), 2)
    out["periodic_7x300"] = (np.tile([0, 1, 1, 2, 0, 2, 1], 300), 3)
    out["blocks_deep"] = (np.concatenate([np.zeros(700), np.ones(700), np.zeros(700)]).astype(np.int64), 2)   # depth > 512
    for n, A in ((17, 2), (300, 3), (2500, 5), (4000, 16)):
        out[f"random_{n}_{A}"] = (rng.integers(0, A, n), A)
    return out


def main():
    assert ctw_oracle.reference_available(), "run `make -C oracle` first"
    rec = {}
    for name, (seq, A) in sequences().items():
        rec[name + "_seq"] = seq.astype(np.int8)
        rec[name + "_A"] = np.int32(A)
        rec[name + "_H"] = np.float64(ctw_oracle.reference_estimate_entropy(seq, A))
        print(f"{name:>20s}  A={A:<3d} n={len(seq):<6d} H={rec[name + '_H']!r}")
    np.savez_compressed(os.path.join(HERE, "ref_ctw.npz"), **rec)
    sweeps = {key: np.array([ctw_oracle.reference_estimate_entropy(seq, A) for seq, A in cases()], dtype=np.float64)
              for key, cases in (("fresh_H", fresh_sequences), ("small_H", small_sequences))}
    np.savez_compressed(os.path.join(HERE, "ref_ctw_sweeps.npz"), **sweeps)
    print({k: len(v) for k, v in sweeps.items()})


if __name__ == "__main__":
    main()
