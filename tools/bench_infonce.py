"""Time the InfoNCE heads on one GPU and write the result as JSON.

    python tools/bench_infonce.py --out DIR

Records the GPU name, power limit and maximum SM clock (nvidia-smi query), then times, with CUDA events over --iters
launches after --warmup launches, the full head (loss and both gradients) at d = 64 for 'l2' and 'cosine':
  * the streaming tensor-core head (dib_infonce_head_tc) at n in {4096, 16384, 32768, 65536};
  * the exact head (dib_infonce_head, S in scratch) at n in {4096, 16384, 32768} (it refuses larger n).
For the tensor-core head it reports the exponentials per second and the MMA FLOP/s the kernels execute (counted from the
shapes below), and the two lower bounds those counts give: MUFU (16 ex2 per clock per SM at the maximum SM clock) and
MMA (the data sheet's 2250 TFLOP/s dense BF16), naming the larger of the two (`larger_count_bound`).  That is a floor
from counts, not a measured bottleneck: the measured rates say whether the kernel is anywhere near it.
Inputs are 3 x n x 64 floats, far below L2: the timings are of an L2-resident working set, as in a training step.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dib_b200 import _lib, utils  # noqa: E402

SMS = 148
MUFU_PER_CLK_PER_SM = 16
BF16_DENSE_FLOPS = 2.25e15


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def tc_counts(n, d):
    """Work the tensor-core head issues: 4 sweeps (lse and grad, both sides) of split-operand Gram products (3 MMAs each)
    plus 2 split-operand weight products; 1 exponential per element per side in pass 1, 2 in pass 2."""
    n_pad, dp = -(-n // 128) * 128, -(-d // 64) * 64
    n_oth = -(-n // 64) * 64
    gram = 4 * 3 * 2.0 * n_pad * n_oth * dp
    wy = 2 * 3 * 2.0 * n_pad * n_oth * dp
    return {"mma_flop": gram + wy, "exps": 6.0 * n * n}


def time_call(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_infonce needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    lib = _lib.load()
    info = gpu_info()
    stream = lambda: torch.cuda.current_stream().cuda_stream   # noqa: E731
    d = 64
    rows = []
    for kind in ("l2", "cosine"):
        k = utils.SIMILARITY_TYPES[kind]
        T = 0.3 if kind == "cosine" else 16.0
        for n in (4096, 16384, 32768, 65536):
            g = torch.Generator(device="cuda").manual_seed(n)
            e1 = torch.randn(n, d, device="cuda", generator=g)
            e2 = e1 + 0.5 * torch.randn(n, d, device="cuda", generator=g)
            loss, d1, d2 = torch.empty(1, device="cuda"), torch.empty_like(e1), torch.empty_like(e2)
            tc_scratch = torch.empty(lib.dib_infonce_head_tc_scratch_bytes(n, d), dtype=torch.uint8, device="cuda")
            tc = lambda: _lib.check(lib.dib_infonce_head_tc(   # noqa: E731
                k, _lib.ptr(e1), _lib.ptr(e2), n, d, T, _lib.ptr(tc_scratch), _lib.ptr(loss), _lib.ptr(d1), _lib.ptr(d2),
                ctypes.c_void_p(stream())))
            ms_tc = time_call(tc, args.warmup, args.iters)
            c = tc_counts(n, d)
            t_mufu = c["exps"] / (MUFU_PER_CLK_PER_SM * SMS * info["max_sm_clock_mhz"] * 1e6) * 1e3
            t_mma = c["mma_flop"] / BF16_DENSE_FLOPS * 1e3
            row = {"kind": kind, "n": n, "d": d, "tc_ms": ms_tc, "tc_scratch_bytes": tc_scratch.numel(),
                   "tc_exps_per_s": c["exps"] / (ms_tc * 1e-3), "tc_mma_flop_per_s": c["mma_flop"] / (ms_tc * 1e-3),
                   "mufu_bound_ms": t_mufu, "mma_bound_ms": t_mma, "larger_count_bound": "MUFU" if t_mufu >= t_mma else "MMA",
                   "tc_share_of_larger_bound": max(t_mufu, t_mma) / ms_tc}
            del tc_scratch
            if n <= 32768:
                ex_scratch = torch.empty(n * n + 4 * n, device="cuda")
                ex = lambda: _lib.check(lib.dib_infonce_head(   # noqa: E731
                    k, _lib.ptr(e1), _lib.ptr(e2), n, d, T, _lib.ptr(ex_scratch), _lib.ptr(loss), _lib.ptr(d1),
                    _lib.ptr(d2), ctypes.c_void_p(stream())))
                row["exact_ms"] = time_call(ex, args.warmup, args.iters)
                row["speedup"] = row["exact_ms"] / ms_tc
                del ex_scratch
            rows.append(row)
            print(json.dumps(row), flush=True)
    out = {"gpu": info, "warmup": args.warmup, "iters": args.iters, "heads": rows,
           "full_step": "not measured: the output encoder and InfoNCE loss in compile/fit are not built yet"}
    with open(os.path.join(args.out, "bench_infonce.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
