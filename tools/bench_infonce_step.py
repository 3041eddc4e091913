"""Time the InfoNCE train step (compile(loss=InfoNCE) + train_on_batch) on one GPU and write the result as JSON.

    python tools/bench_infonce_step.py --out DIR [--warmup 5] [--iters 20]

Workload: the C0 features (16 x 1-dim, feature encoders [128, 128], integration network [256, 256], E = 32), D = 64, a
1-dim y with a [128, 128] output encoder, precision fp16.  For n in {4096, 16384, 65536} and 'l2' / 'cosine' it times
graph-replayed train_on_batch steps on device-resident batches with CUDA events (ms/step), and in a separate eager run
records the dib_profile split of one step: model forward, output encoder (forward + backward), head, model backward and
the optimizer.  The GPU name, power limit and maximum SM clock are read in the same run (nvidia-smi query).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import dib_b200  # noqa: E402
from dib_b200 import _lib  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def make_model(kind):
    m = dib_b200.DistributedIBNet([1] * 16, [128, 128], [256, 256], 64, precision="fp16", seed=0)
    m.compile(optimizer=dib_b200.Adam(1e-4), loss=dib_b200.losses.InfoNCE(kind, 1.0, (128, 128)))
    m.build_output_encoder(1)
    m.beta.assign(1e-3)
    return m


def group_of(label):
    if label.startswith("oe_"):
        return "output_encoder"
    if label == "infonce_head":
        return "head"
    if any(label.startswith(p) for p in ("int_wgrad", "int_dgrad", "int_split", "enc_fused_bwd", "enc_split", "enc_wgrad",
                                         "enc_dgrad", "reparam_kl_bwd", "simple_enc_wgrad")):
        return "backward"
    return "model_forward"


def split_of(m, x, y):
    """One eager step under dib_profile: ms per launch group, summed into the five parts."""
    lib = _lib.load()
    m.use_cuda_graph = False
    m.train_on_batch(x, y)                        # lazy setup outside the profile
    torch.cuda.synchronize()
    _lib.check(lib.dib_profile_enable(m._handle, 1))
    with torch.cuda.device(m.device):
        m._backward(x, y, x.shape[0])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        m._adam()
        b.record()
    torch.cuda.synchronize()
    cap = 512
    ms = (ctypes.c_float * cap)()
    labels = ctypes.create_string_buffer(1 << 16)
    k = lib.dib_profile_read(m._handle, labels, len(labels), ms, cap)
    _lib.check(lib.dib_profile_enable(m._handle, 0))
    parts = {"model_forward": 0.0, "output_encoder": 0.0, "head": 0.0, "backward": 0.0}
    rows = []
    for lab, t in zip(labels.value.decode().split("\n")[:k], ms[:k]):
        parts[group_of(lab)] += t
        rows.append([lab, round(t, 5)])
    parts["optimizer"] = a.elapsed_time(b)
    m.use_cuda_graph = True
    return {k: round(v, 5) for k, v in parts.items()}, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "workload": "C0 features (16 x 1-dim, [128,128], [256,256], E=32), D=64, 1-dim y, "
           "output encoder [128,128], fp16, Adam", "timing": "CUDA events over graph-replayed train_on_batch(sync=False) "
           "on device-resident batches", "warmup": args.warmup, "iters": args.iters, "rows": []}
    rng = np.random.default_rng(0)
    for kind in ("l2", "cosine"):
        for n in (4096, 16384, 65536):
            m = make_model(kind)
            x = torch.from_numpy(rng.uniform(-1, 1, (n, 16)).astype(np.float32)).cuda()
            y = torch.from_numpy(np.sin(3 * x[:, :1].cpu().numpy()) + x[:, 1:2].cpu().numpy()).cuda()
            for _ in range(args.warmup):
                m.train_on_batch(x, y, sync=False)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.iters):
                m.train_on_batch(x, y, sync=False)
            b.record()
            torch.cuda.synchronize()
            step_ms = a.elapsed_time(b) / args.iters
            graphed = len(m._graphs) == 1
            split, launches = split_of(m, x, y)
            row = {"kind": kind, "n": n, "ms_per_step": round(step_ms, 4), "graph_replayed": graphed,
                   "eager_split_ms": split, "kernel_info": m.kernel_info(n), "launch_groups_ms": launches}
            print(json.dumps({k: v for k, v in row.items() if k != "launch_groups_ms"}), flush=True)
            res["rows"].append(row)
            del m
            torch.cuda.empty_cache()
    with open(os.path.join(args.out, "bench_infonce_step.json"), "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
