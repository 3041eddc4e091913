#!/usr/bin/env python
"""bench.py -- training samples/sec of the Distributed-IB hot path on the BASELINE.json workload.

Workload C0 (SURVEY.md section 8d): 16 scalar features, positional encoding (4 frequencies), per-feature encoders
[128,128] relu -> (mu, logvar) with E=32, integration MLP [256,256] -> 1 logit, BCE-from-logits + beta*sum KL,
Keras-Adam lr 3e-4, batch 65 536, synthetic N(0,1) inputs with labels from a fixed nonlinear teacher, random-init
(glorot-uniform) weights.  One "step" = forward + backward + gradient all-reduce (N>1) + Adam on one batch.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path (weak scaling: 65 536 rows/GPU)
    python bench.py --impl reference ...                           # the reference graph's CPU twin (host cores)
    python bench.py --config C2|C3|C4|C4p                          # the other SURVEY 8d shapes (profiles/)
    python bench.py --dump-outputs DIR ...                         # also write the last timed step's results to DIR

Prints ONE JSON line (rank 0).
  value / ms_per_step : device-resident throughput.  Exactly K steps between two CUDA events (barrier + synchronize on
                        both sides) after W untimed warm-up steps; ms_per_step is their mean (max over ranks).
  strong              : the same metric with the 65 536-row GLOBAL batch split over the N GPUs (SURVEY 8d "the metric as
                        stated"), measured in the same run (for N = 1 it equals value).
  e2e                 : the same step through the public API (model.train_on_batch) from pinned HOST buffers with the
                        H2D copy and the D2H read of the metrics inside the timed region (another K steps).
  roofline            : the dominant kernel's algorithmic FLOP/s (SURVEY 8d MAC counts) over its CUDA-event duration,
                        against the measured dense bf16/fp16 tensor peak -- burst or sustained chosen from the SM clock
                        sampled during the timed region.
See DESIGN.md section "Measurement".

--dump-outputs DIR writes, after the device-resident timed steps and before anything else trains the model further, what
a caller of the timed path (model.train_on_batch) receives from its last step: the metrics (loss.npy, accuracy.npy,
kl_per_feature.npy, float64) and the updated weights (weights.npy, the flat float32 parameter vector).  Inputs, initial
weights and noise are seeded, so the same arguments give the same inputs on every run and two builds can be compared
output for output.
"""
import argparse
import glob
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "training samples/sec (16-feat synthetic, batch 65k) at 1/2/4/8 B200; HBM GB/s"
LR = 3e-4
N_DISTINCT_BATCHES = 16          # SURVEY.md 8d: N = 16 * 65536 rows, 16 steps per epoch

# SURVEY.md 8d shapes.  C0 is the metric's configuration; the others are recorded under profiles/.
CONFIGS = {
    "C0": dict(fdims=[1] * 16, enc=[128, 128], integ=[256, 256], out=1, E=32, pe=True, nfreq=5, act="relu", loss="bce",
               batch=65536, note="16 scalar features x batch 65536, PE(4 freq) -> enc[128,128] -> E=32 -> int[256,256] -> 1, "
                                 "BCE-from-logits + beta*KL, Keras-Adam"),
    "C2": dict(fdims=[1] * 12, enc=[128, 128], integ=[256, 256], out=1, E=32, pe=True, nfreq=5, act="relu", loss="mse",
               batch=4096, note="12 scalar features (bikeshare-shaped) x batch 4096, MSE"),
    "C3": dict(fdims=[2, 1, 2, 1], enc=[128, 128], integ=[256, 256], out=6, E=32, pe=True, nfreq=5, act="relu", loss="mse",
               batch=128, note="simulate_pendulum.py regression: d=[2,1,2,1], out 6, MSE, batch 128 (train.py:34)"),
    "C4": dict(fdims=[1] * 100, enc=[128, 128], integ=[256, 256, 256], out=1, E=32, pe=False, nfreq=1, act="tanh", loss="bce",
               batch=256, note="nb-radial reference shape: 100 shell features, tanh, no PE, int [256]*3, batch 256"),
    "C4p": dict(fdims=[1] * 50, enc=[128, 128], integ=[256, 256, 256], out=1, E=32, pe=False, nfreq=1, act="tanh", loss="bce",
                batch=8192, note="BASELINE config 4: 50 shell features, batch 8192 (bf16 storage, 8 GPUs in BASELINE)"),
}
DTYPE_LABEL = {"fp32": "f32", "tf32": "tf32 (fp32 storage, kind::tf32 operands, fp32 accumulate)",
               "fp16": "fp16 operands + fp32 accumulate (tcgen05 kind::f16; PE/exp/KL/loss/Adam fp32)",
               "bf16": "bf16 operands + fp32 accumulate (tcgen05 kind::f16; PE/exp/KL/loss/Adam fp32)"}


def synth_batches(cfg, rank, nb, batch, pinned):
    """x ~ N(0,1) float32, y from a fixed nonlinear teacher with interactions (SURVEY.md 8d)."""
    import torch
    rng = np.random.default_rng(1000 + rank)
    D = sum(cfg["fdims"])
    xs, ys = [], []
    for _ in range(nb):
        x = rng.standard_normal((batch, D), dtype=np.float32)
        t = x[:, 0] * x[:, 1] + np.sin(2 * x[:, 2]) + 0.5 * x[:, 3] + 0.1 * rng.standard_normal(batch, dtype=np.float32)
        if cfg["loss"] == "bce":
            y = np.repeat((t > 0).astype(np.float32)[:, None], cfg["out"], 1)
        else:
            y = np.stack([np.roll(t, k) for k in range(cfg["out"])], 1).astype(np.float32)
        xt, yt = torch.from_numpy(x), torch.from_numpy(np.ascontiguousarray(y))
        if pinned:
            xt, yt = xt.pin_memory(), yt.pin_memory()
        xs.append(xt)
        ys.append(yt)
    return xs, ys


def algorithmic_macs(batch, cfg=None):
    """MACs per launch group (SURVEY.md 8d 'ALGORITHMIC work per sample'); defaults to the C0 shapes."""
    cfg = cfg or CONFIGS["C0"]
    F, E = len(cfg["fdims"]), cfg["E"]
    macs = {}
    enc_h = cfg["enc"]
    for j in range(len(enc_h) + 1):
        n = enc_h[j] if j < len(enc_h) else 2 * E
        ksum = sum(d * (cfg["nfreq"] if cfg["pe"] else 1) for d in cfg["fdims"]) if j == 0 else F * enc_h[j - 1]
        for kind in ("fwd", "wgrad"):
            macs[f"enc_{kind}_l{j}"] = ksum * n * batch
        if j >= 1:
            macs[f"enc_dgrad_l{j}"] = ksum * n * batch
    widths = [F * E] + list(cfg["integ"]) + [cfg["out"]]
    for j in range(len(widths) - 1):
        for kind in ("fwd", "wgrad", "dgrad"):
            macs[f"int_{kind}_l{j}"] = widths[j] * widths[j + 1] * batch
    fwd = sum(v for k, v in macs.items() if "_fwd_" in k)
    train = sum(macs.values())
    # fused per-feature encoder kernels: algorithmic work = the layers they replace (the backward kernel's on-chip
    # recomputation of the forward is overhead, not algorithmic work)
    macs["enc_fused_fwd"] = sum(v for k, v in macs.items() if k.startswith("enc_fwd_"))
    macs["enc_fused_bwd"] = sum(v for k, v in macs.items() if k.startswith("enc_dgrad_") or k.startswith("enc_wgrad_"))
    nl = len(widths) - 1
    for j in range(nl - 1):               # 16-bit integration path groups (the output layer lives in the fused head)
        macs[f"int16_fwd_l{j}"] = macs[f"int_fwd_l{j}"]
        macs[f"int16_wgrad_l{j}"] = macs[f"int_wgrad_l{j}"]
        macs[f"int16_dgrad_l{j}"] = macs[f"int_dgrad_l{j}"]
    for j in range(nl - 2):               # two layers' weight gradients per launch (dib_int16_wgrad_pair)
        macs[f"int16_wgrad_pair_l{j}"] = macs[f"int_wgrad_l{j}"] + macs[f"int_wgrad_l{j + 1}"]
    if nl >= 3:                           # single-output models: last two hidden layers + head in one kernel (dib_int16_fwd2_kernel)
        macs["int16_fwd2_head"] = macs[f"int_fwd_l{nl - 3}"] + macs[f"int_fwd_l{nl - 2}"] + macs[f"int_fwd_l{nl - 1}"]
    return macs, fwd, train


NCU_KERNEL_OF_GROUP = {"enc_fused_bwd": "dib_enc_fused_bwd", "enc_fused_fwd": "dib_enc_fused_fwd"}


def ncu_dram_traffic(group):
    """(bytes, source): dram__bytes_read.sum + dram__bytes_write.sum per launch of `group`'s kernel from the NEWEST
    committed `ncu --set full` summary under profiles/ -- a STATIC figure from that capture, not measured in this run
    (ncu cannot run inside a timed bench); (None, None) if no capture names the kernel."""
    kern = NCU_KERNEL_OF_GROUP.get(group)
    if not kern:
        return None, None
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full.txt")), reverse=True)
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for path in files:
        total, inside = 0.0, False
        for line in open(path):
            if line.startswith("## "):
                if inside:
                    break
                inside = kern in line
            elif inside and ("dram__bytes_read.sum" in line or "dram__bytes_write.sum" in line):
                parts = line.split()
                total += float(parts[1]) * scale.get(parts[2], 1.0)
        if total:
            return total, "static: " + os.path.relpath(path, ROOT)
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md 'clocks' line)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.path = f"/tmp/dib_clocks_{os.getpid()}.csv"
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(index)],
                stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        rows = []
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                try:
                    rows.append((float(parts[0]), float(parts[1]), float(parts[2]), parts[3:7]))
                except ValueError:
                    pass
        os.unlink(self.path)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        pw = np.array([r[2] for r in rows])
        load = [r for r in rows if r[2] >= 0.5 * pw.max()] or rows
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in load for i in range(4) if r[3][i].lower().startswith("active")})
        return {"sm_mhz": float(np.median([r[0] for r in load])), "sm_max_mhz": float(rows[0][1]),
                "power_w_max": float(pw.max()), "samples": len(rows), "samples_under_load": len(load), "reasons": reasons}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "sustained_sm_mhz": (d.get("clocks_under_load") or {}).get("sm_mhz_median"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "sustained_sm_mhz": 1300.0,
            "source": "fallback"}


def pick_peak(peaks, clocks):
    """Burst peak when the SM clock stayed near its maximum during the timed region (this step draws ~250 W of the
    1000 W cap, so it does), the sustained figure when the clock sagged toward the power-capped GEMM's."""
    sm, mx = (clocks or {}).get("sm_mhz"), (clocks or {}).get("sm_max_mhz")
    sus = peaks.get("sustained_sm_mhz") or 1400.0
    if sm and mx and sm < 0.5 * (mx + sus):
        return peaks["tflops_sustained"], "sustained"
    return peaks["tflops_burst"], "burst"


def oracle_cfg(cfg):
    from oracle import dib_oracle as O
    return O.DIBConfig(cfg["fdims"], cfg["enc"], cfg["integ"], cfg["out"], use_positional_encoding=cfg["pe"],
                       number_positional_encoding_frequencies=cfg["nfreq"], activation_fn=cfg["act"],
                       feature_embedding_dimension=cfg["E"])


_BEST_THREADS = {}


def cpu_twin_rate(cfg, sample_rows, steps, warmup, threads=None):
    """samples/s of the reference graph's eager CPU twin.  `threads=None`: use the thread count that is fastest on
    this host AT THE SAMPLE SIZE BEING TIMED (a 128-thread pool on a shared box can be far slower than 16 threads for
    these small per-feature ops, so "all the threads it can use" is found by a probe at the real size)."""
    from oracle import dib_oracle as O
    from oracle.torch_twin import time_train_steps
    ocfg = oracle_cfg(cfg)
    loss = O.LOSS_BCE_LOGITS if cfg["loss"] == "bce" else O.LOSS_MSE
    rng = np.random.default_rng(0)
    x = rng.standard_normal((sample_rows, sum(cfg["fdims"])), dtype=np.float32)
    y = np.repeat((x[:, 0] * x[:, 1] > 0).astype(np.float32)[:, None], cfg["out"], 1)
    if threads is None:
        key = (tuple(cfg["fdims"]), sample_rows)
        if key not in _BEST_THREADS:
            ncpu = os.cpu_count() or 1
            cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
            best = None
            for c in cands:
                med, _, _ = time_train_steps(ocfg, loss, x, y, LR, 1, 1, threads=c)
                if best is None or med < best[0]:
                    best = (med, c)
            _BEST_THREADS[key] = best[1]
        threads = _BEST_THREADS[key]
    med, total, threads = time_train_steps(ocfg, loss, x, y, LR, steps, warmup, threads=threads)
    return sample_rows / med, med, threads


def run_reference(args, rank, cfg):
    """The reference graph's CPU twin (oracle/torch_twin.py; TensorFlow is not installable here) on the host cores."""
    if rank != 0:
        return
    batch = cfg["batch"]
    # bounded sample: probe a small batch, then size the per-step sample so that the whole run (warm-up + timed steps)
    # takes about 90 s of CPU time, at most one full batch and at most ~1.5 s per step
    _, probe, _ = cpu_twin_rate(cfg, min(4096, batch), 1, 1, threads=8)
    per_step = min(1.5, 90.0 / max(args.steps + args.warmup, 1))
    rows = int(min(batch, max(min(1024, batch), 2 ** int(np.log2(max(per_step / probe, 0.25) * min(4096, batch))))))
    rate, med, threads = cpu_twin_rate(cfg, rows, args.steps, args.warmup)
    sample = (f"{rows} of {batch} rows per step, {args.steps} timed steps, PyTorch-CPU eager twin of models.py "
              f"(TF unavailable), threads picked at this size; host nproc {os.cpu_count()}")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": med * 1e3 * batch / rows,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args.config, args.gpus, "cpu"),
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": threads, "host_nproc": os.cpu_count(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(cfg, name, n_gpus=None, precision=None, per_gpu=None):
    if isinstance(cfg, int):            # short form workload_config(n_gpus, precision, per_gpu) -> C0
        cfg, name, n_gpus, precision, per_gpu = CONFIGS["C0"], "C0", cfg, name, n_gpus
    per_gpu = cfg["batch"] if per_gpu is None else per_gpu
    return {"workload": f"{name}: {cfg['note']}; {per_gpu} rows/GPU",
            "global_batch": per_gpu * n_gpus, "per_gpu_batch": per_gpu, "parallelism": f"dp{n_gpus}", "precision": precision,
            "l2": "no explicit flush: every step streams its intermediates through the 126 MB L2 (16-bit path ~0.33 GB of "
                  "activations/gradients/partials per 65536 rows), evicting the 16 rotating input batches between their uses"}


def dump_outputs(out_dir, metrics, weights, F):
    """What train_on_batch hands its caller for one step: the metrics dict and the model's updated weights."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": np.array([metrics["loss"]], dtype=np.float64),
              "accuracy": np.array([metrics["accuracy"]], dtype=np.float64),
              "kl_per_feature": np.array([metrics[f"KL{i}"] for i in range(F)], dtype=np.float64),
              "weights": np.asarray(weights, dtype=np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


JSON_OUT = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries print there too (NCCL's version banner, torchrun notices), so
    keep a private handle on the real stdout for the result and point fd 1 at stderr for everything else."""
    global JSON_OUT
    if JSON_OUT is None:
        sys.stdout.flush()
        JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    JSON_OUT.write(json.dumps(line) + "\n")
    JSON_OUT.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DIB_PRECISION", "fp16"), choices=["fp16", "bf16", "tf32", "fp32"],
                    help="fp16 = fused tcgen05 kernels on fp16 operands (default, the headline); bf16 likewise; "
                         "tf32 = kind::tf32 GEMMs on fp32 storage; fp32 = exact CUDA-core parity path")
    ap.add_argument("--config", default="C0", choices=sorted(CONFIGS))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's metrics and updated weights to DIR/<name>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="what `value` reports -- weak (default): the config batch per GPU; strong: the "
                         "global batch split over the GPUs.  The other one is always reported under its own key.")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
        run_reference(args, rank, cfg)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import dib_b200
    from dib_b200 import _lib

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    BATCH = cfg["batch"]
    lib = _lib.load()
    F = len(cfg["fdims"])

    model = dib_b200.DistributedIBNet(cfg["fdims"], cfg["enc"], cfg["integ"], cfg["out"], use_positional_encoding=cfg["pe"],
                                      number_positional_encoding_frequencies=cfg["nfreq"], activation_fn=cfg["act"],
                                      feature_embedding_dimension=cfg["E"], seed=1, precision=args.precision)
    loss = dib_b200.losses.BinaryCrossentropy(from_logits=True) if cfg["loss"] == "bce" else "mse"
    model.compile(optimizer=dib_b200.Adam(LR), loss=loss, metrics=["accuracy"])
    model.beta.assign(1e-3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(step_fn, steps):
        """Exactly `steps` steps between CUDA events with barrier + synchronize on both sides.
        Returns (ms per step [max over ranks], total s)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for i in range(steps):
            step_fn(i)
        ev1.record()
        barrier()
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        return ms / steps, ms * 1e-3

    def measure(PB, with_e2e, dump_dir=None):
        """Device-resident and (optionally) end-to-end throughput at PB rows per GPU."""
        xs_h, ys_h = synth_batches(cfg, rank, N_DISTINCT_BATCHES, PB, pinned=True)
        xs_d = [x.cuda(non_blocking=True) for x in xs_h]
        ys_d = [y.cuda(non_blocking=True) for y in ys_h]
        torch.cuda.synchronize()

        last_result = [None]

        def device_step(i):       # public API, device-resident batch, no host read inside the step
            last_result[0] = model.train_on_batch(xs_d[i % N_DISTINCT_BATCHES], ys_d[i % N_DISTINCT_BATCHES], sync=False)

        for i in range(args.warmup):
            device_step(i)
        barrier()
        count = lambda: int(lib.dib_launch_count()) + int(getattr(model, "_replayed_launches", 0))   # eager + graph-replayed kernels
        launches0 = count()
        ms_step, total_s = timed(device_step, args.steps)
        launches = count() - launches0
        res = {"ms_per_step": ms_step, "timed_region_s": total_s, "launches": launches,
               "launches_per_step": launches / args.steps, "xs_d": xs_d, "ys_d": ys_d}
        res["value"] = PB * world / (res["ms_per_step"] * 1e-3)
        if dump_dir is not None:
            dump_outputs(dump_dir, last_result[0].get(), model.get_flat_weights(), F)
        if with_e2e:
            for i in range(3):
                model.train_on_batch(xs_h[i], ys_h[i], sync=False).get()
            pend = []
            last = {}

            def e2e_step(i):
                # every step: pinned host batch -> H2D (copy stream) -> step -> async D2H of the metrics into pinned memory
                pend.append(model.train_on_batch(xs_h[i % N_DISTINCT_BATCHES], ys_h[i % N_DISTINCT_BATCHES], sync=False))
                if len(pend) > 4:
                    last.update(pend.pop(0).get())       # the host reads every step's result, a few steps behind the device

            e2e_ms, tot = timed(e2e_step, args.steps)
            for p in pend:
                last.update(p.get())
            res["e2e"] = {"value": PB * world / (e2e_ms * 1e-3), "unit": "samples/s", "ms_per_step": e2e_ms,
                          "timed_region_s": tot,
                          "h2d_bytes_per_step": int(xs_h[0].numel() * 4 + ys_h[0].numel() * 4),
                          "d2h_bytes_per_step": int((F + 3) * 4),
                          "api": "DistributedIBNet.train_on_batch(host x, host y, sync=False).get() -> metrics dict "
                                 "(H2D on a copy stream, D2H async)",
                          "last_loss": last.get("loss")}
        return res

    # ---------------- weak (config batch per GPU) and strong (global batch split) measurements
    sampler = ClockSampler(local_rank) if rank == 0 else None      # sampled under load: warm-up + timed regions
    PB_weak = BATCH
    PB_strong = max(BATCH // world, 1)
    primary_PB = PB_weak if args.scaling == "weak" else PB_strong
    prim = measure(primary_PB, with_e2e=True, dump_dir=args.dump_outputs if rank == 0 else None)
    other = None
    if world > 1 and not args.no_strong:
        other = measure(PB_strong if args.scaling == "weak" else PB_weak, with_e2e=False)
    clocks = sampler.stop() if sampler else None
    weak, strong = (prim, other) if args.scaling == "weak" else (other, prim)
    if world == 1:
        weak = strong = prim

    # ---------------- per-launch-group CUDA-event profile of the same steps -> roofline (rank 0)
    roofline = None
    PB = primary_PB
    ms_per_step = prim["ms_per_step"]
    if rank == 0:
        import ctypes
        model._ensure_handle(PB)
        _lib.check(lib.dib_profile_enable(model._handle, 1))
        nprof = min(args.steps, 8)
        for i in range(nprof):
            model._backward(prim["xs_d"][i], prim["ys_d"][i], global_batch=PB * world, sample_offset=rank * PB)
        cap = 8192
        ms = (ctypes.c_float * cap)()
        labels = ctypes.create_string_buffer(1 << 17)
        n = lib.dib_profile_read(model._handle, labels, len(labels), ms, cap)
        lib.dib_profile_enable(model._handle, 0)
        names = labels.value.decode().split("\n")[:n]
        groups = {}
        for nm, t in zip(names, list(ms)[:n]):
            groups.setdefault(nm, []).append(float(t))
        avg = {k: float(np.mean(v)) for k, v in groups.items()}
        macs, fwd_macs, train_macs = algorithmic_macs(PB, cfg)
        keyed = [k for k in avg if k in macs]
        peaks = measured_peaks()
        peak, which = pick_peak(peaks, clocks)
        step_ach = 2 * train_macs / (ms_per_step * 1e-3) / 1e12
        P = model.count_params()
        roofline = {"bound": "tensor", "unit": "TFLOP/s", "peak": peak,
                    "peak_source": f"{peaks['source']} dense bf16/fp16 tensor peak, {which} (SM clock {clocks and clocks.get('sm_mhz')} MHz "
                                   f"during the timed region); operands {args.precision}",
                    "step_achieved_tflops": step_ach, "step_frac": step_ach / peak,
                    "algorithmic_gflop_per_step": 2 * train_macs / 1e9,
                    "hbm_algorithmic_gbs": (4 * (sum(cfg['fdims']) + cfg['out']) * PB + 7 * P * 4) / (ms_per_step * 1e-3) / 1e9,
                    "hbm_peak_gbs": peaks["hbm_gbs"],
                    "group_ms": {k: round(v, 4) for k, v in sorted(avg.items(), key=lambda kv: -kv[1])}}
        if keyed:
            top = max(keyed, key=lambda k: avg[k])
            ach = 2 * macs[top] / (avg[top] * 1e-3) / 1e12
            traffic, tsrc = ncu_dram_traffic(top)
            roofline.update({"kernel": top, "achieved": ach, "frac": ach / peak, "traffic": traffic, "traffic_source": tsrc,
                             "kernel_ms": avg[top], "kernel_share_of_step": avg[top] / sum(avg.values())})
    barrier()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rows = min(16384, BATCH)
        rate, med, threads = cpu_twin_rate(cfg, rows, 3, 1)
        cpu_baseline = {"value": rate, "unit": "samples/s", "cores": threads, "host_nproc": os.cpu_count(), "kind": "port",
                        "sample": f"{rows} of {BATCH} rows per step, 1 warm-up + 3 timed steps of oracle/torch_twin.py "
                                  f"(PyTorch-CPU eager twin of models.py; TensorFlow is not installable here); thread count "
                                  f"probed at this sample size"}

    if rank == 0:
        pack = lambda r, pb: None if r is None else {"value": r["value"], "unit": "samples/s", "ms_per_step": r["ms_per_step"],
                                                     "per_gpu_batch": pb, "global_batch": pb * world,
                                                     "timed_region_s": r["timed_region_s"]}
        line = {
            "metric": METRIC, "value": prim["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": DTYPE_LABEL[args.precision],
            "data": "synthetic", "config": workload_config(cfg, args.config, world, args.precision, PB),
            "timed_region_s": prim["timed_region_s"],
            "timing": f"mean of {args.steps} steps after {args.warmup} warm-up steps (CUDA events, barrier+sync around "
                      f"the timed region, max over ranks)",
            "weak": pack(weak, PB_weak), "strong": pack(strong, PB_strong),
            "clocks": clocks, "e2e": prim.get("e2e"),
            "gpu_launches": prim["launches"], "launches_per_step": prim["launches_per_step"],
            "roofline": roofline, "cpu_baseline": cpu_baseline, "host_nproc": os.cpu_count(),
            "library": os.path.relpath(_lib.library_path(), ROOT), "build": lib.dib_build_info().decode(),
            "kernels": model.kernel_info(PB),
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
