#!/usr/bin/env python
"""fp32 against bf16 mixed-precision training steps on one GPU (BASELINE.json configs[4] shape), in one process:
    python profiles/train_precision.py [--out profiles/train_bf16_r3.json] [--rounds 5] [--steps 20]

1. Step time: two TrainSteps on identical weight copies, built as ``bench.py --train`` builds its one (ANet shape, B = 64,
   dropout 0.2, ``graph=True``, the same warm-up), one fp32 and one ``precision="bf16"``; timed alternately with CUDA events,
   ``--rounds`` rounds of ``--steps`` steps per mode, the order of the two modes swapped every round.
2. GEMM time per step: ``torch.profiler`` (CUDA activities) over one eager step of each mode, in a separate pass.
3. Kernel rate: one launch of each large GEMM class of the tape (forward linear, dx = g.W, dW = g^T.x with split-K, the
   batched attention adjoint) on both kernels, CUDA events over ``--launches`` launches; FLOP from the shapes.  The operands
   (<= 3.3 MB each) stay L2-resident between launches, as they do inside the tape.
The GPU's name, power limit and maximum SM clock are read in the same run and stored with the numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, synth  # noqa: E402
from vmrframe_b200.train import CudaBackend, TrainStep  # noqa: E402

GEMM_KERNELS = ("t_gemm_kernel", "t_gemm_bf16_kernel")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def make_step(wt, dev, precision):
    torch.manual_seed(0)
    model = SeqPAN(synth.make_configs(wt, droprate=0.2), synth.make_word_vectors(wt), precision="bf16", sync_timing=False).train().to(dev)
    model.repack = lambda: None            # the inference handle is not used between training steps
    return TrainStep(model, lr=1e-4, num_train_steps=1, precision=precision)


def stats(xs):
    xs = sorted(xs)
    return {"mean": sum(xs) / len(xs), "min": xs[0], "max": xs[-1], "spread_pct": 100.0 * (xs[-1] - xs[0]) / xs[0], "rounds": xs}


def step_times(steps, batches, rounds, n):
    for ts in steps.values():           # bench.py --train's warm-up: eager steps, then one capture per input shape
        for i in range(3 + 12):
            ts.step(batches[i % 4], graph=True)
    torch.cuda.synchronize()
    ms = {k: [] for k in steps}
    losses = {}
    order = list(steps)
    for r in range(rounds):
        for mode in (order if r % 2 == 0 else order[::-1]):
            ts = steps[mode]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                loss = ts.step(batches[i % 4], graph=True)[0]
            e1.record()
            torch.cuda.synchronize()
            ms[mode].append(e0.elapsed_time(e1) / n)
            losses[mode] = float(loss)
    return ms, losses


def gemm_profile(ts, batch):
    ts.step(batch)                      # eager warm-up of this shape
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ts.step(batch)
        torch.cuda.synchronize()
    out = {"gpu_ms_per_step": 0.0, "launches": 0}
    for e in prof.key_averages():
        out["gpu_ms_per_step"] += e.device_time_total / 1e3
        out["launches"] += e.count
        for k in GEMM_KERNELS:
            if k + "(" in e.key:
                out[k] = {"ms": out.get(k, {}).get("ms", 0.0) + e.device_time_total / 1e3,
                          "launches": out.get(k, {}).get("launches", 0) + e.count}
    out["gemm_ms_per_step"] = sum(out[k]["ms"] for k in GEMM_KERNELS if k in out)
    return out


def kernel_rates(dev, launches):
    be = CudaBackend(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    x, W, gy = r(6400, 128), r(128, 128), r(6400, 128)
    P, V = r(256, 100, 100), r(256, 100, 32)
    classes = [
        ("forward linear y = x.W^T (A K-major, B K-major)", 6400, 128, 128, 1, lambda: (x, W.t(), 1)),
        ("dx = g.W (A K-major, B N-major)", 6400, 128, 128, 1, lambda: (gy, W, 1)),
        ("dW = g^T.x, split-K 50 (A M-major, B N-major)", 128, 128, 6400, 1, lambda: (gy.t(), x, 50)),
        ("attention dV = P^T.dO, batch 256 (A M-major, B N-major)", 100, 32, 100, 256, lambda: (P.transpose(-1, -2), V, 1)),
    ]
    rows = []
    for name, M, N, K, batch, ops in classes:
        A, B, sk = ops()
        row = {"class": name, "M": M, "N": N, "K": K, "batch": batch, "splitk": sk}
        for mode, mixed in (("fp32", False), ("bf16", True)):
            out = be.gemm(A, B, splitk=sk, mixed=mixed)
            for _ in range(20):
                be.gemm(A, B, out=out, splitk=sk, mixed=mixed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                be.gemm(A, B, out=out, splitk=sk, mixed=mixed)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / launches
            row[mode] = {"us_per_launch": us, "tflops": 2.0 * M * N * K * batch / (us * 1e-6) / 1e12}
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "train_bf16_r3.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    w = synth.WORKLOADS["anet"]
    Bt = args.batch
    wt = synth.Workload(w.name, w.config_id, Bt, w.vlen, w.tmax, w.clen, w.vdim, w.num_words, w.num_chars, w.tlen, 1)
    batches = [{k: v.to(dev) for k, v in synth.add_train_labels(synth.make_batch(wt, i)).items()} for i in range(4)]
    steps = {"fp32": make_step(wt, dev, "fp32"), "bf16": make_step(wt, dev, "bf16")}
    ms, losses = step_times(steps, batches, args.rounds, args.steps)
    res = {"gpu": info, "workload": f"anet B={Bt} L={wt.vlen} Tmax={wt.tmax}, dropout 0.2, TrainStep.step(graph=True), one GPU",
           "timing": f"{args.rounds} rounds x {args.steps} steps per mode, alternating in one process, CUDA events",
           "step_ms": {k: stats(v) for k, v in ms.items()},
           "pairs_per_s": {k: Bt / (sum(v) / len(v) / 1e3) for k, v in ms.items()},
           "last_loss": losses}
    res["speedup_bf16_over_fp32"] = res["step_ms"]["fp32"]["mean"] / res["step_ms"]["bf16"]["mean"]
    res["profile_eager_step"] = {k: gemm_profile(ts, batches[0]) for k, ts in steps.items()}
    res["kernel_rates"] = {"launches": args.launches, "classes": kernel_rates(dev, args.launches)}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
