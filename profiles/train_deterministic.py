#!/usr/bin/env python
"""Deterministic against default training steps on one GPU (the ``bench.py --train`` model, batches and settings), in one process:
    python profiles/train_deterministic.py [--out profiles/train_deterministic.json] [--rounds 5] [--steps 20]

1. Step time, for fp32 and bf16: TrainSteps on identical weight copies, built and warmed up as ``bench.py --train`` builds its
   one (ANet shape, B = 64, dropout 0.2, ``graph=True``), timed alternately with CUDA events, ``--rounds`` rounds of ``--steps``
   graph-replayed steps per mode, the order of the modes rotated every round.  Modes:
     default      the flag off: atomic reductions (what bench.py measures)
     det          ``torch.use_deterministic_algorithms(True)``: the fixed-order kernels, and torch's NaN fill of every
                  ``torch.empty`` (``torch.utils.deterministic.fill_uninitialized_memory``, on by default under the flag)
     det_nofill   the flag on with that fill switched off: the cost of the kernels alone
2. Repeatability: two fresh runs of ``--repeat-steps`` eager steps from the same seed (same weights, dropout and Gumbel draws)
   per precision and mode; the number of gradient elements that differ at each step, and of parameter elements after the last.
The GPU's name, power limit and maximum SM clock are read in the same run and stored with the numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, synth  # noqa: E402
from vmrframe_b200.train import TrainStep  # noqa: E402

MODES = ("default", "det", "det_nofill")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def set_mode(mode):
    torch.use_deterministic_algorithms(mode != "default")
    torch.utils.deterministic.fill_uninitialized_memory = mode != "det_nofill"


def make_step(wt, dev, precision):
    torch.manual_seed(0)
    model = SeqPAN(synth.make_configs(wt, droprate=0.2), synth.make_word_vectors(wt), precision="bf16", sync_timing=False).train().to(dev)
    model.repack = lambda: None            # the inference handle is not used between training steps
    return TrainStep(model, lr=1e-4, num_train_steps=1, precision=precision)


def stats(xs):
    xs = sorted(xs)
    return {"mean": sum(xs) / len(xs), "min": xs[0], "max": xs[-1], "spread_pct": 100.0 * (xs[-1] - xs[0]) / xs[0], "rounds": xs}


def step_times(steps, batches, rounds, n):
    for mode, ts in steps.items():      # bench.py --train's warm-up, in the step's own mode: eager steps, then one capture per shape
        set_mode(mode)
        for i in range(3 + 12):
            ts.step(batches[i % 4], graph=True)
    torch.cuda.synchronize()
    ms = {k: [] for k in steps}
    order = list(steps)
    for r in range(rounds):
        for mode in order[r % len(order):] + order[:r % len(order)]:
            set_mode(mode)
            ts = steps[mode]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                ts.step(batches[i % 4], graph=True)
            e1.record()
            torch.cuda.synchronize()
            ms[mode].append(e0.elapsed_time(e1) / n)
    return ms


def run(wt, dev, batches, precision, nsteps):
    ts = make_step(wt, dev, precision)
    torch.manual_seed(1)
    grads = []
    for i in range(nsteps):
        ts.step(batches[i % 4])
        grads.append(ts.flat.clone())
    return grads, torch.cat([p.detach().reshape(-1) for p in ts.model.parameters()])


def repeatability(wt, dev, batches, precision, nsteps):
    out = {}
    for mode in ("default", "det"):
        set_mode(mode)
        (g1, p1), (g2, p2) = run(wt, dev, batches, precision, nsteps), run(wt, dev, batches, precision, nsteps)
        out[mode] = {"gradient_elements": g1[0].numel(), "parameter_elements": p1.numel(),
                     "differing_gradient_elements_per_step": [int((a != b).sum()) for a, b in zip(g1, g2)],
                     "differing_parameter_elements_after_last_step": int((p1 != p2).sum())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "train_deterministic.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeat-steps", type=int, default=4)
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
    res = {"gpu": info, "workload": f"anet B={Bt} L={wt.vlen} Tmax={wt.tmax}, dropout 0.2, TrainStep.step(graph=True), one GPU",
           "timing": f"{args.rounds} rounds x {args.steps} graph-replayed steps per mode, rotating in one process, CUDA events",
           "repeatability": f"two fresh runs of {args.repeat_steps} eager steps from the same seed per precision and mode"}
    try:
        for precision in ("fp32", "bf16"):
            steps = {mode: make_step(wt, dev, precision) for mode in MODES}
            ms = step_times(steps, batches, args.rounds, args.steps)
            del steps
            torch.cuda.empty_cache()
            r = {"step_ms": {k: stats(v) for k, v in ms.items()}}
            r["cost_det_over_default"] = r["step_ms"]["det"]["mean"] / r["step_ms"]["default"]["mean"]
            r["cost_det_nofill_over_default"] = r["step_ms"]["det_nofill"]["mean"] / r["step_ms"]["default"]["mean"]
            r["repeatability"] = repeatability(wt, dev, batches, precision, args.repeat_steps)
            res[precision] = r
    finally:
        set_mode("default")
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
