#!/usr/bin/env python
"""One eager training step by each of the two autograd routes on one GPU, alternating in one process:
    python profiles/autograd_forward.py [--out profiles/autograd_forward.json] [--rounds 5] [--steps 10]

* ``model(...)``: ``SeqPAN.forward`` in ``train()`` (the tape recorded as one autograd node), ``engine.lossfun_loc`` +
  ``engine.lossfun_match`` in torch on the outputs, ``loss.backward()`` (the tape's adjoints), ``torch.optim.AdamW``.
* ``train_engine_SeqPAN``: forward, both losses and the backward on the tape in one call, ``loss.backward()`` (hands out the
  finished gradients), the same optimizer.

The ``bench.py --train`` shape: ANet-shaped batches of 64 pairs, dropout 0.2.  Each route owns a model on identical weights and
its own optimizer; ``--rounds`` rounds of ``--steps`` steps per route, the order swapped every round, timed with CUDA events.
Both routes are eager (no CUDA graph) and host-bound: the tape issues ~1200 small launches from Python per step.  This is a
report, not a gate.  The GPU's name and power limit are read in the same run and stored with the numbers."""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, synth, train_engine_SeqPAN  # noqa: E402
from vmrframe_b200.engine import lossfun_loc, lossfun_match  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def make_model(wt, dev):
    torch.manual_seed(0)
    return SeqPAN(synth.make_configs(wt, droprate=0.2), synth.make_word_vectors(wt), sync_timing=False).train().to(dev)


def step_module(model, opt, bd, cfg):
    out = model(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
    loss = lossfun_loc(out["slogits"], out["elogits"], bd["label1ds"][:, 0, :], bd["label1ds"][:, 1, :], bd["vmasks"]) + \
        lossfun_match(out["match_score"], out["label_embs"], bd["NER_labels"], bd["vmasks"])
    opt.zero_grad(set_to_none=True)
    loss.backward()
    opt.step()
    return loss


def step_engine(model, opt, bd, cfg):
    loss, _ = train_engine_SeqPAN(model, bd, cfg, "train")
    opt.zero_grad(set_to_none=True)
    loss.backward()
    opt.step()
    return loss


def stats(xs):
    s = sorted(xs)
    return {"mean": sum(s) / len(s), "min": s[0], "max": s[-1], "spread_pct": 100.0 * (s[-1] - s[0]) / s[0], "rounds": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "autograd_forward.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    w = synth.WORKLOADS["anet"]
    wt = synth.Workload(w.name, w.config_id, args.batch, w.vlen, w.tmax, w.clen, w.vdim, w.num_words, w.num_chars, w.tlen, 1)
    batches = [{k: v.to(dev) for k, v in synth.add_train_labels(synth.make_batch(wt, i)).items()} for i in range(4)]
    cfg = SimpleNamespace(device=dev)
    routes = {}
    for name, fn in (("model_call_torch_losses", step_module), ("train_engine_SeqPAN", step_engine)):
        m = make_model(wt, dev)
        routes[name] = (fn, m, torch.optim.AdamW(m.parameters(), lr=1e-4))
    for fn, m, opt in routes.values():        # warm-up: every input shape once, lazy state (optimizer moments) created
        for i in range(4):
            fn(m, opt, batches[i], cfg)
    torch.cuda.synchronize()
    ms, losses = {k: [] for k in routes}, {}
    order = list(routes)
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            fn, m, opt = routes[name]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                loss = fn(m, opt, batches[i % 4], cfg)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / args.steps)
            losses[name] = float(loss.detach())
    res = {"gpu": info, "workload": f"anet B={args.batch} L={wt.vlen} Tmax={wt.tmax}, dropout 0.2, fp32, eager steps, one GPU",
           "timing": f"{args.rounds} rounds x {args.steps} steps per route, alternating in one process, CUDA events",
           "step_ms": {k: stats(v) for k, v in ms.items()},
           "last_loss": losses}
    res["ratio_model_call_over_engine"] = res["step_ms"]["model_call_torch_losses"]["mean"] / res["step_ms"]["train_engine_SeqPAN"]["mean"]
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
