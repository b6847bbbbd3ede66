#!/usr/bin/env python
"""Step time of the two drop-in training routes, eager and replayed from CUDA graphs, against TrainStep on one GPU:
    python profiles/dropin_train_graph.py [--out profiles/dropin_train_graph.json] [--rounds 3] [--steps 10] [--stream 40]

Routes, each on its own model on identical weights with its own ``torch.optim.AdamW`` (``TrainStep`` has its own AdamW):
* ``engine``: ``train_engine_SeqPAN`` -> ``loss.backward()`` -> ``clip_grad_norm_(1.0)`` -> ``optimizer.step()`` (main.py:88-96).
* ``module``: ``model(...)`` -> ``engine.lossfun_loc + lossfun_match`` in torch -> the same backward, clipping and optimizer.
* ``trainstep``: ``TrainStep.step(batch, graph=True)``, the native loop: the floor.
``*_eager`` runs a route with a cache that holds no graph (``max_graphs = 0``); ``*_graph`` is the default.

The ``bench.py --train`` workload: ANet shape, B = 64, dropout 0.2, fp32 and bf16.  Two input streams:
* fixed: one batch, every route warmed up (captured) first; ``--rounds`` rounds of ``--steps`` steps per route, the order
  reversed every other round, timed with CUDA events;
* stream: ``synth.make_batch`` over ``--stream`` successive batch indices (T = the batch maximum of random query lengths, as in
  the reference's collate), the graph routes from a cold cache; reports the replay hit rate and the time per step.
Also the graph-pool size of one captured shape per route (``memory_reserved`` growth over the capture, after ``empty_cache``).
The GPU's name and power limit are read in the same run and stored with the numbers.  A report, not a gate."""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, synth, train, train_engine_SeqPAN  # noqa: E402
from vmrframe_b200.engine import lossfun_loc, lossfun_match  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip()


def make_model(wt, dev, precision):
    torch.manual_seed(0)
    m = SeqPAN(synth.make_configs(wt, droprate=0.2), synth.make_word_vectors(wt), sync_timing=False).train().to(dev)
    m.configs.model.train_precision = precision
    m.repack = lambda: None            # the inference handle is not used between training steps
    return m


class Route:
    def __init__(self, kind, graph, wt, dev, precision, cfg):
        self.kind, self.cfg = kind, cfg
        self.m = make_model(wt, dev, precision)
        self.hits = self.calls = 0
        if kind == "trainstep":
            self.ts = train.TrainStep(self.m, lr=1e-4, num_train_steps=1)
            return
        self.opt = torch.optim.AdamW(self.m.parameters(), lr=1e-4)
        self.ts = train._train_step_of(self.m)
        if not graph:
            self.ts.max_graphs = 0

    def step(self, bd):
        self.calls += 1
        if self.kind == "trainstep":
            return self.ts.step(bd, graph=True)[0]
        if self.kind == "engine":
            captured = [e for e in self.ts._graphs.values() if "graph" in e]
            loss, _ = train_engine_SeqPAN(self.m, bd, self.cfg, "train")
            used = next(reversed(self.ts._graphs.values()))          # the entry of this call: replayed if captured before it
            self.hits += any(e is used for e in captured)
        else:
            out = self.m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
            rec = out["slogits"].grad_fn.rec
            self.hits += isinstance(rec, train._InFlight) and bool(rec.ent.get("bwd"))     # forward and backward both replay
            del rec
            loss = lossfun_loc(out["slogits"], out["elogits"], bd["label1ds"][:, 0, :], bd["label1ds"][:, 1, :], bd["vmasks"]) + \
                lossfun_match(out["match_score"], out["label_embs"], bd["NER_labels"], bd["vmasks"])
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.m.parameters(), 1.0)
        self.opt.step()
        return loss


def stats(xs):
    s = sorted(xs)
    return {"mean": sum(s) / len(s), "min": s[0], "max": s[-1], "rounds": xs}


def reserved():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.memory_reserved()


def run_precision(precision, wt, dev, args):
    cfg = SimpleNamespace(device=dev)
    bd = {k: v.to(dev) for k, v in synth.add_train_labels(synth.make_batch(wt, 0)).items()}
    names = ["engine_eager", "engine_graph", "module_eager", "module_graph", "trainstep_graph"]
    routes = {n: Route(n.split("_")[0], n.endswith("graph"), wt, dev, precision, cfg) for n in names}
    pool_mb = {}
    for n, r in routes.items():             # warm-up: two eager steps, then the capture (measured) and a replay
        for i in range(4):
            before = reserved() if i == 2 else None
            r.step(bd)
            if before is not None:
                pool_mb[n] = (reserved() - before) / 2 ** 20
    torch.cuda.synchronize()
    ms = {n: [] for n in names}
    for rd in range(args.rounds):
        for n in (names if rd % 2 == 0 else names[::-1]):
            r = routes[n]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                r.step(bd)
            e1.record()
            torch.cuda.synchronize()
            ms[n].append(e0.elapsed_time(e1) / args.steps)
    fixed = {n: stats(v) for n, v in ms.items()}
    for n in ("engine_graph", "module_graph"):
        fixed[n]["replayed_steps"] = f"{routes[n].hits} of {routes[n].calls}"
    del routes
    # varying shapes from a cold cache
    stream = [synth.add_train_labels(synth.make_batch(wt, 1 + i)) for i in range(args.stream)]
    shapes = sorted({tuple(b["words_ids"].shape) for b in stream})
    res_stream = {"batches": args.stream, "distinct_shapes": [list(s) for s in shapes]}
    for n in ("engine_graph", "module_graph", "engine_eager", "module_eager"):
        r = Route(n.split("_")[0], n.endswith("graph"), wt, dev, precision, cfg)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for b in stream:
            r.step({k: v.to(dev, non_blocking=True) for k, v in b.items()})
        e1.record()
        torch.cuda.synchronize()
        res_stream[n] = {"ms_per_step": e0.elapsed_time(e1) / args.stream, "replayed": r.hits,
                         "hit_rate": r.hits / args.stream}
        del r
    return {"fixed_shape_step_ms": fixed, "graph_pool_mb_per_shape": pool_mb, "varying_shape_stream": res_stream}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "dropin_train_graph.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--stream", type=int, default=40)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    w = synth.WORKLOADS["anet"]
    wt = synth.Workload(w.name, w.config_id, args.batch, w.vlen, w.tmax, w.clen, w.vdim, w.num_words, w.num_chars, w.tlen, 1)
    res = {"gpu": gpu_info(), "workload": f"anet B={args.batch} L={wt.vlen} Tmax={wt.tmax}, dropout 0.2, one GPU",
           "timing": f"fixed shape: {args.rounds} rounds x {args.steps} steps per route, alternating in one process, CUDA events; "
                     f"stream: {args.stream} batches per route from a cold cache",
           "graph_cache_size": train.GRAPH_CACHE_SIZE}
    for precision in ("fp32", "bf16"):
        res[precision] = run_precision(precision, wt, dev, args)
        print(json.dumps({precision: res[precision]}, indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
