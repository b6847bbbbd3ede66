#!/usr/bin/env python
"""Cost of top-k span retrieval with temporal NMS on one GPU:
    python profiles/topk_decode.py [--out profiles/topk_decode.json] [--rounds 5] [--batches 24]

* Kernel time: ``seqpan_span_topk`` (and ``seqpan_span_decode`` for comparison) at the Charades (B=32, L=64), ANet (B=256,
  L=100) and TACoS (B=128, L=256) shapes, k in {1, 5, 10}, NMS thresholds 0.5 and 1.0, on seeded random logits (scale 2,
  random valid lengths).  CUDA events around 200 back-to-back launches after 20 warm-up launches; the inputs are a few hundred
  KB, so they sit in L2, as they do right after the forward that produced them.
* The device-resident ANet forward (bf16, B=256), the yardstick of the 5 % budget: CUDA events around 50 forwards.
* The ANet ``evaluate()`` sweep (bf16, default streams) with and without ``topk=5``, alternating in one process for
  ``--rounds`` rounds, wall clock of each call.

The GPU's name, power limit and SM clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, _cabi, engine, synth  # noqa: E402

SHAPES = {"charades": (32, 64), "anet": (256, 100), "tacos": (128, 256)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def logits(B, L, dev, seed):
    g = torch.Generator().manual_seed(seed)
    s, e = torch.randn(B, L, generator=g) * 2, torch.randn(B, L, generator=g) * 2
    lens = torch.randint(L // 4, L + 1, (B,), generator=g)
    m = (torch.arange(L).expand(B, L) < lens.unsqueeze(1)).float()
    return s.to(dev), e.to(dev), m.to(dev)


def time_launches(fn, n=200, warm=20):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / n      # microseconds per launch


def kernel_table(dev):
    L_ = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    rows = []
    for name, (B, L) in SHAPES.items():
        s, e, m = logits(B, L, dev, B + L)
        fr = torch.empty(B, 2, device=dev)
        dec = time_launches(lambda: _cabi.check(L_.seqpan_span_decode(s.data_ptr(), e.data_ptr(), m.data_ptr(), B, L, None, None,
                                                                      fr.data_ptr(), st)))
        rows.append({"shape": name, "B": B, "L": L, "kernel": "span_decode", "us": dec})
        for k in (1, 5, 10):
            si = torch.empty(B, k, dtype=torch.int64, device=dev)
            ei, sc, tf = torch.empty_like(si), torch.empty(B, k, device=dev), torch.empty(B, k, 2, device=dev)
            for thr in (0.5, 1.0):
                us = time_launches(lambda: _cabi.check(L_.seqpan_span_topk(
                    s.data_ptr(), e.data_ptr(), m.data_ptr(), B, L, k, thr, si.data_ptr(), ei.data_ptr(), sc.data_ptr(),
                    tf.data_ptr(), st)))
                rows.append({"shape": name, "B": B, "L": L, "kernel": "span_topk", "k": k, "nms_thresh": thr, "us": us})
                print(json.dumps(rows[-1]), flush=True)
    return rows


def stats(xs):
    s = sorted(xs)
    return {"mean": sum(s) / len(s), "min": s[0], "max": s[-1], "spread_pct": 100.0 * (s[-1] - s[0]) / s[0], "rounds": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "topk_decode.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batches", type=int, default=24)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "kernels": kernel_table(dev)}

    w = synth.WORKLOADS["anet"]
    model = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision="bf16", sync_timing=False).eval()
    model.load_state_dict(synth.randomize_state_dict(model.state_dict(), seed=w.config_id))
    model.to(dev)
    b = {k: v.to(dev) for k, v in synth.make_batch(w, 0).items()}
    g = synth.gumbel_noise(w.batch, w.vlen).to(dev)
    fwd = time_launches(lambda: model(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], gumbel=g),
                        n=50, warm=5)
    res["anet_forward_us"] = fwd
    topk5 = [r["us"] for r in res["kernels"] if r["shape"] == "anet" and r.get("k") == 5]
    res["anet_topk5_share_of_forward_pct"] = {thr: 100.0 * us / fwd for thr, us in zip((0.5, 1.0), topk5)}

    host = [synth.make_batch(w, i, pin=True) for i in range(args.batches)]
    engine.evaluate(model, host[:4], dev)                     # warm-up, both variants
    engine.evaluate(model, host[:4], dev, topk=5)
    walls = {"plain": [], "topk5": []}
    for r in range(args.rounds):
        order = ("plain", "topk5") if r % 2 == 0 else ("topk5", "plain")
        for v in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, _, info = engine.evaluate(model, host, dev, topk=5 if v == "topk5" else None)
            walls[v].append(time.perf_counter() - t0)
            if v == "topk5":
                res["anet_sweep_recall_at_5"] = info["topk"]["recall"]
    res["anet_sweep_s"] = {v: stats(x) for v, x in walls.items()}
    res["anet_sweep_batches"] = args.batches
    res["anet_sweep_overhead_pct"] = 100.0 * (res["anet_sweep_s"]["topk5"]["mean"] / res["anet_sweep_s"]["plain"]["mean"] - 1)
    print(json.dumps({k: v for k, v in res.items() if k != "kernels"}, indent=1))
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
