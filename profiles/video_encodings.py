#!/usr/bin/env python
"""Stored video encodings on one GPU (DESIGN.md section 12):
    python profiles/video_encodings.py [--out profiles/video_encodings.json] [--rounds 5] [--batches 256] [--distinct 8]

* Encode cost: ``encode_videos`` of 1024 seeded random clips (chunk 256) at the ANet (L=100) and TACoS (L=256) shapes, wall
  clock between two synchronises, per clip.
* Device-resident forward at the ANet shape (B=256, one stream, no graph replay at this size): ``forward_into`` on resident
  raw features (``seqpan_forward``) against ``forward_into`` on resident encodings of the same clips (``video_index=None``),
  CUDA events around 50 forwards after 10 warm-up forwards.
* End-to-end sweep: ``evaluate()`` (default streams, ragged copies) over ``--batches`` pinned host batches cycled from
  ``--distinct`` distinct ones.  Raw arm: ANet copies the valid rows of every clip, TACoS (128 queries per clip) copies each
  clip once with ``video_index`` (the shared-video path).  Encoded arm: the same batches without ``vfeats`` and with
  ``video_encodings`` of all their clips, encoded before the sweep (the encode is not part of the timed call).  Wall clock
  around each ``evaluate()`` call (it ends in a synchronise), queries/s and ``info["h2d_bytes"]``.

All arms alternate inside one process for ``--rounds`` rounds (medians reported).  The GPU's name, power limit and SM
clocks are read in the same run and stored with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vmrframe_b200 import SeqPAN, engine, synth  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def make_model(w, precision, dev):
    m = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision=precision).eval()
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=1))
    return m.to(dev)


def encode_cost(m, w, dev, n=1024):
    v = torch.randn(n, w.vlen, w.vdim, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    m.encode_videos(v[:256])                               # warm-up (and the handle sized for chunks of 256)
    torch.cuda.synchronize()
    t = time.perf_counter()
    m.encode_videos(v)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) / n * 1e6             # us per clip


def resident_arms(m, w, dev):
    b = synth.make_batch(w, 0, device=dev)
    B, L = w.batch, w.vlen
    g = synth.gumbel_noise(B, L).to(dev)
    enc = m.encode_videos(b["vfeats"])
    out = {k: (torch.empty(B, L, device=dev), torch.empty(B, L, device=dev), torch.empty(B, L, 4, device=dev)) for k in ("raw", "encoded")}

    def raw():
        m.forward_into(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], g, *out["raw"])

    def encoded():
        m.forward_into(b["words_ids"], b["char_ids"], None, b["vmasks"], b["tmasks"], g, *out["encoded"], None, video_encodings=enc)

    raw(); encoded()
    torch.cuda.synchronize()
    diff = max(float((x - y).abs().max()) for x, y in zip(out["raw"], out["encoded"]))
    return {"raw": raw, "encoded": encoded}, diff


def time_forwards(fn, n=50, warm=10):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / n                  # us per forward


def sweep_arms(m, w, dev, distinct, nbatches):
    host = [synth.make_batch(w, i, pin=True) for i in range(distinct)]
    if w.group > 1:
        host = [synth.share_clips(b, w.group) for b in host]
    clips = [b["vfeats"] for b in host]
    enc = m.encode_videos(torch.cat(clips).to(dev))
    enc_host, base = [], 0
    for b, c in zip(host, clips):
        e = {k: v for k, v in b.items() if k != "vfeats"}
        vi = b["video_index"] if "video_index" in b else torch.arange(b["vmasks"].shape[0], dtype=torch.int32)
        e["video_index"] = (vi + base).to(torch.int32).pin_memory()
        base += c.shape[0]
        enc_host.append(e)
    raw = [host[i % distinct] for i in range(nbatches)]
    encd = [enc_host[i % distinct] for i in range(nbatches)]
    return {"raw": (raw, None), "encoded": (encd, enc)}


def run_sweep(m, dev, batches, enc):
    torch.manual_seed(0)
    torch.cuda.synchronize()
    t = time.perf_counter()
    _, _, info = engine.evaluate(m, batches, dev, return_fracs=True, video_encodings=enc)
    wall = time.perf_counter() - t
    q = sum(b["vmasks"].shape[0] for b in batches)
    return {"queries_per_s": q / wall, "wall_s": wall, "h2d_bytes": info["h2d_bytes"], "queries": q}, info["fracs"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/video_encodings.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batches", type=int, default=256)
    ap.add_argument("--distinct", type=int, default=8)
    ap.add_argument("--precision", default="bf16")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "precision": args.precision, "rounds": args.rounds, "batches": args.batches,
           "distinct_batches": args.distinct}
    shapes = {"anet": synth.WORKLOADS["anet"], "tacos": synth.WORKLOADS["tacos"]}
    models = {k: make_model(w, args.precision, dev) for k, w in shapes.items()}
    arms, diff = resident_arms(models["anet"], shapes["anet"], dev)
    res["resident_anet_max_abs_diff_raw_vs_encoded"] = diff
    sweeps = {k: sweep_arms(models[k], w, dev, args.distinct, args.batches) for k, w in shapes.items()}
    for k in shapes:                                        # warm-up of every sweep arm
        for batches, enc in sweeps[k].values():
            engine.evaluate(models[k], batches[: 2 * args.distinct], dev, video_encodings=enc)
    rounds = []
    for r in range(args.rounds):
        row = {}
        for k, w in shapes.items():
            row[f"encode_us_per_clip_{k}"] = encode_cost(models[k], w, dev)
        for arm, fn in arms.items():
            row[f"resident_anet_us_{arm}"] = time_forwards(fn)
        for k in shapes:
            fr = {}
            for arm, (batches, enc) in sweeps[k].items():
                row[f"e2e_{k}_{arm}"], fr[arm] = run_sweep(models[k], dev, batches, enc)
            row[f"e2e_{k}_equal_span_share"] = float(np.mean(np.concatenate([np.all(a == b, axis=1) for a, b in
                                                                             zip(fr["raw"], fr["encoded"])])))
        rounds.append(row)
        print(json.dumps(row), flush=True)
    res["rounds_raw"] = rounds
    med = {}
    for key in rounds[0]:
        v = rounds[0][key]
        if isinstance(v, dict):
            med[key] = {f: statistics.median(rw[key][f] for rw in rounds) for f in v}
        else:
            med[key] = statistics.median(rw[key] for rw in rounds)
    res["median"] = med
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(med, indent=1))


if __name__ == "__main__":
    main()
