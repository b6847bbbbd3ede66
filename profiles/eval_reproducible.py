#!/usr/bin/env python
"""Reproducible evaluation sweeps (DESIGN.md section 13):
    python profiles/eval_reproducible.py [--out profiles/eval_reproducible.json] [--rounds 5] [--batches 256] [--distinct 8]
    torchrun --nproc-per-node N profiles/eval_reproducible.py --counters [--out profiles/eval_reproducible.json]

One process:
* Cost: ``evaluate()`` at the ANet shape (bf16, default streams, ragged copies) over ``--batches`` pinned host batches cycled
  from ``--distinct`` distinct ones, with ``seed=None`` (torch's draw, plain counters) against ``seed=`` (one
  ``seqpan_gumbel_noise`` launch per batch, exact counters), on raw clips (copied by the default zero-copy kernel of 32 CTAs,
  and by DMA, ``h2d_ctas=0``) and on stored encodings of the same clips.  The six arms run in one order and then the reverse, for ``--rounds`` rounds; wall clock around each call (it ends in a
  synchronise), medians reported.  Each round also times the noise of one ANet batch alone: torch's three element-wise
  launches against one ``seqpan_gumbel_noise`` launch, CUDA events around 500 draws on one stream.
* Spread: R1@{0.3,0.5,0.7} / mIoU of the raw-clip sweep under 5 seeds (random weights: the spread is the noise's effect,
  the values themselves mean nothing).
* Counters: the fp64 bit patterns of one seeded call over ``--counter-batches`` ANet batches on this GPU.

Under torchrun (``--counters``): the same counters from N ranks, once with static round-robin shards
(``shard_batches`` ids) and once with whole batches drawn from the ``draw_chunks`` work queue over a TCPStore (one
``allreduce=False`` call per chunk, summed, one all-reduce).  Rank 0 adds them to ``--out`` under ``counters_bits``.

The GPU's name, power limit and SM clocks are read in the same run and stored with the numbers."""
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
from vmrframe_b200 import SeqPAN, _cabi, draw_chunks, engine, shard_batches, synth  # noqa: E402

COUNTER_SEED = 20261022


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def make_model(w, precision, dev):
    m = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision=precision).eval()
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=1))
    return m.to(dev)


def bits(counters):
    return [f"{int(x):016x}" for x in counters.detach().cpu().numpy().view(np.uint64)]


def host_batches(w, distinct, n):
    host = [synth.make_batch(w, i, pin=True) for i in range(distinct)]
    return host, [host[i % distinct] for i in range(n)]


def sweep_arms(m, w, dev, distinct, nbatches):
    host, raw = host_batches(w, distinct, nbatches)
    enc = m.encode_videos(torch.cat([b["vfeats"] for b in host]).to(dev))
    enc_host = []
    for i, b in enumerate(host):
        e = {k: v for k, v in b.items() if k != "vfeats"}
        e["video_index"] = (torch.arange(w.batch, dtype=torch.int32) + i * w.batch).pin_memory()
        enc_host.append(e)
    encd = [enc_host[i % distinct] for i in range(nbatches)]
    return {"raw": (raw, None, 32), "raw_dma": (raw, None, 0), "encoded": (encd, enc, 32)}


def run_sweep(m, dev, batches, enc, seed, h2d_ctas=32):
    torch.manual_seed(0)
    torch.cuda.synchronize()
    t = time.perf_counter()
    metrics, counters, info = engine.evaluate(m, batches, dev, video_encodings=enc, seed=seed, h2d_ctas=h2d_ctas)
    wall = time.perf_counter() - t
    q = sum(b["vmasks"].shape[0] for b in batches)
    return {"queries_per_s": q / wall, "wall_s": wall, "queries": q}, metrics, counters


def noise_us(dev, B, L, n=500):
    """us per draw of one batch's noise on one stream: torch's three element-wise launches against seqpan_gumbel_noise."""
    g = torch.empty(B, L, 4, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    lib = _cabi.lib()
    draws = {"noise_us_torch": lambda i: g.exponential_().log_().neg_(),
             "noise_us_seeded": lambda i: _cabi.check(lib.seqpan_gumbel_noise(7, i, B, L, g.data_ptr(), st))}
    out = {}
    for k, fn in draws.items():
        for i in range(20):
            fn(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        b.synchronize()
        out[k] = a.elapsed_time(b) * 1000.0 / n
    return out


def single(args):
    dev = torch.device("cuda:0")
    w = synth.WORKLOADS["anet"]
    res = {"gpu": gpu_info(), "precision": args.precision, "rounds": args.rounds, "batches": args.batches,
           "distinct_batches": args.distinct, "workload": "anet B=256 L=100"}
    m = make_model(w, args.precision, dev)
    arms = sweep_arms(m, w, dev, args.distinct, args.batches)
    seeds = {"unseeded": None, "seeded": 7}
    for batches, enc, h2d_ctas in arms.values():                    # warm-up of every arm
        for seed in seeds.values():
            engine.evaluate(m, batches[: 2 * args.distinct], dev, video_encodings=enc, seed=seed, h2d_ctas=h2d_ctas)
    runs = [(arm, name) for arm in arms for name in seeds]
    rounds = []
    for r in range(args.rounds):
        row = {}
        for arm, name in (runs if r % 2 == 0 else runs[::-1]):      # the order reverses every round
            batches, enc, h2d_ctas = arms[arm]
            row[f"{arm}_{name}"] = run_sweep(m, dev, batches, enc, seeds[name], h2d_ctas)[0]
        row.update(noise_us(dev, w.batch, w.vlen))
        rounds.append(row)
        print(json.dumps(row), flush=True)
    res["rounds_raw"] = rounds
    res["median"] = {k: ({f: statistics.median(rw[k][f] for rw in rounds) for f in v} if isinstance(v, dict) else
                         statistics.median(rw[k] for rw in rounds)) for k, v in rounds[0].items()}
    spread = {}
    raw = arms["raw"][0]
    for seed in range(5):
        _, metrics, _ = run_sweep(m, dev, raw, None, seed)
        spread[str(seed)] = dict(zip(("r1_iou0.3", "r1_iou0.5", "r1_iou0.5_again", "r1_iou0.7", "miou"), metrics))
    res["metrics_by_seed"] = spread
    res["metrics_spread_max_minus_min"] = {k: max(s[k] for s in spread.values()) - min(s[k] for s in spread.values())
                                           for k in next(iter(spread.values()))}
    _, counter_batches = host_batches(w, args.distinct, args.counter_batches)
    _, c, _ = engine.evaluate(m, counter_batches, dev, seed=COUNTER_SEED)
    res["counters_bits"] = {"one process": {"batches": args.counter_batches, "seed": COUNTER_SEED, "one_call": bits(c),
                                    "values": c.cpu().tolist()}}
    res["gpu_after"] = gpu_info()
    write(args.out, res)
    print(json.dumps(res["median"], indent=1))
    print(json.dumps(res["metrics_spread_max_minus_min"], indent=1))


def distributed(args):
    import datetime

    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
    w = synth.WORKLOADS["anet"]
    m = make_model(w, args.precision, dev)
    _, batches = host_batches(w, args.distinct, args.counter_batches)
    mine = shard_batches(len(batches), rank, world)
    _, static, _ = engine.evaluate(m, [batches[k] for k in mine], dev, seed=COUNTER_SEED, batch_ids=mine)
    port = int(os.environ.get("MASTER_PORT", "29500")) + 17
    store = dist.TCPStore(os.environ.get("MASTER_ADDR", "127.0.0.1"), port, world, rank == 0)
    total = torch.zeros(5, dtype=torch.float64, device=dev)
    drawn = 0
    for ids in draw_chunks(store, len(batches), world, chunk=8):
        _, c, _ = engine.evaluate(m, [batches[k] for k in ids], dev, seed=COUNTER_SEED, batch_ids=ids, allreduce=False)
        total += c
        drawn += len(ids)
    dist.all_reduce(total)
    got = [None] * world
    dist.all_gather_object(got, drawn)
    if rank == 0:
        res = {}
        if os.path.exists(args.out):
            with open(args.out) as f:
                res = json.load(f)
        res.setdefault("counters_bits", {})[f"torchrun N={world}"] = {
            "batches": args.counter_batches, "seed": COUNTER_SEED, "static_shards": bits(static), "work_queue": bits(total),
            "work_queue_batches_per_rank": got, "gpu": gpu_info()}
        write(args.out, res)
        print(json.dumps(res["counters_bits"], indent=1))
    dist.barrier()
    dist.destroy_process_group()


def write(path, res):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/eval_reproducible.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batches", type=int, default=256)
    ap.add_argument("--distinct", type=int, default=8)
    ap.add_argument("--counter-batches", type=int, default=96)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--counters", action="store_true", help="torchrun: the counters of N ranks")
    args = ap.parse_args()
    if args.counters:
        distributed(args)
    else:
        single(args)


if __name__ == "__main__":
    main()
