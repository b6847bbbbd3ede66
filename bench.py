#!/usr/bin/env python
"""SeqPAN hot-path benchmark: queries/s of forward + span decode on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload anet|charades|tacos] [--dump-outputs DIR]

One "step" = one pass of the hot path (SeqPAN.forward + infer_basic span decode + IoU counters) over one
ActivityNet-shaped batch (B=256, L=100, 1024-d features; BASELINE.json configs[1]) of synthetic input.
  value      whole-job queries/s with the inputs already resident in HBM (8 distinct batches per GPU are cycled:
             8 x 105 MB > the 126 MB L2, so no step finds its input in cache), timed with CUDA events on the
             launching stream between barrier+synchronize pairs, max over ranks.
  e2e        the same metric through the public host API (vmrframe_b200.evaluate) with PINNED HOST batches: every
             step's host->device copy and the device->host read of its span fractions are inside the timed region.
  roofline   the dominant kernel of the step (per-launch CUDA-event timing inside the library, seqpan_set_profile).
  cpu_baseline / --impl reference
             the reference's algorithm on the box's host cores: the oracle port (oracle/seqpan_oracle.py, a fp32
             restatement pinned to reference-generated fixtures; the reference itself is pure Python + torch and
             cannot travel to the GPU box) with all host threads, on a bounded sample of the same workload.
  parity     GPU outputs of one timed batch against the oracle's (same weights, same injected noise): error of the logits /
             match scores and span equality outside near-ties (computed in the cpu_baseline leg, which already runs the oracle).
  gpu_eager_baseline
             the reference's algorithm (oracle port) in PyTorch eager on the same B200 -- cuDNN / cuBLAS library kernels,
             sync-bracketed like models/SeqPAN.py:51-52,85-87 -- with cudnn.allow_tf32 True and False: the on-box bar.
  sustained  the same device-resident sweep and the same e2e sweep run for >= 3 s each (after the driver-timed region),
             with their own clock / power samples.
  --sweep N  BASELINE.json configs[3]: N synthetic pairs through vmrframe_b200.evaluate (host batches, sharded over the
             ranks, one NCCL all-reduce of the counters), reported as its own JSON line.
With torchrun (N>1) every rank owns whole batches (weights replicated, no collective in the forward) and the sweep
ends with ONE NCCL all-reduce of the 5 IoU counters; scaling is weak (per-GPU work fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before the CUDA context exists (see vmrframe_b200/_cabi.py)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "seqpan_queries_per_sec"
UNIT = "queries/s"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm": p["hbm_gbs"], "tc_burst": p["bf16_tflops"], "tc_sustained": p["bf16_tflops_sustained"],
                "src": "measured"}
    except Exception:
        return {"hbm": 6650.0, "tc_burst": 1590.0, "tc_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(local):
    """Pins this rank's CPU affinity to the NUMA node its GPU hangs off (sysfs), BEFORE the pinned host batches are
    allocated, so that they are first-touched on that node: with 8 ranks per box the e2e sweep otherwise pulls half of its
    PCIe reads across the socket interconnect.  Best effort: returns the node or None."""
    try:
        prop = torch.cuda.get_device_properties(local)
        bdf = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def workload_string(w):
    """config.workload: identical in the native and the reference arm (the driver compares them)."""
    tag = {"charades": " (BASELINE.json configs[0])", "anet": " (BASELINE.json configs[1])", "tacos": " (BASELINE.json configs[2])"}
    return f"{w.name}: B={w.batch} L={w.vlen} vdim={w.vdim} Tmax={w.tmax} C={w.clen}" + tag.get(w.name, "")


def step_work(B, L, T, C, vdim):
    """Algorithmic work of ONE forward step per launch tag: tag -> (FLOPs, HBM bytes), both per step (all launches of
    the tag).  DESIGN.md section 5 states the same figures.  Rows: Mv = B*L video, Mt = B*T text, M = Mv + Mt."""
    Mv, Mt = B * L, B * T
    M, D = Mv + Mt, 128
    lin = lambda m, n, k, inb=4, outb=4: (2.0 * m * n * k, m * k * inb + m * n * outb + n * k * 2)
    enc_rows = M + 2 * Mv                                  # shared encoder (joint rows) + 2 predictor conv blocks
    cq_core = lambda F, S: 2.0 * B * D * (F + S) + 4.0 * B * F * S * D + 2.0 * B * F * S * D * 2
    conv = (4 * (2.0 * enc_rows * D * D + 2.0 * enc_rows * D * 7), 2.0 * enc_rows * D * 4)
    # the same three launches with the consumer's LayerNorm + projections fused behind the last layer: the shared encoder
    # also emits q|fk|fv|tk|tv of the first DualAttentionBlock (bf16), the two predictor blocks emit in_proj's q|k|v
    # (head-blocked bf16 rows: 3 x 128 values + the 16-column mask boxes of q and k = 1024 bytes per predictor row)
    tails = (2.0 * M * D * 640 + 2 * 2.0 * Mv * D * 384, M * 640 * 2 + 2 * Mv * 512 * 2)
    return {
        "chain_conv_block": conv,
        "chain_conv_block+proj": (conv[0] + tails[0], conv[1] + tails[1]),
        "chain_enc_layer": (4 * (2.0 * enc_rows * D * D + 2.0 * enc_rows * D * 7), 4 * 2.0 * enc_rows * D * 4),
        # ONE launch per step in the fused default: LN1 -> q|fk|fv, LNt -> tk|tv (bf16) of the second DualAttentionBlock
        # (the first block's and the predictor's projections ride behind the conv blocks, see `tails`)
        "chain_proj_ln": (2.0 * M * D * 640, M * D * 4 + M * 640 * 2),
        "attn_dual_tc": (2 * 4.0 * B * D * (L + T) ** 2, 2 * (M * 640 * 2 + 2 * M * D * 2)),
        "launch_dual_attention": (2 * 4.0 * B * D * (L + T) ** 2, 2 * (M * 640 * 4 + 2 * M * D * 4)),
        "chain_dab_post": (2 * 11 * 2.0 * M * D * D, 2 * (2 * M * D * 2 + 2 * M * D * 4)),
        "launch_cq_attention": (cq_core(L, T) + cq_core(T, L), M * D * 4 + M * 512 * 4),
        # fused CQAttention + cqa_linear: joint rows (fp32) in, t2v / v2t rows (fp32) out; the 512-wide concat never exists
        "cq_attention_tc": (cq_core(L, T) + cq_core(T, L) + 2.0 * M * 512 * D, 2 * M * D * 4),
        # head-blocked q|k|v rows (1024 bytes with the mask boxes) in, bf16 rows out
        "attn_batch_tc": (2 * 4.0 * L * B * B * D, 2 * (Mv * 512 * 2 + Mv * D * 2)),
        "launch_batch_attention": (2 * 4.0 * L * B * B * D, 2 * (Mv * 384 * 4 + Mv * D * 4)),
        "chain_fep_tail": (2 * 2 * 2.0 * Mv * D * D, 2 * (Mv * D * 2 + 2 * Mv * D * 4)),
        # FEP tail + logit head in one launch: out_proj, dense, hidden (K = 256); att + x (bf16) and h (fp32) in, out (fp32) + logit out
        "chain_fep_head": (2 * (2 * 2.0 * Mv * D * D + 2.0 * Mv * 256 * D), 2 * (2 * Mv * D * 2 + 2 * Mv * D * 4 + Mv * 4)),
        # concat projection (t2v half, K = 128) + match head: t2v (fp32) in, fuse2 fp32 + bf16 + match_score out
        "chain_fuse_match": (2.0 * Mv * D * D + 2.0 * Mv * D * 8, Mv * D * 4 + Mv * D * 6 + Mv * 32.0),
        "pool_bias": (4.0 * Mt * D + 2.0 * B * D * D, Mt * D * 4.0 + B * D * 4.0),
        "gather_clips": (0.0, 2.0 * Mv * D * 4),
        "chain_head": (2 * 2.0 * Mv * 256 * D, 2 * (2 * Mv * D * 4 + Mv * 4)),
        "tc_linear_tf32_video": lin(Mv, D, vdim),
        "tc_linear_tf32_video+ln": lin(Mv, D, vdim),
        "tc_linear_N128_K1024": lin(Mv, D, vdim),
        "tc_linear_N128_K400": lin(Mt, D, 400),
        "tc_linear_tf32_query+ln": lin(Mt, D, 400),
        "tc_linear_N128_K512": (lin(Mv, D, 512)[0] + lin(Mt, D, 512)[0], lin(Mv, D, 512)[1] + lin(Mt, D, 512)[1]),
        "tc_linear_N128_K256": lin(Mv, D, 256),
        "launch_embed_text": (0.0, Mt * 400 * 4.0 + Mt * 300 * 4.0 + Mt * (C + 1) * 8.0),
        "launch_match_head": (2.0 * Mv * D * 8, 2.0 * Mv * D * 4 + Mv * 32.0),
        "launch_layernorm": (0.0, 2.0 * M * D * 4),
        "launch_pool_tile": (4.0 * Mt * D, Mt * D * 4.0 + Mv * D * 4.0),
        "launch_build_rowmask": (0.0, 2.0 * M * 4),
    }


def roofline_of(tag, n_launches, ms_total, work, peaks, share, traffic=None):
    """Roofline entry of one kernel tag.  bound = the slower of (FLOPs / tensor peak) and (DRAM bytes / HBM peak), where the DRAM
    bytes are the ncu-measured dram__bytes of the launch when profiles/ncu_traffic.json has them (intermediates that stay in the
    126 MB L2 between two kernels never reach HBM, so counting them would label a contraction "hbm-bound") and the algorithmic
    bytes otherwise.  Both fractions are always reported."""
    flops, nbytes = work
    per_launch_s = ms_total * 1e-3 / max(n_launches, 1)
    f_l, b_l = flops / n_launches, nbytes / n_launches
    dram = float(traffic) if traffic else b_l
    t_tc, t_hbm = f_l / (peaks["tc_sustained"] * 1e12), dram / (peaks["hbm"] * 1e9)
    tf, gbs = f_l / per_launch_s / 1e12, b_l / per_launch_s / 1e9
    common = {"kernel": tag, "traffic": traffic, "us_per_launch": per_launch_s * 1e6, "share_of_step": share,
              "algorithmic_flops_per_launch": f_l, "algorithmic_bytes_per_launch": b_l,
              "tensor_frac": tf / peaks["tc_sustained"], "hbm_frac_algorithmic": gbs / peaks["hbm"],
              "hbm_frac_dram": (dram / per_launch_s / 1e9) / peaks["hbm"]}
    if t_tc >= t_hbm:
        return {"bound": "tensor", "achieved": tf, "peak": peaks["tc_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["tc_sustained"],
                "peak_source": peaks["src"] + " (sustained bf16)", **common}
    ach = dram / per_launch_s / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
            "peak_source": peaks["src"], **common}


def run_reference(args, w, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port) on the host cores, rank 0 only."""
    if rank != 0:
        return
    from oracle import seqpan_oracle as O
    from vmrframe_b200 import SeqPAN, synth
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    sd = {k: v.detach() for k, v in SeqPAN(synth.make_configs(w), synth.make_word_vectors(w)).state_dict().items()}
    Bs = w.batch

    def one(batch, g):
        with torch.no_grad():
            out = O.forward(sd, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
            return O.infer_basic(out["slogits"], out["elogits"], batch["vmasks"])

    # bound the sample so the whole run ends within a few minutes on any host
    probe = synth.make_batch(w, 0)
    g = synth.gumbel_noise(w.batch, w.vlen)
    t0 = time.perf_counter(); one(probe, g); t1 = time.perf_counter() - t0
    budget = 150.0 / max(args.steps + args.warmup, 1)
    while t1 * Bs / w.batch > budget and Bs > 8:
        Bs //= 2
    ws = synth.Workload(w.name, w.config_id, Bs, w.vlen, w.tmax, w.clen, w.vdim, w.num_words, w.num_chars, w.tlen, w.group)
    batches = [synth.make_batch(ws, i) for i in range(4)]
    gs = synth.gumbel_noise(Bs, w.vlen)
    for i in range(args.warmup):
        one(batches[i % 4], gs)
    t0 = time.perf_counter()
    for i in range(args.steps):
        one(batches[i % 4], gs)
    dt = time.perf_counter() - t0
    qps = args.steps * Bs / dt
    cores = torch.get_num_threads()
    sample = f"{args.steps} steps x {Bs} pairs of the {w.name} shape (B={Bs}, L={w.vlen}), fp32, torch CPU, {cores} threads"
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(w), "sample_batch": Bs},
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_train(args, w, dev, rank, world):
    """BASELINE.json configs[4]: one optimisation step = train_engine_SeqPAN's forward (dropout 0.2) + lossfun_loc + lossfun_match +
    backward + ONE flat-bucket NCCL all-reduce of the live gradients + clip_grad_norm_(1.0) + AdamW, per rank on its own batch
    of --train-batch ANet-shaped pairs (data parallel, weak scaling).  fp32 kernels (csrc/train_ops.cu): first correct version."""
    from vmrframe_b200 import SeqPAN, synth
    from vmrframe_b200.train import TrainStep
    Bt = args.train_batch
    wt = synth.Workload(w.name, w.config_id, Bt, w.vlen, w.tmax, w.clen, w.vdim, w.num_words, w.num_chars, w.tlen, 1)
    torch.manual_seed(0)
    model = SeqPAN(synth.make_configs(wt, droprate=0.2), synth.make_word_vectors(wt), precision="bf16", sync_timing=False).train().to(dev)
    batches = [{k: v.to(dev) for k, v in synth.add_train_labels(synth.make_batch(wt, 1000 * rank + i)).items()} for i in range(4)]
    ts = TrainStep(model, lr=1e-4, num_train_steps=1)
    ts_repack, model.repack = model.repack, (lambda: None)     # the inference handle is not used between training steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    losses = []
    use_graph = not args.no_train_graph
    for i in range(max(3, args.warmup) + (12 if use_graph else 0)):      # graph mode: two eager steps + one capture per input shape
        losses.append(float(ts.step(batches[i % 4], graph=use_graph)[0]))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    th0 = time.perf_counter()
    for i in range(args.steps):
        loss = ts.step(batches[i % 4], graph=use_graph)[0]
    e1.record()
    host_ms = (time.perf_counter() - th0) * 1e3 / args.steps
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    if rank != 0:
        return
    eager = None
    if world == 1 and not args.no_eager_baseline:
        # the on-box bar of this config: the reference's training step in PyTorch eager on the same GPU -- oracle port forward with
        # F.dropout at the reference's sites, the two losses, autograd backward, clip_grad_norm_(1.0), torch.optim.AdamW
        from oracle import seqpan_oracle as O
        import torch.nn.functional as F
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        params = {k: sd[k].requires_grad_(True) for k, p in model.named_parameters() if p.requires_grad}
        opt = torch.optim.AdamW(list(params.values()), lr=1e-4)
        O.DROP = lambda x: F.dropout(x, 0.2, True)
        try:
            def one(b):
                g = -torch.empty(Bt, wt.vlen, 4, device=dev).exponential_().log()
                out = O.forward(sd, b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], g)
                l = O.lossfun_loc(out["slogits"], out["elogits"], b["label1ds"][:, 0], b["label1ds"][:, 1]) + \
                    O.lossfun_match(out["match_score"], sd["label_embs"], b["NER_labels"], b["vmasks"])
                opt.zero_grad()
                l.backward()
                torch.nn.utils.clip_grad_norm_(list(params.values()), 1.0)
                opt.step()
            for i in range(3):
                one(batches[i % 4])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(10):
                one(batches[i % 4])
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / 10
            eager = {"value": Bt / dt, "unit": "pairs/s", "ms_per_step": dt * 1e3,
                     "what": "oracle port + torch autograd + clip_grad_norm_ + torch.optim.AdamW in PyTorch eager on this GPU, fp32 "
                             f"(cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}), 10 steps"}
        except Exception as ex:
            eager = {"error": repr(ex)[:200]}
        finally:
            O.DROP = None
    nlive = sum(g.numel() for g in [ts.flat]) if ts.flat is not None else 0
    line = {"metric": "seqpan_train_pairs_per_sec", "value": world * args.steps * Bt / (ms / 1e3), "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"training step on {wt.name}-shaped batches: B={Bt} per GPU, L={wt.vlen}, Tmax={wt.tmax}, droprate 0.2 "
                                   "(BASELINE.json configs[4])",
                       "global_batch": world * Bt, "parallelism": f"data parallel x{world}: one flat-bucket all-reduce of {nlive} live gradient "
                       "elements per step (NCCL), then clip_grad_norm_(1.0) + AdamW on every rank",
                       "timing": "CUDA events around K optimisation steps, barrier+synchronize both sides, max over ranks"},
            "first_losses": losses[:3], "last_loss": float(loss), "gpu_launches": None, "host_enqueue_ms_per_step": host_ms,
            "cuda_graph": use_graph, "gpu_eager_baseline": eager}
    print(json.dumps(line), flush=True)


def run_sweep(args, w, model, host, dev, rank, world, numa_node):
    """BASELINE.json configs[3]: a batch-sharded eval sweep of `--sweep` synthetic pairs.  Whole reference batches are dealt
    round-robin to the ranks (batch k -> rank k mod N; the predictor attends across a batch, so a batch is the unit), every
    rank runs vmrframe_b200.evaluate on its share (host batches: `--resident` distinct pinned batches cycled, H2D copies and
    the D2H read of every batch's spans inside the timed region), and ONE NCCL all-reduce of the 5 IoU counters closes it."""
    from vmrframe_b200 import evaluate, shard_batches, draw_chunks
    B = w.batch
    n_batches = (args.sweep + B - 1) // B
    ragged = not args.no_ragged_h2d
    es = args.e2e_streams or max(1, args.streams)
    dynamic = world > 1 and not args.static_shards
    store = None
    if dynamic:
        # Work queue instead of static round-robin shards: the 8-GPU box feeds its GPUs unevenly over PCIe (23.5 vs 36.5 GB/s,
        # profiles/h2d_ceiling_8gpu.json), so with equal shares the slow-fed ranks set the time.  Ranks draw CHUNKS of whole
        # batches from one atomic counter (a TCPStore next to the rendezvous store); a batch is still never split.
        port = int(os.environ.get("MASTER_PORT", "29500")) + 17
        store = dist.TCPStore(os.environ.get("MASTER_ADDR", "127.0.0.1"), port, world, rank == 0)
    chunk = max(8, args.sweep_chunk)
    mine = shard_batches(n_batches, rank, world)
    warm = [host[k % len(host)] for k in mine[: min(6, len(mine))]]
    evaluate(model, warm, dev, streams=es, ragged_h2d=ragged, h2d_ctas=args.h2d_ctas)   # warm-up
    model.freeze()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    barrier()
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES")
    local = dev.index or 0
    sampler = ClockSampler(cvd.split(",")[local] if cvd else local) if rank == 0 else None
    t0 = time.perf_counter()
    done, h2d_bytes = 0, 0
    if not dynamic:
        batches = [host[k % len(host)] for k in mine]
        metrics, cnt, info = evaluate(model, batches, dev, streams=es, ragged_h2d=ragged, h2d_ctas=args.h2d_ctas)
        done, h2d_bytes = len(batches), info["h2d_bytes"]
        total = cnt.clone()
    else:
        total = torch.zeros(5, dtype=torch.float64, device=dev)
        # guided self-scheduling (vmrframe_b200.engine.draw_chunks): big chunks while much is left (a chunk ends with a pipeline
        # drain), small ones at the end (the last chunk of the slowest rank is the imbalance)
        for ids in draw_chunks(store, n_batches, world, chunk):
            _, cnt, info = evaluate(model, [host[k % len(host)] for k in ids], dev, streams=es, ragged_h2d=ragged,
                                    h2d_ctas=args.h2d_ctas, allreduce=False)
            total += cnt
            done += len(ids)
            h2d_bytes += info["h2d_bytes"]
        dist.all_reduce(total, op=dist.ReduceOp.SUM)   # the sweep's single collective: the 5 IoU counters
        from vmrframe_b200 import metrics_from_counters
        metrics = metrics_from_counters(total.cpu().tolist())
        cnt = total
    barrier()
    sec = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    h2d = torch.tensor([float(h2d_bytes)], device=dev, dtype=torch.float64)
    per_rank = torch.zeros(world, device=dev, dtype=torch.float64)
    per_rank[rank] = done
    if world > 1:
        dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        dist.all_reduce(h2d, op=dist.ReduceOp.SUM)
        dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    clocks = sampler.stop() if sampler else None
    if rank != 0:
        return
    pairs = n_batches * B
    sec = float(sec.item())
    line = {"metric": METRIC, "value": pairs / sec, "unit": UNIT, "n_gpus": world, "steps": n_batches, "warmup": len(warm),
            "ms_per_step": sec / max(n_batches / world, 1) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "tf32": "tf32", "fp32": "f32"}[args.precision], "data": "synthetic",
            "config": {"workload": f"sweep of {pairs} pairs = {n_batches} batches of {workload_string(w)} (BASELINE.json configs[3])",
                       "global_batch": world * B, "streams": es, "numa_node": numa_node, "model": args.model,
                       "parallelism": (f"whole batches drawn in guided chunks (8..{2 * chunk}) from one atomic counter by {world} ranks" if dynamic else
                                       f"whole batches round-robin over {world} rank(s)") + ", no forward collective, 1 all-reduce of 5 IoU counters",
                       "batches_per_rank": [int(x) for x in per_rank.cpu().tolist()],
                       "cache": f"{len(host)} distinct pinned host batches per rank cycled ({len(host) * B * w.vlen * w.vdim * 4 / 1e6:.0f} MB)",
                       "timing": "wall clock around evaluate() between barrier+synchronize pairs, max over ranks"},
            "clocks": clocks, "seconds": sec, "pairs": pairs, "counted_pairs": float(cnt[0].item()),
            "e2e": {"value": pairs / sec, "unit": UNIT, "h2d_bytes_per_step": float(h2d.item()) / n_batches,
                    "d2h_bytes_per_step": B * 8, "aggregate_h2d_GBps": float(h2d.item()) / sec / 1e9},
            "gpu_launches": None,
            "metrics_check": {"r1i3": metrics[0], "r1i5": metrics[1], "r1i7": metrics[3], "miou": metrics[4]}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="anet", choices=["anet", "charades", "tacos"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--resident", type=int, default=8, help="distinct batches kept resident in HBM per GPU")
    ap.add_argument("--streams", type=int, default=2, help="CUDA streams (kernel contexts) consecutive batches alternate on")
    ap.add_argument("--no-ragged-h2d", action="store_true", help="e2e: copy the full zero-padded feature tensor")
    ap.add_argument("--h2d-ctas", type=int, default=32, help="e2e ragged copy: CTAs of the zero-copy kernel (0: one DMA per sample)")
    ap.add_argument("--e2e-streams", type=int, default=0, help="compute streams of the e2e sweep (0: same as --streams)")
    ap.add_argument("--model", default="seqpan", choices=["seqpan", "basefast"],
                    help="seqpan (the BASELINE.json metric) or the sibling model BaseFast (SURVEY.md section 8 row f3)")
    ap.add_argument("--sweep", type=int, default=0, metavar="PAIRS",
                    help="BASELINE.json configs[3]: run PAIRS synthetic query-video pairs through evaluate() (host batches, "
                         "sharded over the ranks) and print that as the JSON line instead of the step benchmark")
    ap.add_argument("--train", action="store_true",
                    help="BASELINE.json configs[4]: time the TRAINING step (forward with dropout + losses + backward + gradient "
                         "all-reduce + clip + AdamW, vmrframe_b200.train.TrainStep) on ANet-shaped batches of --train-batch pairs per GPU")
    ap.add_argument("--train-batch", type=int, default=64)
    ap.add_argument("--no-train-graph", action="store_true", help="--train: issue every kernel from the Python tape instead of replaying a CUDA graph")
    ap.add_argument("--static-shards", action="store_true", help="--sweep at N > 1: batch k -> rank k mod N instead of the work queue")
    ap.add_argument("--sweep-chunk", type=int, default=32, help="--sweep at N > 1: batches a rank draws from the queue at a time")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the eager-GPU baseline (oracle port on the B200)")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 3 s sustained sweeps")
    ap.add_argument("--sustain-seconds", type=float, default=3.0)
    ap.add_argument("--shared-video", action="store_true",
                    help="dense-query workloads (tacos: 128 pairs per clip): every clip is stored, copied and encoded once "
                         "(forward(video_index=...), SURVEY.md section 8 row f1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (slogits, elogits, match_score, "
                         "span_fracs; rank 0) as DIR/<name>.npy in float32, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.train or args.sweep > 0):
        ap.error("--dump-outputs applies to the step benchmark (not to --impl reference, --train or --sweep)")

    from vmrframe_b200 import synth
    w = synth.WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return

    from vmrframe_b200 import BaseFast, IouCounters, SeqPAN, evaluate, infer_basic_device, _cabi
    if args.model == "basefast":
        SeqPAN = BaseFast
    _cabi.require_device()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout at the first collective: keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            import datetime
            # a short collective timeout: a rank-asymmetric bug must fail in two minutes, not hold 8 GPUs for NCCL's default ten
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)

    numa_node = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.manual_seed(0)  # PyTorch default init under seed 0 (BASELINE.md §3)
    model = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision=args.precision, sync_timing=False).eval().to(dev)
    host = [synth.make_batch(w, 1000 * rank + i, pin=True) for i in range(args.resident)]
    if args.shared_video:
        if w.group <= 1:
            raise SystemExit(f"--shared-video needs a workload whose pairs share clips (tacos); {w.name} has group=1")
        host = [synth.share_clips(b, w.group) for b in host]
    resident = [{k: v.to(dev) for k, v in b.items()} for b in host]
    B, L = w.batch, w.vlen
    T, C = host[0]["words_ids"].shape[1], host[0]["char_ids"].shape[2]
    if args.train:
        run_train(args, w, dev, rank, world)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.sweep > 0:
        run_sweep(args, w, model, host, dev, rank, world, numa_node)
        if world > 1:
            dist.destroy_process_group()
        return
    counters = IouCounters(dev)
    launches = [0]
    lib = _cabi.lib()

    main_stream = torch.cuda.current_stream(dev)
    lanes = [main_stream] + [torch.cuda.Stream(dev) for _ in range(max(1, args.streams) - 1)]
    # every lane owns its noise / output buffers (nothing is allocated inside the timed region)
    f32 = torch.float32
    bufs = [{"gumbel": torch.empty(B, L, 4, dtype=f32, device=dev), "slogits": torch.empty(B, L, dtype=f32, device=dev),
             "elogits": torch.empty(B, L, dtype=f32, device=dev), "match": torch.empty(B, L, 4, dtype=f32, device=dev),
             "fracs": torch.empty(B, 2, dtype=f32, device=dev)} for _ in lanes]

    def step(i, lane_id=None):
        k = (i % len(lanes)) if lane_id is None else lane_id
        b, o = resident[i % len(resident)], bufs[k]
        with torch.cuda.stream(lanes[k]):
            model.use_context(k)
            o["gumbel"].exponential_().log_().neg_()     # F.gumbel_softmax's draw (models/SeqPAN.py:79), 3 torch kernels
            model.forward_into(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], o["gumbel"],
                               o["slogits"], o["elogits"], o["match"], b.get("video_index"))
            st = lanes[k].cuda_stream
            _cabi.check(lib.seqpan_span_decode(o["slogits"].data_ptr(), o["elogits"].data_ptr(), b["vmasks"].data_ptr(),
                                               B, L, None, None, o["fracs"].data_ptr(), st))
            _cabi.check(lib.seqpan_iou_counters(o["fracs"].data_ptr(), b["se_fracs"].data_ptr(), B,
                                                counters.buf.data_ptr(), st))
        launches[0] += model.last_launch_count() + 2   # + span decode + IoU counters (torch's 3 RNG kernels not counted)

    def fork():      # every lane starts after what the main stream has enqueued so far
        ev = torch.cuda.Event(); ev.record(main_stream)
        for ln in lanes[1:]:
            ln.wait_event(ev)

    def join():      # the main stream waits for every lane
        for ln in lanes[1:]:
            ev = torch.cuda.Event(); ev.record(ln)
            main_stream.wait_event(ev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: at least W steps, and enough for every (lane, resident batch) argument set to have been seen twice -- the
    # library replays a forward as ONE CUDA graph from the second time it sees the same pointers (seqpan_api.cu), so the
    # captures happen here and not inside the timed region
    import math
    n_warm = max(args.warmup, 2 * math.lcm(len(lanes), len(resident)))
    fork()
    for i in range(n_warm):
        step(i)
    join()
    model.freeze()
    barrier()
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES")
    smi_index = cvd.split(",")[local] if cvd else local
    sampler = ClockSampler(smi_index) if rank == 0 else None
    launches[0] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    th0 = time.perf_counter()
    e0.record()
    fork()
    for i in range(args.steps):
        step(i)
    join()
    counters.allreduce()     # the sweep's single collective (NCCL) sits inside the timed region
    e1.record()
    timed_launches = launches[0]   # the timed region only (the sustained legs below keep calling step())
    host_enqueue_ms = (time.perf_counter() - th0) * 1e3 / args.steps
    barrier()
    if args.dump_outputs and rank == 0:
        # read back now: the e2e, sustained and profiling passes below reuse the lane buffers
        import numpy as np
        o = bufs[(args.steps - 1) % len(lanes)]
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, key in (("slogits", "slogits"), ("elogits", "elogits"), ("match_score", "match"), ("span_fracs", "fracs")):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), o[key].cpu().numpy().astype(np.float32))
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop() if sampler else None
    value = world * args.steps * B / (ms / 1e3)

    # ---- e2e through the public API with pinned host batches --------------------------------------------------
    e2e_batches = [host[i % len(host)] for i in range(args.steps)]
    ragged = not args.no_ragged_h2d
    es = args.e2e_streams or len(lanes)
    evaluate(model, e2e_batches[: min(6, len(e2e_batches))], dev, streams=es, ragged_h2d=ragged, h2d_ctas=args.h2d_ctas)   # warm-up
    barrier()
    t0 = time.perf_counter()
    metrics, cnt, info = evaluate(model, e2e_batches, dev, streams=es, ragged_h2d=ragged, h2d_ctas=args.h2d_ctas)
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e = {"value": world * args.steps * B / float(e2e_s.item()), "unit": UNIT,
           "h2d_bytes_per_step": info["h2d_bytes"] // args.steps, "d2h_bytes_per_step": info["d2h_bytes"] // args.steps,
           "ms_per_step": float(e2e_s.item()) / args.steps * 1e3,
           "h2d": ("ragged: only the valid rows of every zero-padded clip cross PCIe (seqpan_h2d_ragged), padding rows "
                   "are rewritten as zeros on the device" if ragged else "dense: the full zero-padded [B,L,vdim] tensor"),
           "dense_input_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host[0].values()))}

    # ---- sustained: the same two sweeps for >= 3 s each, with their own clock samples ---------------------------
    sustained = None
    if not args.no_sustained:
        n_res = max(args.steps, int(args.sustain_seconds * 1e3 / max(ms / args.steps, 1e-3)) + 1)
        n_e2e = max(args.steps, int(args.sustain_seconds / max(float(e2e_s.item()) / args.steps, 1e-6)) + 1)
        barrier()
        sampler2 = ClockSampler(smi_index) if rank == 0 else None
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        fork()
        for i in range(n_res):
            step(i)
        join()
        s1.record()
        barrier()
        sms = torch.tensor([s0.elapsed_time(s1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(sms, op=dist.ReduceOp.MAX)
        clocks_res = sampler2.stop() if sampler2 else None
        long_batches = [host[i % len(host)] for i in range(n_e2e)]
        barrier()
        sampler3 = ClockSampler(smi_index) if rank == 0 else None
        t0 = time.perf_counter()
        evaluate(model, long_batches, dev, streams=es, ragged_h2d=ragged, h2d_ctas=args.h2d_ctas)
        barrier()
        ss = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ss, op=dist.ReduceOp.MAX)
        clocks_e2e = sampler3.stop() if sampler3 else None
        sustained = {"device_resident": {"value": world * n_res * B / (float(sms.item()) / 1e3), "unit": UNIT, "steps": n_res,
                                         "seconds": float(sms.item()) / 1e3, "clocks": clocks_res},
                     "e2e": {"value": world * n_e2e * B / float(ss.item()), "unit": UNIT, "steps": n_e2e,
                             "seconds": float(ss.item()), "clocks": clocks_e2e}}

    # ---- per-kernel timing pass (CUDA events around every launch, on the launching stream) ---------------------
    peaks = load_peaks()
    roof, kernels, path_tflops = None, [], None
    if rank == 0 and not args.no_profile:
        model.use_context(0)
        model.set_profile(True)
        psteps = min(args.steps, 10)
        for i in range(psteps):
            step(i, 0)
        summ = model.profile_summary()
        model.set_profile(False)
        total = sum(v[1] for v in summ.values())
        work = step_work(B, L, T, C, w.vdim)
        traffic = {}
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                traffic = json.load(f).get(w.name, {})
        except Exception:
            pass
        for k, (n, t) in sorted(summ.items(), key=lambda kv: -kv[1][1]):
            tag = k if k in work else ("launch_" + k if "launch_" + k in work else k)
            ent = {"kernel": k, "launches_per_step": n / psteps, "ms_per_step": t / psteps, "share": t / total}
            if tag in work:
                r = roofline_of(k, n / psteps, t / psteps, work[tag], peaks, t / total, traffic.get(k))
                ent["roofline"] = {kk: r[kk] for kk in ("bound", "achieved", "peak", "unit", "frac", "traffic", "tensor_frac", "hbm_frac_dram")}
                if roof is None:
                    roof = r
            kernels.append(ent)
        path_tflops = value / world * synth.flops_per_batch(B, L, T, C, w.vdim) / B / 1e12     # per GPU

    # ---- CPU baseline beside it (rank 0, N=1 only) -----------------------------------------------------------------
    cpu = parity = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import seqpan_oracle as O
        torch.set_num_threads(os.cpu_count() or 1)
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        hb = [{k: v.clone() for k, v in b.items()} for b in host[:2]]     # unpinned copies
        for b in hb:       # the oracle (like the reference) takes one clip per pair
            if "video_index" in b:
                b["vfeats"] = b["vfeats"][b.pop("video_index").long()]
        g = synth.gumbel_noise(B, L)

        def one(b, keep=False):
            with torch.no_grad():
                o = O.forward(sd, b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], g)
                fr = O.infer_basic(o["slogits"], o["elogits"], b["vmasks"])
                return (o, fr) if keep else fr
        want, want_fr = one(hb[0], keep=True)
        # parity of the timed configuration on one of the timed batches: same weights, same injected Gumbel noise
        from oracle.parity import parity_stats, summary
        from vmrframe_b200 import infer_basic
        model.use_context(0)
        rb = resident[0]
        got = model(rb["words_ids"], rb["char_ids"], rb["vfeats"], rb["vmasks"], rb["tmasks"], gumbel=g.to(dev),
                    video_index=rb.get("video_index"))
        pstats = parity_stats(got, want, hb[0]["vmasks"], infer_basic(got["slogits"], got["elogits"], got["vmask"]), want_fr)
        parity = summary(pstats, args.precision, {"bf16": 1e-2, "tf32": 2e-3, "fp32": 1e-4}[args.precision])
        parity["tie_ladder"] = pstats["tie"]
        parity["batch"] = f"resident batch 0 of the {w.name} workload, default-init weights (the timed model), oracle on CPU fp32"
        t0 = time.perf_counter(); one(hb[1]); t1 = time.perf_counter() - t0
        n = int(max(3, min(30, 20.0 / max(t1, 1e-3))))
        t0 = time.perf_counter()
        for i in range(n):
            one(hb[i % 2])
        dt = time.perf_counter() - t0
        cores = torch.get_num_threads()
        cpu = {"value": n * B / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n} batches of the same {w.name} shape (B={B}, L={L}), oracle port of the reference, fp32 torch CPU, "
                         f"{cores} threads, {dt:.1f} s"}
        if not args.no_eager_baseline:
            sys.path.insert(0, os.path.join(ROOT, "profiles"))
            from eager_gpu import eager_gpu_baseline
            try:
                eager = eager_gpu_baseline(sd, hb, g, dev, n_batches=20)
            except Exception as ex:     # e.g. out of memory on a shape the eager path cannot hold
                eager = {"error": repr(ex)[:200]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "warmup_steps_run": n_warm,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"bf16": "bf16", "tf32": "tf32", "fp32": "f32"}[args.precision], "data": "synthetic",
                "config": {"workload": workload_string(w), "batch_T": T,
                           "global_batch": world * B, "streams": len(lanes), "shared_video": bool(args.shared_video),
                           "model": args.model, "numa_node": numa_node,
                           "parallelism": f"batch-sharded x{world}, no forward collective, "
                           "1 all-reduce of 5 IoU counters per sweep",
                           "cache": f"{args.resident} distinct resident batches/GPU cycled ({args.resident * B * L * w.vdim * 4 / 1e6:.0f} MB > 126 MB L2)",
                           "weights": "PyTorch default init, torch.manual_seed(0); GloVe-shaped N(0,0.4^2) table",
                           "timing": "CUDA events on the launching stream, barrier+synchronize both sides, max over ranks; "
                                     "module runs with sync_timing=False (the reference's two host syncs per forward are a host artefact)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": timed_launches, "host_enqueue_ms_per_step": host_enqueue_ms,
                "roofline": roof, "cpu_baseline": cpu, "parity": parity, "gpu_eager_baseline": eager, "sustained": sustained,
                "kernels": kernels[:10] if kernels else None,
                "path_tflops": path_tflops if kernels else None,
                "path_frac_of_tensor_peak": (path_tflops / peaks["tc_sustained"]) if kernels else None,
                "metrics_check": {"r1i3": metrics[0], "r1i5": metrics[1], "r1i7": metrics[3], "miou": metrics[4]}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
