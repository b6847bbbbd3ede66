"""Evaluation engine around the hot path: metrics, the pipelined eval sweep and batch sharding across GPUs.

Mirrors (reference file:line):
  * ``append_ious`` / ``get_i345_mi``            models/loss.py:83-90, 103-109
  * ``calculate_iou`` / ``calculate_iou_accuracy`` utils/utils.py:161-167, 179-185
  * the eval loop of ``main.py:112-134,138-153``  (forward -> infer -> IoU -> R1@{0.3,0.5,0.7}, mIoU)
  * ``lossfun_loc`` / ``lossfun_match``          models/loss.py:24-54 (value only; used by train_engine_SeqPAN)

Multi-GPU (SURVEY.md §8e): the unit of independent work is the reference BATCH (the predictor attends across
the samples of a batch, SURVEY.md §0 #8), so whole batches are dealt round-robin to ranks, weights are
replicated, there is no collective in the forward, and one all-reduce(sum) of the 5 IoU counters
``[n, sum IoU, #>=0.3, #>=0.5, #>=0.7]`` (fp64, 40 bytes) reproduces ``get_i345_mi`` over the whole sweep.
"""
from __future__ import annotations

import operator
import time

import numpy as np
import torch

from . import _cabi
from .seqpan import infer_basic_device


# ---- metrics (host, reference semantics) ---------------------------------------------------------------
def calculate_iou(i0, i1):
    union = (min(i0[0], i1[0]), max(i0[1], i1[1]))
    inter = (max(i0[0], i1[0]), min(i0[1], i1[1]))
    if (union[1] - union[0]) == 0.0:
        return 0.0
    return max(0.0, 1.0 * (inter[1] - inter[0]) / (union[1] - union[0]))


def calculate_iou_accuracy(ious, threshold):
    return float(sum(1 for i in ious if i >= threshold)) / float(len(ious)) * 100.0


def append_ious(ious, se_gts, se_props):
    for gt, prop in zip(se_gts, se_props):
        ious.append(calculate_iou(gt, prop))
    return ious


def get_i345_mi(ious):
    # the reference returns r1i5 twice (models/loss.py:109)
    r3, r5, r7 = (calculate_iou_accuracy(ious, t) for t in (0.3, 0.5, 0.7))
    return r3, r5, r5, r7, float(np.mean(ious) * 100.0)


def metrics_from_counters(counters):
    """``get_i345_mi`` from the summable counters ``[n, sum IoU, #>=0.3, #>=0.5, #>=0.7]``."""
    c = [float(x) for x in counters]
    n = max(c[0], 1.0)
    return c[2] / n * 100.0, c[3] / n * 100.0, c[3] / n * 100.0, c[4] / n * 100.0, c[1] / n * 100.0


class IouCounters:
    """Device-side IoU counters (seqpan_iou_counters): no host loop, no sync until ``.result()``.  ``exact=True``
    (seqpan_iou_counters_exact, DESIGN.md section 13) adds each IoU rounded to a multiple of 2^-28, so the sum is the same
    bits in any order of samples, calls, streams and ranks (up to 2^25 samples in all)."""

    def __init__(self, device, exact: bool = False):
        self.exact = bool(exact)
        self.buf = torch.zeros(5, dtype=torch.float64, device=device)

    def update(self, fracs: torch.Tensor, gt_fracs: torch.Tensor):
        dev = self.buf.device
        fr = fracs.to(device=dev, dtype=torch.float32).contiguous()
        gt = gt_fracs.to(device=dev, dtype=torch.float32).contiguous()
        fn = _cabi.lib().seqpan_iou_counters_exact if self.exact else _cabi.lib().seqpan_iou_counters
        with torch.cuda.device(dev):
            _cabi.check(fn(fr.data_ptr(), gt.data_ptr(), fr.shape[0], self.buf.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))

    def allreduce(self):
        """Sum over ranks: the only collective of the sharded sweep (NCCL on GPUs)."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.buf, op=dist.ReduceOp.SUM)
        return self

    def result(self):
        return metrics_from_counters(self.buf.cpu().tolist())


# ---- top-k retrieval metrics (R@k after temporal NMS) -------------------------------------------------------
TOPK_THRESHOLDS = (0.3, 0.5, 0.7)


def append_ious_topk(ious, se_gts, se_props):
    """R@k analogue of ``append_ious``: for each sample, the best ``calculate_iou`` over its filled top-k proposals
    (``se_props`` ``[B,k,2]`` as returned by ``infer_topk``; empty slots have a negative start) against its ground truth,
    0 when no slot is filled."""
    for gt, props in zip(se_gts, se_props):
        ious.append(max((calculate_iou(gt, p) for p in props if p[0] >= 0), default=0.0))
    return ious


def recall_at_k(ious):
    """``(R@k IoU>=0.3, >=0.5, >=0.7)`` in percent from the per-sample best IoUs of :func:`append_ious_topk`."""
    return tuple(calculate_iou_accuracy(ious, t) for t in TOPK_THRESHOLDS)


def metrics_topk_from_counters(counters):
    """:func:`recall_at_k` from the summable counters ``[n, #>=0.3, #>=0.5, #>=0.7]``."""
    c = [float(x) for x in counters]
    n = max(c[0], 1.0)
    return tuple(x / n * 100.0 for x in c[1:4])


def _allreduce_sum(t: torch.Tensor) -> torch.Tensor:
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


class TopkCounters:
    """Device-side R@k counters (seqpan_topk_counters) of top-``k`` spans retrieved with NMS threshold ``nms_thresh``:
    ``[n, #>=0.3, #>=0.5, #>=0.7]`` in fp64, no sync until ``.result()``.  ``buf`` may be a caller's 4-element fp64 view."""

    def __init__(self, device, k: int, nms_thresh: float = 0.5, buf: torch.Tensor | None = None):
        self.k, self.nms_thresh = int(k), float(nms_thresh)
        self.buf = torch.zeros(4, dtype=torch.float64, device=device) if buf is None else buf

    def update(self, fracs: torch.Tensor, gt_fracs: torch.Tensor):
        """``fracs`` ``[B,k,2]`` from :func:`infer_topk` / the top-k kernel, ``gt_fracs`` ``[B,2]``."""
        dev = self.buf.device
        fr = fracs.to(device=dev, dtype=torch.float32).contiguous()
        gt = gt_fracs.to(device=dev, dtype=torch.float32).contiguous()
        if fr.dim() != 3 or fr.shape[1] != self.k or fr.shape[2] != 2 or gt.shape != (fr.shape[0], 2):
            raise ValueError(f"fracs must be [B,{self.k},2] and gt_fracs [B,2], got {tuple(fr.shape)} and {tuple(gt.shape)}")
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib().seqpan_topk_counters(fr.data_ptr(), gt.data_ptr(), fr.shape[0], self.k,
                                                         self.buf.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))

    def allreduce(self):
        _allreduce_sum(self.buf)
        return self

    def result(self):
        return metrics_topk_from_counters(self.buf.cpu().tolist())


# ---- sharding ---------------------------------------------------------------------------------------------
def shard_batches(num_batches: int, rank: int, world_size: int) -> list[int]:
    """Whole reference batches, round-robin: batch k -> rank k mod world_size."""
    return list(range(rank, num_batches, world_size))


def draw_chunks(store, num_batches: int, world_size: int, chunk: int = 32, key: str = "sweep_next"):
    """Work queue over WHOLE reference batches for ranks that are fed unevenly (DESIGN.md section 7).

    Yields ``range(lo, hi)`` of batch ids this rank owns next.  ``store`` is anything with the atomic ``add(key, n) -> new value``
    of ``torch.distributed.TCPStore``; every rank iterates its own generator against the same store and key.  Guided
    self-scheduling: a draw takes ``left / (2 * world_size)`` batches, clamped to ``[8, 2 * chunk]`` -- large while much is left
    (the caller drains its pipeline between draws), small at the end (the last draw of the slowest rank is the imbalance).
    Every id in ``[0, num_batches)`` is yielded exactly once over all ranks; a batch is never split (SURVEY.md section 8e).
    """
    chunk = max(8, int(chunk))
    while True:
        left = num_batches - store.add(key, 0)
        if left <= 0:
            return
        c = int(min(2 * chunk, max(8, left // (2 * world_size))))
        hi = store.add(key, c)              # atomic fetch-and-add: this rank owns batches [hi - c, hi)
        lo = hi - c
        if lo >= num_batches:
            return
        yield range(lo, min(hi, num_batches))


def allreduce_counters_cpu(counters: torch.Tensor) -> torch.Tensor:
    """gloo-side equivalent of :meth:`IouCounters.allreduce` for host tests."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    return counters


# ---- seeded sweeps (DESIGN.md section 13) ----------------------------------------------------------------------
EXACT_MAX_SAMPLES = 1 << 25   # the exact IoU sums stay exact up to this many samples


def _check_seed(seed) -> int:
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)):
        raise ValueError(f"seed must be an int in [0, 2^64), got {seed!r}")
    if not 0 <= int(seed) < 1 << 64:
        raise ValueError(f"seed={seed} outside [0, 2^64)")
    return int(seed)


def _check_batch_id(i) -> int:
    try:
        if isinstance(i, bool):
            raise TypeError
        i = operator.index(i)
    except TypeError:
        raise ValueError(f"batch ids must be integers, got {i!r}") from None
    if not 0 <= i < 1 << 32:
        raise ValueError(f"batch id {i} outside [0, 2^32)")
    return i


def _resolve_device(device) -> torch.device:
    device = torch.device(device or "cuda")
    if device.index is None:     # "cuda" = the current device; the handles and the parameters compare full device names
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def _sweep_ids(batches, seed, batch_ids):
    """``(seed, one id per batch)`` of a seeded sweep after the argument checks of :func:`evaluate`; ``(None, None)`` without
    a seed."""
    if seed is None:
        if batch_ids is not None:
            raise ValueError("batch_ids name the noise of a seeded sweep: pass seed= too")
        return None, None
    seed = _check_seed(seed)
    ids = list(range(len(batches))) if batch_ids is None else [_check_batch_id(i) for i in batch_ids]
    if len(ids) != len(batches):
        raise ValueError(f"{len(ids)} batch ids for {len(batches)} batches")
    if len(set(ids)) != len(ids):
        raise ValueError("duplicate batch ids: two batches would get the same noise")
    n = sum(int(b["vmasks"].shape[0]) for b in batches)
    if n > EXACT_MAX_SAMPLES:
        raise ValueError(f"{n} samples in one seeded call: the exact IoU sum holds up to 2^25")
    return seed, ids


def gumbel_noise(B: int, L: int, seed: int, batch_id: int, device=None) -> torch.Tensor:
    """The Gumbel noise ``[B, L, 4]`` fp32 that ``evaluate(seed=seed)`` uses for the batch with id ``batch_id``
    (seqpan_gumbel_noise, DESIGN.md section 13): a function of ``(seed, batch_id, B, L)`` alone.  Pass it as
    ``forward(..., gumbel=)`` to reproduce one batch of a seeded sweep.  ``device`` defaults to the current CUDA device."""
    seed, batch_id = _check_seed(seed), _check_batch_id(batch_id)
    B, L = int(B), int(L)
    if B < 0:
        raise ValueError(f"B={B} < 0")
    _cabi.require_device()
    device = _resolve_device(device)
    out = torch.empty(B, L, 4, dtype=torch.float32, device=device)
    if B == 0:
        return out
    with torch.cuda.device(device):
        _cabi.check(_cabi.lib().seqpan_gumbel_noise(seed, batch_id, B, L, out.data_ptr(),
                                                    torch.cuda.current_stream(device).cuda_stream))
    return out


# ---- pipelined evaluation sweep (the public e2e call) -----------------------------------------------------
_INPUT_KEYS = ("words_ids", "char_ids", "vfeats", "vmasks", "tmasks", "se_fracs")


def valid_rows_from_mask(vmask: torch.Tensor) -> torch.Tensor:
    """Rows of each zero-padded clip that carry data: index of the last non-zero mask entry + 1 (int32 [B])."""
    L = vmask.shape[1]
    pos = torch.arange(1, L + 1, dtype=torch.float32)
    return ((vmask != 0).to(torch.float32) * pos).amax(dim=1).to(torch.int32)


class _Slot:
    """Device-side landing buffers of one in-flight batch (inputs, noise, outputs): allocated once per sweep."""

    def __init__(self, device, B, L, V, T, C, topk=0):
        f32, i64 = torch.float32, torch.int64
        self.words = torch.empty(B * T, dtype=i64, device=device)
        self.chars = torch.empty(B * T * C, dtype=i64, device=device)
        self.vfeats = torch.empty(B * L * V, dtype=f32, device=device)
        self.vmask = torch.empty(B * L, dtype=f32, device=device)
        self.tmask = torch.empty(B * T, dtype=f32, device=device)
        self.gt = torch.empty(B * 2, dtype=f32, device=device)
        self.gumbel = torch.empty(B * L * 4, dtype=f32, device=device)
        self.slogits = torch.empty(B * L, dtype=f32, device=device)
        self.elogits = torch.empty(B * L, dtype=f32, device=device)
        self.match = torch.empty(B * L * 4, dtype=f32, device=device)
        self.fracs = torch.empty(B * 2, dtype=f32, device=device)
        self.valid_dev = torch.empty(B, dtype=torch.int32, device=device)
        self.vindex = torch.empty(B, dtype=torch.int32, device=device)
        if topk:
            self.topk_si = torch.empty(B * topk, dtype=i64, device=device)
            self.topk_ei = torch.empty(B * topk, dtype=i64, device=device)
            self.topk_scores = torch.empty(B * topk, dtype=f32, device=device)
            self.topk_fracs = torch.empty(B * topk * 2, dtype=f32, device=device)
        self.copied = torch.cuda.Event()      # recorded on the copy stream when the inputs have landed
        self.consumed = torch.cuda.Event()    # recorded on the compute lane when the batch is done with the slot
        self.used = False


def evaluate(model, host_batches, device=None, depth: int = 2, return_fracs: bool = False, streams: int = 2,
             ragged_h2d: bool = True, h2d_ctas: int = 32, profile: bool = False, check_padding: bool | None = None,
             allreduce: bool = True, topk: int | None = None, nms_thresh: float = 0.5, video_encodings=None,
             seed: int | None = None, batch_ids=None):
    """Runs forward + span decode + IoU counters over an iterable of HOST batches (dicts in ``BaseCollate``'s key
    naming, ideally pinned) -- the eval loop of ``main.py:112-134`` as one pipelined call.

    Every batch is copied host->device inside this call on a copy stream into a static ring of ``depth + streams``
    device slots (no allocation per batch), ``depth`` batches ahead of compute; the span fractions are read back
    device->host per batch.  ``streams`` > 1 runs consecutive batches on different CUDA streams (one kernel context
    each, see ``SeqPAN.use_context``) so that tail waves and latency-bound phases of one batch's kernels are filled by
    the next batch's; batches stay whole, so results equal the single-stream sweep.  With ``ragged_h2d`` only the valid
    rows of every zero-padded clip cross PCIe (``seqpan_h2d_ragged``; the padding rows are zeros by ``BaseCollate``'s
    contract, ``utils/BaseDataset.py:209``, and are rewritten as zeros on the device); ``h2d_ctas`` >= 1 does that
    with one zero-copy kernel of that many CTAs reading the pinned buffer, 0 with one DMA copy per sample.
    A batch may carry ``video_index`` (int32 ``[B]``): its ``vfeats`` then hold every clip once (``[U,L,V]``, dense-query
    datasets; SURVEY.md section 8 row f1), only the U clips cross PCIe and the video branch runs once per clip.
    ``check_padding`` (default: the ``SEQPAN_CHECK_PADDING=1`` environment switch) verifies on the host, before a ragged
    copy, that the rows it skips really are zero -- a caller that violates the collate contract would otherwise silently
    lose the reference's padding leak (SURVEY.md section 0 #11); it costs one pass over the host tensor per batch.
    ``allreduce=False`` leaves the counters rank-local (a caller that evaluates several chunks sums them and all-reduces once).
    Returns ``(metrics 5-tuple, counters tensor, info dict)``; with ``return_fracs`` the info holds all ``(B,2)``
    fractions.
    ``topk=k`` additionally retrieves the k best spans of every sample after temporal NMS at ``nms_thresh`` (the kernel of
    :func:`extract_topk`) on the batch's lane and accumulates R@k counters; ``info["topk"]`` then holds ``k``, ``nms_thresh``,
    ``recall`` (R@k at IoU 0.3, 0.5, 0.7, percent) and ``counters`` (``[n, #>=0.3, #>=0.5, #>=0.7]``), and with
    ``return_fracs`` ``info["topk_fracs"]`` holds all ``(B,k,2)`` fractions.  Both counter sets live in one fp64 buffer, so
    the sweep still ends in a single all-reduce.
    ``video_encodings`` (from ``model.encode_videos``, on ``device``; DESIGN.md section 12): the batches carry no ``vfeats``,
    their ``video_index`` names clips of the encodings (without it, pair b reads clip b), and no video byte crosses PCIe --
    ``info["h2d_bytes"]`` counts ids, masks, ground truth and indices only.  Results equal the sweep over the raw clips with the
    same ``video_index``.  Under ``torchrun`` every rank encodes the clips its batches use onto its own device (encodings are
    device memory and are not shared between ranks).
    ``seed`` (an int in ``[0, 2^64)``; DESIGN.md section 13) makes the sweep reproducible: batch ``i`` gets the Gumbel noise
    :func:`gumbel_noise` ``(B, L, seed, batch_ids[i])`` instead of a draw from torch's generator, and the IoU counters add
    exactly (``IouCounters(exact=True)``), so counters, metrics and spans are the same bits however the batches are split
    over streams, calls, ranks and work-queue schedules.  ``batch_ids`` (default ``range(len(batches))``) are the batches'
    global ids: a caller that shards passes ``shard_batches(...)`` or the ranges ``draw_chunks`` yields.  Ids must be distinct
    and in ``[0, 2^32)``, and one call (and, after the all-reduce, the whole sweep) holds at most 2^25 samples.
    ``info["seed"]`` records the seed.  Without a seed the sweep makes exactly the calls it always made.
    """
    batches = list(host_batches)
    seed, batch_ids = _sweep_ids(batches, seed, batch_ids)
    _cabi.require_device()
    if topk is not None:
        topk = int(topk)
        if not (1 <= topk <= 32 and 0.0 < nms_thresh <= 1.0):
            raise ValueError(f"topk={topk} must be in [1,32] and nms_thresh={nms_thresh} in (0,1]")
    device = _resolve_device(device)
    L_ = _cabi.lib()
    import os
    if check_padding is None:
        check_padding = os.environ.get("SEQPAN_CHECK_PADDING") == "1"
    enc = video_encodings
    if enc is not None:
        model._check_encoded_call(enc, None, None)
        if enc.device != device:
            raise _cabi.SeqpanError(f"the encodings live on {enc.device}, the sweep runs on {device}: encode on every rank's device")
        for i, b in enumerate(batches):
            B = b["vmasks"].shape[0]
            if "vfeats" in b:
                raise _cabi.SeqpanError(f"batch {i} carries vfeats: with video_encodings the clips come from the encodings")
            if "video_index" in b:
                idx = b["video_index"]
                if idx.shape != (B,) or (B and (int(idx.min()) < 0 or int(idx.max()) >= len(enc))):
                    raise _cabi.SeqpanError(f"batch {i}: video_index must be [{B}] with values in [0,{len(enc)})")
            elif B > len(enc):
                raise _cabi.SeqpanError(f"batch {i} has no video_index and {B} pairs > {len(enc)} encoded clips")
    main = torch.cuda.current_stream(device)
    nstreams = max(1, int(streams))
    counters = IouCounters(device, exact=seed is not None)
    iou_counters = L_.seqpan_iou_counters_exact if counters.exact else L_.seqpan_iou_counters
    tk = None
    if topk is not None:   # one fp64 buffer [5 IoU counters | 4 R@k counters]: one all-reduce for both
        joint = torch.zeros(9, dtype=torch.float64, device=device)
        counters.buf = joint[:5]
        tk = TopkCounters(device, topk, nms_thresh, buf=joint[5:])

    def topk_info():
        return {"k": tk.k, "nms_thresh": tk.nms_thresh, "recall": tk.result(), "counters": tk.buf}

    if not batches:
        info = {"h2d_bytes": 0, "d2h_bytes": 0, "wall_s": 0.0, "batches": 0}
        if tk is not None:
            info["topk"] = topk_info()
        if seed is not None:
            info["seed"] = seed
        return counters.result(), counters.buf, info
    lanes = [main] + [torch.cuda.Stream(device) for _ in range(nstreams - 1)]
    copy_stream = torch.cuda.Stream(device)
    depth = max(1, int(depth))
    Bm = max(b["vmasks"].shape[0] for b in batches)
    Tm = max(b["words_ids"].shape[1] for b in batches)
    Cm = max(b["char_ids"].shape[2] for b in batches)
    Lv, V = (batches[0]["vfeats"].shape[1], batches[0]["vfeats"].shape[2]) if enc is None else (enc.rows.shape[1], 0)
    was_sync, was_ctx, was_side = model.sync_timing, model._ctx_key, getattr(model, "_side_stream", True)
    if hasattr(model, "set_side_stream"):
        model.set_side_stream(False)      # the sweep is bound by its own host->device copy kernel (include/seqpan_b200.h)
    with torch.cuda.device(device):
        slots = [_Slot(device, Bm, Lv, V, Tm, Cm, topk or 0) for _ in range(min(depth + nstreams, len(batches)))]
        # every kernel context is sized for the largest batch of the sweep up front (no handle re-creation / weight
        # re-packing in the middle of it)
        for k in range(nstreams):
            model.use_context(k)._ensure_handle(device, Bm, Tm, Cm)
            if enc is not None:
                model._check_encoding_weights(enc)
        model.use_context(was_ctx)
        # the slots and contexts were allocated / packed on the caller's stream: the copy stream and the lanes start after it
        ready = torch.cuda.Event()
        ready.record(main)
        copy_stream.wait_event(ready)
    host_fracs = torch.empty(len(batches), Bm, 2, dtype=torch.float32, pin_memory=True)
    valid_host = torch.empty(len(batches), Bm, dtype=torch.int32, pin_memory=True)   # one row per batch: never rewritten
    host_topk = torch.empty(len(batches), Bm, topk, 2, dtype=torch.float32, pin_memory=True) if tk is not None and return_fracs else None
    h2d = d2h = 0
    views = {}
    prof = []   # profile=True: (copy start, copy end, compute start, compute end) events per batch
    ev_t = lambda: torch.cuda.Event(enable_timing=True)

    def issue(i):
        """Host -> device copy of batch i into slot i % len(slots) on the copy stream."""
        nonlocal h2d
        b, sl = batches[i], slots[i % len(slots)]
        B, T, Cc = b["words_ids"].shape[0], b["words_ids"].shape[1], b["char_ids"].shape[2]
        U = b["vfeats"].shape[0] if enc is None else 0   # == B unless the batch shares clips through video_index
        v = {"words": sl.words[: B * T].view(B, T), "chars": sl.chars[: B * T * Cc].view(B, T, Cc),
             "vfeats": sl.vfeats[: U * Lv * V].view(U, Lv, V), "vmask": sl.vmask[: B * Lv].view(B, Lv),
             "vindex": sl.vindex[:B] if "video_index" in b else None,
             "tmask": sl.tmask[: B * T].view(B, T), "gt": sl.gt[: B * 2].view(B, 2) if "se_fracs" in b else None,
             "gumbel": sl.gumbel[: B * Lv * 4].view(B, Lv, 4), "slogits": sl.slogits[: B * Lv].view(B, Lv),
             "elogits": sl.elogits[: B * Lv].view(B, Lv), "match": sl.match[: B * Lv * 4].view(B, Lv, 4),
             "fracs": sl.fracs[: B * 2].view(B, 2)}
        if tk is not None:
            v.update(topk_si=sl.topk_si[: B * topk], topk_ei=sl.topk_ei[: B * topk], topk_scores=sl.topk_scores[: B * topk],
                     topk_fracs=sl.topk_fracs[: B * topk * 2].view(B, topk, 2))
        views[i] = v
        with torch.cuda.stream(copy_stream):
            if sl.used:
                copy_stream.wait_event(sl.consumed)       # the lane that last computed out of this slot is done
            if profile:
                prof.append([ev_t(), ev_t(), ev_t(), ev_t()])
                prof[i][0].record(copy_stream)
            v["words"].copy_(b["words_ids"], non_blocking=True)
            v["chars"].copy_(b["char_ids"], non_blocking=True)
            v["vmask"].copy_(b["vmasks"], non_blocking=True)
            v["tmask"].copy_(b["tmasks"], non_blocking=True)
            h2d += (b["words_ids"].numel() + b["char_ids"].numel()) * 8 + (b["vmasks"].numel() + b["tmasks"].numel()) * 4
            if v["gt"] is not None:
                v["gt"].copy_(b["se_fracs"], non_blocking=True)
                h2d += b["se_fracs"].numel() * 4
            vf = b.get("vfeats")
            if v["vindex"] is not None:
                v["vindex"].copy_(b["video_index"].to(torch.int32), non_blocking=True)
                h2d += B * 4
            if enc is not None:
                pass                                      # the clips are resident as encodings
            elif (ragged_h2d and v["vindex"] is None and vf.is_pinned() and vf.dtype == torch.float32 and vf.is_contiguous()
                    and V % 4 == 0):
                valid_host[i, :B].copy_(valid_rows_from_mask(b["vmasks"]))
                if check_padding:
                    rows = torch.arange(Lv).unsqueeze(0) >= valid_host[i, :B].unsqueeze(1).long()
                    if bool((vf[rows] != 0).any()):
                        raise _cabi.SeqpanError(f"batch {i}: non-zero clip rows behind the last valid mask position; the ragged "
                                                f"host->device copy would drop them (pass ragged_h2d=False)")
                _cabi.check(L_.seqpan_h2d_ragged(v["vfeats"].data_ptr(), vf.data_ptr(), valid_host[i].data_ptr(),
                                                 sl.valid_dev.data_ptr(), B, Lv, V, int(h2d_ctas), copy_stream.cuda_stream))
                h2d += int(valid_host[i, :B].sum()) * V * 4 + B * 4
            else:
                v["vfeats"].copy_(vf, non_blocking=True)
                h2d += vf.numel() * 4
            sl.copied.record(copy_stream)
            if profile:
                prof[i][1].record(copy_stream)
            sl.used = True

    model.sync_timing = False
    try:
        with torch.cuda.device(device):
            for i in range(min(depth, len(batches))):
                issue(i)
            start_ev = torch.cuda.Event()
            start_ev.record(main)
            for ln in lanes[1:]:
                ln.wait_event(start_ev)
            t0 = time.time()
            for i in range(len(batches)):
                sl, v = slots[i % len(slots)], views.pop(i)
                lane = lanes[i % nstreams]
                with torch.cuda.stream(lane):
                    lane.wait_event(sl.copied)
                    if profile:
                        prof[i][2].record(lane)
                    model.use_context(i % nstreams)
                    B = v["vmask"].shape[0]
                    st = lane.cuda_stream
                    if seed is None:
                        # == F.gumbel_softmax's draw (models/SeqPAN.py:79): -empty_like(logits).exponential_().log()
                        v["gumbel"].exponential_().log_().neg_()
                    else:
                        _cabi.check(L_.seqpan_gumbel_noise(seed, batch_ids[i], B, Lv, v["gumbel"].data_ptr(), st))
                    model.forward_into(v["words"], v["chars"], v["vfeats"], v["vmask"], v["tmask"], v["gumbel"],
                                       v["slogits"], v["elogits"], v["match"], v["vindex"], video_encodings=enc)
                    _cabi.check(L_.seqpan_span_decode(v["slogits"].data_ptr(), v["elogits"].data_ptr(), v["vmask"].data_ptr(),
                                                      B, Lv, None, None, v["fracs"].data_ptr(), st))
                    if v["gt"] is not None:
                        _cabi.check(iou_counters(v["fracs"].data_ptr(), v["gt"].data_ptr(), B, counters.buf.data_ptr(), st))
                    host_fracs[i, :B].copy_(v["fracs"], non_blocking=True)     # device -> host read of the step's result
                    d2h += B * 2 * 4
                    if tk is not None:
                        _cabi.check(L_.seqpan_span_topk(v["slogits"].data_ptr(), v["elogits"].data_ptr(), v["vmask"].data_ptr(),
                                                        B, Lv, topk, tk.nms_thresh, v["topk_si"].data_ptr(),
                                                        v["topk_ei"].data_ptr(), v["topk_scores"].data_ptr(),
                                                        v["topk_fracs"].data_ptr(), st))
                        if v["gt"] is not None:
                            _cabi.check(L_.seqpan_topk_counters(v["topk_fracs"].data_ptr(), v["gt"].data_ptr(), B, topk,
                                                                tk.buf.data_ptr(), st))
                        if host_topk is not None:
                            host_topk[i, :B].copy_(v["topk_fracs"], non_blocking=True)
                            d2h += B * topk * 2 * 4
                    sl.consumed.record(lane)
                    if profile:
                        prof[i][3].record(lane)
                if i + depth < len(batches):
                    issue(i + depth)
            for ln in lanes[1:]:       # the main stream (and the counters read below) waits for every lane
                e = torch.cuda.Event()
                e.record(ln)
                main.wait_event(e)
            if allreduce:
                if tk is None:
                    counters.allreduce()
                else:
                    _allreduce_sum(joint)
            metrics = counters.result()  # synchronises
            if seed is not None and allreduce and float(counters.buf[0]) > EXACT_MAX_SAMPLES:
                raise ValueError(f"{int(counters.buf[0])} samples over all ranks: the exact IoU sum holds up to 2^25")
    finally:
        model.use_context(was_ctx)
        model.sync_timing = was_sync
        if hasattr(model, "set_side_stream"):
            model.set_side_stream(was_side)
    info = {"h2d_bytes": h2d, "d2h_bytes": d2h + (40 if tk is None else 72), "wall_s": time.time() - t0,
            "batches": len(batches)}
    if tk is not None:
        info["topk"] = topk_info()
    if seed is not None:
        info["seed"] = seed
    if profile:
        info["copy_ms"] = [p[0].elapsed_time(p[1]) for p in prof]
        info["compute_ms"] = [p[2].elapsed_time(p[3]) for p in prof]
        info["copy_to_compute_start_ms"] = [prof[0][0].elapsed_time(p[2]) for p in prof]
    if return_fracs:  # counters.result() above synchronised the device, so the pinned buffer is complete
        info["fracs"] = [host_fracs[i, : b["vmasks"].shape[0]].numpy().copy() for i, b in enumerate(batches)]
        if host_topk is not None:
            info["topk_fracs"] = [host_topk[i, : b["vmasks"].shape[0]].numpy().copy() for i, b in enumerate(batches)]
    return metrics, counters.buf, info


# ---- training losses of the reference (values only) ---------------------------------------------------------
def lossfun_match(m_probs, label_embs, m_labels, vmask):
    # models/loss.py:24-41
    import torch.nn.functional as F
    onehot = F.one_hot(m_labels).float()
    per = -torch.sum(onehot * m_probs, dim=-1)
    loss = torch.sum(per * vmask) / (torch.sum(vmask) + 1e-12)
    ortho = torch.matmul(label_embs.T, label_embs) * (1.0 - torch.eye(4, device=label_embs.device))
    return loss + torch.norm(ortho, p=2)


def lossfun_loc(start_logits, end_logits, s_labels, e_labels, vmask):
    # models/loss.py:43-54 (cross entropy with soft [B,L] targets on UNMASKED logits)
    ce = torch.nn.CrossEntropyLoss(reduction="mean")
    return ce(start_logits, s_labels) + ce(end_logits, e_labels)
