"""CPU reference of top-k span retrieval with greedy temporal NMS (the definition in DESIGN.md section 11).

The reference repository has no top-k; this extends its ``infer_basic`` / ``extract_index`` (restated in
``oracle/seqpan_oracle.py``) and reduces to it at k = 1: torch fp32 probabilities on the ``infer_basic`` path, fp32 products
``sp[i] * ep[j]``, candidates ``i <= j`` with a positive score ordered by (score desc, i asc, j asc), and k greedy rounds that
each keep the best candidate no kept span removes.  Suppression is decided on the integer indices with one fp32 multiply
(``inter >= thr * union``), so it is exact and the kernel makes the same decision bit for bit.
"""
import numpy as np
import torch

from oracle import seqpan_oracle as O


def probabilities(start_logits, end_logits, vmask=None):
    """``softmax(mask_logits(.))`` as in ``infer_basic`` (no mask: ``extract_index``), fp32 numpy ``[B,L]`` each."""
    s, e = start_logits.float(), end_logits.float()
    if vmask is not None:
        s, e = O.mask_logits(s, vmask), O.mask_logits(e, vmask)
    return torch.softmax(s, dim=1).numpy(), torch.softmax(e, dim=1).numpy()


def suppressed(i, j, a, b, thr):
    """Whether candidates ``(i, j)`` (integer arrays) leave the set once ``(a, b)`` is kept."""
    uni = np.maximum(j, b) - np.minimum(i, a)
    inter = np.maximum(0, np.minimum(j, b) - np.maximum(i, a))
    return ((i == a) & (j == b)) | ((uni > 0) & (inter.astype(np.float32) >= np.float32(thr) * uni.astype(np.float32)))


def topk_one(sp, ep, k, thr):
    """One sample: (starts, ends, scores, margins) of length <= k in selection order.  ``margins[r]`` is the kept score over
    the best other candidate still in the set at round r (inf when there is none): how far round r is from a tie."""
    L = sp.shape[0]
    i, j = np.triu_indices(L)
    sc = sp[i].astype(np.float32) * ep[j].astype(np.float32)
    pos = sc > 0
    i, j, sc = i[pos], j[pos], sc[pos]
    order = np.lexsort((j, i, -sc))
    i, j, sc = i[order], j[order], sc[order]
    alive = np.ones(len(sc), dtype=bool)
    starts, ends, scores, margins = [], [], [], []
    for _ in range(k):
        idx = np.flatnonzero(alive)
        if len(idx) == 0:
            break
        p = idx[0]
        starts.append(int(i[p])); ends.append(int(j[p])); scores.append(float(sc[p]))
        margins.append(float(sc[p]) / float(sc[idx[1]]) if len(idx) > 1 else float("inf"))
        alive &= ~suppressed(i, j, i[p], j[p], thr)
    return starts, ends, scores, margins


def extract_topk(start_logits, end_logits, vmask=None, k=5, nms_thresh=0.5):
    """``(start_idx, end_idx, scores, margins)`` as numpy ``[B,k]`` (int64, int64, float32, float64); empty slots are
    ``-1, -1, 0`` with margin inf."""
    sp, ep = probabilities(start_logits, end_logits, vmask)
    B = sp.shape[0]
    si = np.full((B, k), -1, dtype=np.int64)
    ei = np.full((B, k), -1, dtype=np.int64)
    sc = np.zeros((B, k), dtype=np.float32)
    mg = np.full((B, k), np.inf)
    for b in range(B):
        s, e, v, m = topk_one(sp[b], ep[b], k, nms_thresh)
        n = len(s)
        si[b, :n], ei[b, :n], sc[b, :n], mg[b, :n] = s, e, v, m
    return si, ei, sc, mg


def fractions(si, ei, vmask, L):
    """Indices divided by ``vmask.sum(1)`` (``L`` without a mask) in fp32, ``-1`` for empty slots: ``[B,k,2]``."""
    n = vmask.float().sum(dim=1).numpy() if vmask is not None else np.full(si.shape[0], L, dtype=np.float32)
    n = n.astype(np.float32)[:, None]
    with np.errstate(divide="ignore", invalid="ignore"):        # a fully masked sample divides by 0, as in the reference
        fr = np.stack([si.astype(np.float32) / n, ei.astype(np.float32) / n], axis=-1).astype(np.float32)
    fr[si < 0] = -1.0
    return fr


def infer_topk(start_logits, end_logits, vmask, k=5, nms_thresh=0.5):
    """``infer_basic``'s top-k counterpart: ``(fracs [B,k,2] float32, margins [B,k])``."""
    si, ei, _, mg = extract_topk(start_logits, end_logits, vmask, k, nms_thresh)
    return fractions(si, ei, vmask, start_logits.shape[1]), mg
