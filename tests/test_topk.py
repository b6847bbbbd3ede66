"""Top-k span retrieval with greedy temporal NMS and R@k counters (DESIGN.md section 11).

CPU: the reference oracle (tests/topk_oracle.py) against the reference's ``extract_index`` / ``infer_basic`` at k = 1, against a
stable sort at thr = 1, NMS invariants by brute force, the host R@k mirrors, shard sums over gloo and the C ABI's argument
checks.  B200: the kernel against the existing decoder (device against device, no tolerance), against the oracle, on exact
ties, its counters, determinism and graph capture, and ``evaluate(topk=)``."""
import ctypes as C
import itertools
import os
import socket

import numpy as np
import pytest
import torch

import topk_oracle as TO
from conftest import golden_case
from oracle import seqpan_oracle as O
from vmrframe_b200 import _cabi, engine, synth

DEV = "cuda:0"
CASES = ["charades_small", "anet_small", "tacos_small", "edge_b1", "charades_full"]
THRESHOLDS = (0.3, 0.5, 0.7, 1.0)


def _golden_logits(name):
    _, _, batch, fx = golden_case(name)
    return torch.from_numpy(fx["slogits"]), torch.from_numpy(fx["elogits"]), batch["vmasks"], batch


def _random_logits(B, L, seed, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    s, e = torch.randn(B, L, generator=g) * scale, torch.randn(B, L, generator=g) * scale
    lens = torch.randint(max(1, L // 4), L + 1, (B,), generator=g)
    lens[0] = L
    m = (torch.arange(L).expand(B, L) < lens.unsqueeze(1)).float()
    return s, e, m


# ---- oracle (CPU) -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_oracle_top1_is_the_reference_decode(name):
    s, e, m, _ = _golden_logits(name)
    si, ei, sc, _ = TO.extract_topk(s, e, m, k=1, nms_thresh=0.5)
    wsi, wei = O.extract_index(O.mask_logits(s, m), O.mask_logits(e, m))
    assert np.array_equal(si[:, 0], wsi.numpy())
    sp, ep = TO.probabilities(s, e, m)
    outer = np.triu(sp[:, :, None] * ep[:, None, :])
    unique = (outer == outer.max(axis=(1, 2), keepdims=True)).sum(axis=(1, 2)) == 1
    assert np.array_equal(ei[unique, 0], wei.numpy()[unique])
    fr, _ = TO.infer_topk(s, e, m, k=1)
    assert np.array_equal(fr[unique, 0], O.infer_basic(s, e, m)[unique].astype(np.float32))


@pytest.mark.parametrize("L", [1, 5, 12, 40])
def test_oracle_without_suppression_is_a_stable_sort(L):
    s, e, m = _random_logits(6, L, 100 + L)
    s[1] = 0.0; e[1] = 0.0           # every span ties: (i, j) order
    k = min(32, L * (L + 1) // 2)
    si, ei, sc, _ = TO.extract_topk(s, e, m, k=k, nms_thresh=1.0)
    sp, ep = TO.probabilities(s, e, m)
    for b in range(6):
        outer = sp[b][:, None] * ep[b][None, :]
        flat = [(float(outer[i, j]), i, j) for i in range(L) for j in range(L) if j >= i and outer[i, j] > 0]
        want = sorted(flat, key=lambda t: -t[0])[:k]          # stable: ties keep row-major (i, j) order
        n = len(want)
        assert [(int(a), int(c)) for a, c in zip(si[b, :n], ei[b, :n])] == [(i, j) for _, i, j in want]
        assert np.array_equal(sc[b, :n], np.float32([v for v, _, _ in want]))
        assert np.all(si[b, n:] == -1) and np.all(sc[b, n:] == 0)


def _removed(c, kept, thr):
    (i, j), (a, b) = c, kept
    if (i, j) == (a, b):
        return True
    uni, inter = max(j, b) - min(i, a), max(0, min(j, b) - max(i, a))
    return uni > 0 and np.float32(inter) >= np.float32(thr) * np.float32(uni)


def _hand_built(L):
    yield torch.zeros(1, L), torch.zeros(1, L)                                        # every span ties
    v = torch.tensor([0.0, 3.0])[torch.arange(L) % 2]
    yield v.unsqueeze(0), (0.7 * (torch.arange(L) % 3 == 0)).float().unsqueeze(0)    # duplicated values
    yield torch.linspace(-2, 2, L).unsqueeze(0), torch.linspace(2, -2, L).unsqueeze(0)


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_oracle_nms_invariants(thr):
    g = torch.Generator().manual_seed(int(thr * 10))
    for L in range(1, 13):
        inputs = [(torch.randn(1, L, generator=g) * 2, torch.randn(1, L, generator=g) * 2) for _ in range(3)]
        for s, e in inputs + list(_hand_built(L)):
            m = torch.ones(1, L)
            m[0, L - L // 4:] = 0
            sp, ep = TO.probabilities(s, e, m)
            cands = sorted(((float(np.float32(sp[0, i]) * np.float32(ep[0, j])), i, j) for i in range(L) for j in range(i, L)),
                           key=lambda t: (-t[0], t[1], t[2]))
            cands = [(i, j) for v, i, j in cands if v > 0]
            rank = {c: r for r, c in enumerate(cands)}
            for k in range(1, 13):
                si, ei, _, _ = TO.extract_topk(s, e, m, k=k, nms_thresh=thr)
                kept = [(int(a), int(b)) for a, b in zip(si[0], ei[0]) if a >= 0]
                assert all(si[0, len(kept):] == -1)
                for p, q in itertools.combinations(range(len(kept)), 2):    # pairwise below the threshold
                    assert not _removed(kept[q], kept[p], thr)
                for c in cands:
                    if c in kept:
                        continue
                    later = [r for r, kk in enumerate(kept) if rank[kk] > rank[c]]
                    if later or len(kept) < k:     # c was passed over (or the set ran out): an earlier kept span removed it
                        upto = later[0] if later else len(kept)
                        assert any(_removed(c, kept[r], thr) for r in range(upto)), (L, k, thr, c, kept)


# ---- host R@k mirrors and shard sums (CPU) ------------------------------------------------------------------------
def _fake_topk_batches(n=7, B=12, k=5, seed=5):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        s = torch.rand(B, generator=g) * 0.6
        gt = torch.stack([s, s + 0.1 + torch.rand(B, generator=g) * 0.3], 1)
        p = torch.rand(B, k, generator=g) * 0.6
        pr = torch.stack([p, p + 0.05 + torch.rand(B, k, generator=g) * 0.35], -1)
        pr[torch.rand(B, k, generator=g) < 0.2] = -1.0                          # empty slots
        out.append((gt.numpy().astype(np.float32), pr.numpy().astype(np.float32)))
    return out


def _topk_counts(batches):
    ious = []
    for gt, pr in batches:
        engine.append_ious_topk(ious, gt, pr)
    return [len(ious)] + [sum(i >= t for i in ious) for t in (0.3, 0.5, 0.7)], ious


def test_host_recall_at_k_matches_brute_force():
    batches = _fake_topk_batches()
    counts, ious = _topk_counts(batches)
    flat = []
    for gt, pr in batches:
        for b in range(gt.shape[0]):
            best = 0.0
            for q in range(pr.shape[1]):
                if pr[b, q, 0] < 0:
                    continue
                g0, g1, p0, p1 = (float(x) for x in (gt[b, 0], gt[b, 1], pr[b, q, 0], pr[b, q, 1]))
                u, i = max(g1, p1) - min(g0, p0), min(g1, p1) - max(g0, p0)
                best = max(best, 0.0 if u == 0 else max(0.0, i / u))
            flat.append(best)
    assert np.allclose(ious, flat, rtol=1e-6, atol=0)
    want = [100.0 * sum(x >= t for x in flat) / len(flat) for t in (0.3, 0.5, 0.7)]
    assert np.allclose(engine.recall_at_k(ious), want, rtol=1e-12)
    assert np.allclose(engine.metrics_topk_from_counters(counts), want, rtol=1e-12)
    # k = 1 reduces to the R1 entries of get_i345_mi
    gt, pr = batches[0]
    pr1 = np.where(pr[:, :1] < 0, np.float32(0.0), pr[:, :1])
    r1 = engine.get_i345_mi(engine.append_ious([], gt, pr1[:, 0]))
    assert np.allclose(engine.recall_at_k(engine.append_ious_topk([], gt, pr1)), (r1[0], r1[1], r1[3]), rtol=1e-12)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    batches = _fake_topk_batches()
    mine = [batches[i] for i in engine.shard_batches(len(batches), rank, world)]
    tk = engine.TopkCounters("cpu", 5, 0.5, buf=torch.tensor(_topk_counts(mine)[0], dtype=torch.float64))
    tk.allreduce()
    if rank == 0:
        q.put((tk.buf.tolist(), tk.result()))
    dist.destroy_process_group()


def test_topk_counter_allreduce_equals_single_process():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got, rec = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    counts, ious = _topk_counts(_fake_topk_batches())
    assert got == [float(c) for c in counts]
    assert np.allclose(rec, engine.recall_at_k(ious), rtol=1e-12)


# ---- C ABI argument checks (rejected before any launch) -----------------------------------------------------------
def test_invalid_arguments_are_reported_not_crashed():
    lib = _cabi.lib()
    p = C.c_void_p(16)       # never dereferenced: every call below is rejected first
    ok = dict(s=p, e=p, m=None, B=2, L=8, k=5, thr=0.5, si=p, ei=p, sc=p, fr=None)
    bad = [(dict(L=_cabi_max_vlen() + 1), b"L="), (dict(L=0), b"L="), (dict(k=0), b"k="), (dict(k=33), b"k="),
           (dict(thr=0.0), b"nms_thresh"), (dict(thr=1.5), b"nms_thresh"), (dict(thr=float("nan")), b"nms_thresh"),
           (dict(s=None), b"NULL"), (dict(e=None), b"NULL"), (dict(si=None), b"NULL"), (dict(ei=None), b"NULL"),
           (dict(sc=None), b"NULL"), (dict(B=-1), b"B=")]
    for change, msg in bad:
        a = {**ok, **change}
        rc = lib.seqpan_span_topk(a["s"], a["e"], a["m"], a["B"], a["L"], a["k"], a["thr"], a["si"], a["ei"], a["sc"], a["fr"], None)
        assert rc == -1 and msg in lib.seqpan_last_error(), (change, lib.seqpan_last_error())
    for args, msg in [((None, p, 2, 5, p), b"NULL"), ((p, None, 2, 5, p), b"NULL"), ((p, p, 2, 5, None), b"NULL"),
                      ((p, p, 2, 0, p), b"k="), ((p, p, 2, 33, p), b"k="), ((p, p, -1, 5, p), b"B=")]:
        assert lib.seqpan_topk_counters(*args, None) == -1 and msg in lib.seqpan_last_error(), args


def _cabi_max_vlen():
    return 256   # SEQPAN_MAX_VLEN in include/seqpan_b200.h


# ---- B200 -----------------------------------------------------------------------------------------------------------
def _device_topk(s, e, m, k, thr):
    from vmrframe_b200.seqpan import _topk
    si, ei, sc, fr = _topk(s.to(DEV), e.to(DEV), m.to(DEV) if m is not None else None, k, thr, True)
    return si.cpu().numpy(), ei.cpu().numpy(), sc.cpu().numpy(), fr.cpu().numpy()


def _k1_inputs():
    out = [_golden_logits(n)[:3] for n in CASES]
    out += [_random_logits(256, 100, 1), _random_logits(128, 256, 2)]
    return out


@pytest.mark.gpu
def test_top1_equals_the_device_decoder():
    from vmrframe_b200.seqpan import _decode
    n_unique = n_all = 0
    for s, e, m in _k1_inputs():
        for mask in (m, None):
            si, ei, sc, fr = _device_topk(s, e, mask, 2, 1.0)
            dsi, dei, dfr = _decode(s.to(DEV), e.to(DEV), mask.to(DEV) if mask is not None else None, True, True)
            dsi, dei, dfr = dsi.cpu().numpy(), dei.cpu().numpy(), dfr.cpu().numpy()
            assert np.array_equal(si[:, 0], dsi)
            unique = sc[:, 1] < sc[:, 0]               # the kernel's own bits: the maximum is attained by one span
            n_unique, n_all = n_unique + int(unique.sum()), n_all + len(unique)
            assert np.array_equal(ei[unique, 0], dei[unique])
            assert np.array_equal(fr[unique, 0].view(np.int32), dfr[unique].view(np.int32))
            # k = 1 is the first slot of any k
            si1, ei1, sc1, fr1 = _device_topk(s, e, mask, 1, 0.5)
            assert np.array_equal(si1[:, 0], si[:, 0]) and np.array_equal(ei1[:, 0], ei[:, 0])
            assert np.array_equal(sc1[:, 0], sc[:, 0])
    assert n_unique >= 0.9 * n_all


def _oracle_inputs():
    out = [(n,) + _golden_logits(n)[:3] for n in CASES]
    out += [("anet", *_random_logits(256, 100, 3)), ("tacos", *_random_logits(128, 256, 4))]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 5, 10])
def test_kernel_matches_oracle(k):
    taking_part = total = 0
    for name, s, e, m in _oracle_inputs():
        for thr in (0.3, 0.5, 0.7, 1.0):
            si, ei, sc, fr = _device_topk(s, e, m, k, thr)
            wsi, wei, wsc, mg = TO.extract_topk(s, e, m, k, thr)
            keep = np.all(mg > 1 + 1e-5, axis=1)
            taking_part, total = taking_part + int(keep.sum()), total + len(keep)
            assert np.array_equal(si[keep], wsi[keep]) and np.array_equal(ei[keep], wei[keep]), f"{name} k={k} thr={thr}"
            filled = keep[:, None] & (wsi >= 0)
            assert np.allclose(sc[filled], wsc[filled], rtol=1e-6, atol=0), f"{name} k={k} thr={thr}"
            assert np.array_equal(fr[keep], TO.fractions(wsi, wei, m, s.shape[1])[keep])
    assert taking_part >= 0.95 * total, f"only {taking_part} of {total} samples clear the tie margin"


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 7, 64, 100, 256])
def test_exact_ties_follow_the_index_rule(L):
    B = 6
    s, e = torch.zeros(B, L), torch.zeros(B, L)                          # rows 0-1: every span ties
    s[2:4] = torch.tensor([0.0, 3.0])[torch.arange(L) % 2]               # rows 2-3: duplicated values, distinct sums
    e[2:4] = 0.7 * (torch.arange(L) % 3 == 0).float()
    s[4], e[4] = s[2], e[2]
    s[5], e[5] = torch.randn(L), torch.randn(L)
    m = torch.ones(B, L)
    m[1, L - L // 3:] = 0
    m[3, L // 2:] = 0
    m[5] = 0                                                             # fully masked: uniform, as in the reference
    for k, thr in ((1, 0.5), (5, 0.5), (10, 0.3), (32, 1.0), (7, 0.7)):
        si, ei, sc, fr = _device_topk(s, e, m, k, thr)
        wsi, wei, wsc, _ = TO.extract_topk(s, e, m, k, thr)
        assert np.array_equal(si, wsi) and np.array_equal(ei, wei), (L, k, thr)
        assert np.array_equal(si[2], si[4]) and np.array_equal(sc[2], sc[4])
        assert np.array_equal(np.isnan(fr[5]), np.isnan(TO.fractions(wsi, wei, m, L)[5]))


@pytest.mark.gpu
def test_top1_counters_equal_the_iou_counters():
    from vmrframe_b200.seqpan import _decode
    _, _, batch, fx = golden_case("charades_full")
    inputs = [(torch.from_numpy(fx["slogits"]), torch.from_numpy(fx["elogits"]), batch["vmasks"], batch["se_fracs"])]
    s, e, m = _random_logits(256, 100, 9)
    g = torch.Generator().manual_seed(9)
    st = torch.rand(256, generator=g) * 0.6
    inputs.append((s, e, m, torch.stack([st, st + 0.05 + torch.rand(256, generator=g) * 0.35], 1)))
    for s, e, m, gt in inputs:
        _, _, _, fr = _device_topk(s, e, m, 1, 0.5)
        dfr = _decode(s.to(DEV), e.to(DEV), m.to(DEV), False, True)[2].cpu().numpy()
        same = np.all(fr[:, 0] == dfr, axis=1)
        assert same.mean() > 0.9
        tk = engine.TopkCounters(DEV, 1, 0.5)
        tk.update(torch.from_numpy(fr[same]), gt[torch.from_numpy(same)])
        ic = engine.IouCounters(DEV)
        ic.update(torch.from_numpy(dfr[same]), gt[torch.from_numpy(same)])
        t, i = tk.buf.cpu().tolist(), ic.buf.cpu().tolist()
        assert t[0] == i[0] and t[1:] == i[2:], (t, i)
        # and against the host mirror on the whole batch (best over filled slots, k = 5)
        _, _, _, fr5 = _device_topk(s, e, m, 5, 0.5)
        tk5 = engine.TopkCounters(DEV, 5, 0.5)
        tk5.update(torch.from_numpy(fr5), gt)
        ious = engine.append_ious_topk([], gt.numpy(), fr5)
        assert np.allclose(tk5.result(), engine.recall_at_k(ious), rtol=1e-12)


@pytest.mark.gpu
def test_repeated_and_graph_replayed_launches_are_bit_identical():
    s, e, m = (t.to(DEV) for t in _random_logits(128, 256, 5))
    B, L, k = 128, 256, 10
    outs = [torch.full((B, k), -7, dtype=torch.int64, device=DEV) for _ in range(2)] + \
        [torch.full((B, k), -7.0, device=DEV), torch.full((B, k, 2), -7.0, device=DEV)]

    def launch():
        _cabi.check(_cabi.lib().seqpan_span_topk(s.data_ptr(), e.data_ptr(), m.data_ptr(), B, L, k, 0.5,
                                                 *(o.data_ptr() for o in outs), torch.cuda.current_stream().cuda_stream))

    launch()
    first = [o.clone() for o in outs]
    for _ in range(3):
        for o in outs:
            o.fill_(-7)
        launch()
        assert all(torch.equal(a, b) for a, b in zip(outs, first))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch()                                    # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        launch()
    for o in outs:
        o.fill_(-7)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(outs, first))


def _pipe_model():
    from vmrframe_b200.seqpan import SeqPAN
    w = synth.small_workload("pipe", 8, 64, 10, 10, 77)
    m = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision="fp32").eval()
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=5))
    return w, m.to(DEV)


@pytest.mark.gpu
def test_evaluate_topk_equals_batchwise_calls():
    from vmrframe_b200 import extract_topk, infer_topk
    w, m = _pipe_model()
    batches = [synth.make_batch(w, i, pin=True) for i in range(5)]
    torch.manual_seed(11)
    metrics, counters, info = engine.evaluate(m, batches, DEV, return_fracs=True, streams=1, topk=5, nms_thresh=0.5)
    torch.manual_seed(11)
    metrics2, counters2, info2 = engine.evaluate(m, batches, DEV, return_fracs=True, streams=2, topk=5, nms_thresh=0.5)
    torch.manual_seed(11)
    metrics0, counters0, info0 = engine.evaluate(m, batches, DEV, return_fracs=True, streams=1)
    assert "topk" not in info0 and "topk_fracs" not in info0 and counters0.numel() == 5 and info0["d2h_bytes"] == 40 + 5 * 8 * 8
    tinfo = info["topk"]
    assert tinfo["k"] == 5 and tinfo["nms_thresh"] == 0.5 and len(tinfo["recall"]) == 3
    assert counters.numel() == 5 and tinfo["counters"].numel() == 4
    # R1 counts exact; the mIoU sum is added with fp64 atomics (order-dependent)
    c, c0 = counters.cpu().tolist(), counters0.cpu().tolist()
    assert c[0] == c0[0] and c[2:] == c0[2:] and abs(c[1] - c0[1]) <= 1e-12 * abs(c0[1])
    assert all(np.array_equal(a, b) for a, b in zip(info["fracs"], info0["fracs"]))
    # streams=2 equals streams=1
    assert all(np.array_equal(a, b) for a, b in zip(info["topk_fracs"], info2["topk_fracs"]))
    assert torch.equal(tinfo["counters"].cpu(), info2["topk"]["counters"].cpu()) and tinfo["recall"] == info2["topk"]["recall"]
    # batch by batch: the same forward, extract_topk / infer_topk and TopkCounters
    torch.manual_seed(11)
    tk = engine.TopkCounters(DEV, 5, 0.5)
    ious = []
    for hb, tf in zip(batches, info["topk_fracs"]):
        b = {k: v.to(DEV) for k, v in hb.items()}
        out = m(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"])
        fr = infer_topk(out, k=5, nms_thresh=0.5)
        assert fr.dtype == np.float32 and fr.shape == (hb["vmasks"].shape[0], 5, 2)
        assert np.array_equal(fr, tf)
        si, ei, sc = extract_topk(out["slogits"], out["elogits"], out["vmask"], k=5, nms_thresh=0.5)
        assert si.is_cuda and si.dtype == torch.int64 and sc.dtype == torch.float32 and si.shape == (hb["vmasks"].shape[0], 5)
        n = out["vmask"].sum(1, keepdim=True)
        filled = si >= 0
        assert torch.equal(torch.where(filled, si.float() / n, -1.0).cpu(), torch.from_numpy(fr[..., 0]))
        tk.update(torch.from_numpy(fr), hb["se_fracs"])
        engine.append_ious_topk(ious, hb["se_fracs"].numpy(), fr)
    assert torch.equal(tk.buf.cpu(), tinfo["counters"].cpu())
    assert np.allclose(tinfo["recall"], engine.recall_at_k(ious), rtol=1e-12)
    with pytest.raises(ValueError):
        engine.evaluate(m, batches, DEV, topk=0)
    with pytest.raises(ValueError):
        engine.evaluate(m, batches, DEV, topk=5, nms_thresh=0.0)
