"""Stored video encodings (DESIGN.md section 12): ``encode_videos`` + ``forward(video_encodings=)`` and
``evaluate(video_encodings=)``.  On the GPU every encoded result is compared bit for bit with the shared-video forward on
the raw clips (the same kernels on the same rows); on the CPU, the argument checks of the C ABI and of the module."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import seqpan_oracle as O
from test_gpu_parity import TOL, _close
from vmrframe_b200 import BackBone, BaseFast, MultiTeacher, OneTeacher, SeqPAN, VideoEncodings, _cabi, engine, synth

DEV = "cuda:0"
VARIANTS = {"seqpan": SeqPAN, "basefast": BaseFast, "multiteacher": MultiTeacher, "backbone": BackBone}
SHAPES = [(12, 64, 10, 4), (8, 100, 25, 8), (6, 256, 19, 3)]   # (B, L, T, pairs per clip) of the shared-video test


def _model(cls, w, precision, seed=3, device=DEV):
    m = cls(synth.make_configs(w), synth.make_word_vectors(w), precision=precision).eval()
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=seed))
    return m.to(device)


def _keys(m):
    return ("slogits", "elogits") + (("match_score",) if m._MATCH_HEAD else ())


def _shared_batch(w, group, idx=0):
    return {k: v.to(DEV) for k, v in synth.share_clips(synth.make_batch(w, idx), group).items()}


def _fwd(m, b, vfeats, g, **kw):
    return m(b["words_ids"], b["char_ids"], vfeats, b["vmasks"], b["tmasks"], gumbel=g, **kw)


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("shape", SHAPES)
def test_encoded_forward_equals_shared_video_forward(variant, precision, shape):
    B, L, T, group = shape
    w = synth.Workload("encoded", 40 + B, B, L, T, 10, num_words=300, group=group)
    m = _model(VARIANTS[variant], w, precision)
    b = _shared_batch(w, group)
    g = synth.gumbel_noise(B, L).to(DEV)
    want = _fwd(m, b, b["vfeats"], g, video_index=b["video_index"])
    enc = m.encode_videos(b["vfeats"])
    assert enc.rows.shape == (b["vfeats"].shape[0], L, 128) and enc.precision == precision
    out = _fwd(m, b, None, g, video_index=b["video_index"], video_encodings=enc)
    for k in _keys(m):
        assert torch.equal(out[k], want[k]), k
    assert set(out) == set(want)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("L", [64, 100, 256])
def test_encoding_does_not_depend_on_neighbours(precision, L):
    """One call, chunks of 3 and one clip at a time give equal rows (L = 64 packs two clips per conv-block tile)."""
    w = synth.Workload("neighbours", 9, 7, L, 10, 10, num_words=300)
    m = _model(SeqPAN, w, precision)
    v = synth.make_batch(w, 0)["vfeats"]
    whole = m.encode_videos(v.to(DEV)).rows
    assert torch.equal(m.encode_videos(v.to(DEV), chunk=3).rows, whole)
    assert torch.equal(torch.cat([m.encode_videos(v[i:i + 1].to(DEV)).rows for i in range(v.shape[0])]), whole)


@pytest.mark.gpu
def test_fp32_encoded_forward_against_oracle():
    B, L, T, group = 8, 100, 25, 4
    w = synth.Workload("encoded_oracle", 71, B, L, T, 10, num_words=300, group=group)
    m = _model(SeqPAN, w, "fp32")
    batch = synth.make_batch(w, 0)
    b = {k: v.to(DEV) for k, v in synth.share_clips(batch, group).items()}
    g = synth.gumbel_noise(B, L)
    out = _fwd(m, b, None, g.to(DEV), video_index=b["video_index"], video_encodings=m.encode_videos(b["vfeats"]))
    with torch.no_grad():
        want = O.forward({k: v.cpu() for k, v in m.state_dict().items()}, batch["words_ids"], batch["char_ids"],
                         batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    for k in ("slogits", "elogits", "match_score"):
        _close(out[k].cpu(), want[k], f"encoded/fp32/{k}", **TOL["fp32"])


@pytest.mark.gpu
def test_large_library_scattered_index_and_identity():
    """4096 encoded clips against batches of 16: scattered indices and video_index=None (pair b -> clip b); a chunk above the
    library's batch limit (768) is lowered to it."""
    B, L, U = 16, 64, 4096
    w = synth.Workload("library", 12, B, L, 10, 10, num_words=300)
    m = _model(SeqPAN, w, "bf16")
    gen = torch.Generator(device=DEV).manual_seed(5)
    lib = torch.randn(U, L, 1024, device=DEV, generator=gen)
    enc = m.encode_videos(lib, chunk=1000)
    assert len(enc) == U and m._limits[0] == 768
    b = {k: v.to(DEV) for k, v in synth.make_batch(w, 0).items()}
    g = synth.gumbel_noise(B, L).to(DEV)
    idx = torch.randint(0, U, (B,), device=DEV, generator=gen)
    idx[0], idx[1], idx[2] = 0, U - 1, idx[3]                       # both ends of the library and a repeated clip
    out = _fwd(m, b, None, g, video_index=idx, video_encodings=enc)
    uniq, inv = torch.unique(idx, return_inverse=True)
    want = _fwd(m, b, lib[uniq], g, video_index=inv.to(torch.int32))
    for k in _keys(m):
        assert torch.equal(out[k], want[k]), k
    out = _fwd(m, b, None, g, video_encodings=enc)
    want = _fwd(m, b, lib[:B], g, video_index=torch.arange(B, device=DEV, dtype=torch.int32))
    for k in _keys(m):
        assert torch.equal(out[k], want[k]), k
    # the encode call is bounded by the workspace: at most max_batch clips per call
    over = m._limits[0] + 1
    rc = _cabi.lib().seqpan_encode_videos(m._handle, lib.data_ptr(), over, enc.rows.data_ptr(), m._workspace.data_ptr(),
                                          m._workspace.numel(), torch.cuda.current_stream().cuda_stream)
    assert rc < 0 and b"max_batch" in _cabi.lib().seqpan_last_error()


@pytest.mark.gpu
def test_graph_replay_of_encoded_forward_is_bitwise_equal():
    """Repeated encoded forwards on the same buffers are captured and replayed as one CUDA graph (B*L <= 8192 rows)."""
    B, L, T, group = 12, 64, 10, 4
    w = synth.Workload("encoded_graph", 52, B, L, T, 10, num_words=300, group=group)
    m = _model(SeqPAN, w, "bf16")
    b = _shared_batch(w, group)
    enc = m.encode_videos(b["vfeats"])
    g = synth.gumbel_noise(B, L).to(DEV)
    vi = b["video_index"].to(torch.int32).contiguous()
    static = (torch.empty(B, L, device=DEV), torch.empty(B, L, device=DEV), torch.empty(B, L, 4, device=DEV))
    outs = []
    for _ in range(4):       # plain launches, capture + launch, replay, replay
        for t in static:
            t.fill_(float("nan"))
        m.forward_into(b["words_ids"], b["char_ids"], None, b["vmasks"], b["tmasks"], g, *static, vi, video_encodings=enc)
        torch.cuda.synchronize()
        outs.append(tuple(t.clone() for t in static))
    for o in outs[1:]:
        assert all(torch.equal(x, y) for x, y in zip(o, outs[0]))
    want = _fwd(m, b, b["vfeats"], g, video_index=vi)
    assert torch.equal(outs[0][0], want["slogits"]) and torch.equal(outs[0][2], want["match_score"])


@pytest.mark.gpu
def test_debug_taps_on_the_encoded_forward():
    B, L, T, group = 8, 100, 25, 8
    w = synth.Workload("encoded_taps", 48, B, L, T, 10, num_words=300, group=group)
    m = _model(SeqPAN, w, "fp32")
    b = _shared_batch(w, group)
    g = synth.gumbel_noise(B, L).to(DEV)
    m.set_debug_taps(True)
    _fwd(m, b, b["vfeats"], g, video_index=b["video_index"])
    want = {n: m.debug_tap(n).clone() for n in ("text_emb", "venc", "tenc", "dab1_v", "fuse2", "fep_e")}
    _fwd(m, b, None, g, video_index=b["video_index"], video_encodings=m.encode_videos(b["vfeats"]))
    for n, t in want.items():
        assert torch.equal(m.debug_tap(n), t), n
    with pytest.raises(_cabi.SeqpanError, match="video_affine"):
        m.debug_tap("video_affine")


@pytest.mark.gpu
@pytest.mark.parametrize("topk", [None, 5])
def test_evaluate_from_encodings_matches_raw_clips(topk):
    w = synth.Workload("encoded_sweep", 61, 16, 64, 10, 10, num_words=300, group=8)
    m = _model(SeqPAN, w, "bf16", seed=9)
    batches = [synth.share_clips(synth.make_batch(w, i, pin=True), w.group) for i in range(4)]
    lib = torch.cat([bt["vfeats"] for bt in batches])                 # one library over the sweep: batch i owns rows [2i, 2i+2)
    enc = m.encode_videos(lib.to(DEV))
    enc_batches = []
    for i, bt in enumerate(batches):
        e = {k: v for k, v in bt.items() if k != "vfeats"}
        e["video_index"] = (bt["video_index"] + 2 * i).to(torch.int32)
        enc_batches.append(e)
    torch.manual_seed(3)
    metrics, counters, info = engine.evaluate(m, batches, DEV, return_fracs=True, streams=2, topk=topk)
    torch.manual_seed(3)
    metrics_e, counters_e, info_e = engine.evaluate(m, enc_batches, DEV, return_fracs=True, streams=2, topk=topk,
                                                    video_encodings=enc)
    assert metrics == metrics_e and torch.equal(counters, counters_e)
    torch.manual_seed(3)                                                # the device left to the caller's current one
    metrics_d, counters_d, _ = engine.evaluate(m, enc_batches, streams=2, topk=topk, video_encodings=enc)
    assert metrics_d == metrics_e and torch.equal(counters_d, counters_e)
    assert all(np.array_equal(a, b) for a, b in zip(info["fracs"], info_e["fracs"]))
    if topk:
        assert info["topk"]["recall"] == info_e["topk"]["recall"] and torch.equal(info["topk"]["counters"], info_e["topk"]["counters"])
        assert all(np.array_equal(a, b) for a, b in zip(info["topk_fracs"], info_e["topk_fracs"]))
    # ids, masks, ground truth and clip indices: not one video byte
    no_video = sum((bt["words_ids"].numel() + bt["char_ids"].numel()) * 8 + (bt["vmasks"].numel() + bt["tmasks"].numel()
                   + bt["se_fracs"].numel() + bt["video_index"].numel()) * 4 for bt in enc_batches)
    assert info_e["h2d_bytes"] == no_video
    assert info["h2d_bytes"] - no_video == lib.numel() * 4


@pytest.mark.gpu
def test_stale_and_mismatched_encodings_raise():
    B, L, T, group = 12, 64, 10, 4
    w = synth.Workload("encoded_stale", 44, B, L, T, 10, num_words=300, group=group)
    m = _model(SeqPAN, w, "bf16")
    b = _shared_batch(w, group)
    g = synth.gumbel_noise(B, L).to(DEV)
    vi = b["video_index"]
    enc = m.encode_videos(b["vfeats"])
    _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    opt = torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=1e-3)
    for p in m.parameters():
        p.grad = torch.zeros_like(p) if p.requires_grad else None
    opt.step()                                                          # an optimizer step
    with pytest.raises(_cabi.SeqpanError, match="weights changed"):
        _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    enc = m.encode_videos(b["vfeats"])
    _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    m.load_state_dict(m.state_dict())                                  # load_state_dict
    with pytest.raises(_cabi.SeqpanError, match="weights changed"):
        _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    enc = m.encode_videos(b["vfeats"])
    for other in (_model(SeqPAN, w, "fp32"), _model(BaseFast, w, "bf16")):   # another precision, another variant
        with pytest.raises(_cabi.SeqpanError, match="made by"):
            _fwd(other, b, None, g, video_index=vi, video_encodings=enc)
    w_aff = m.video_affine.video_conv1d.conv1d.weight
    with torch.no_grad():
        w_aff.data.mul_(1.01)                                          # an edit no version counter sees ...
    m.repack()                                                          # ... followed by repack()
    with pytest.raises(_cabi.SeqpanError, match="weights changed"):
        _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    enc = m.encode_videos(b["vfeats"])
    m.freeze()                                                          # frozen: the weight check is skipped
    opt.step()
    _fwd(m, b, None, g, video_index=vi, video_encodings=enc)
    stale = m.encode_videos(b["vfeats"])                                # made from what was packed before that step
    m.freeze(False)
    with pytest.raises(_cabi.SeqpanError, match="weights changed"):
        _fwd(m, b, None, g, video_index=vi, video_encodings=stale)
    _fwd(m, b, None, g, video_index=vi, video_encodings=m.encode_videos(b["vfeats"]))


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_c_abi_rejects_bad_encoded_arguments():
    lib = _cabi.lib()
    p = C.c_void_p(256)      # never dereferenced: every call below fails its argument checks first
    assert lib.seqpan_encode_videos(None, None, 1, p, p, 1 << 20, None) < 0 and b"NULL" in lib.seqpan_last_error()
    assert lib.seqpan_encode_videos(None, p, 1, None, p, 1 << 20, None) < 0 and b"NULL" in lib.seqpan_last_error()
    assert lib.seqpan_encode_videos(None, p, 0, p, p, 1 << 20, None) < 0 and b"U=0" in lib.seqpan_last_error()
    assert lib.seqpan_encode_videos(None, p, 4, C.c_void_p(264), p, 1 << 20, None) < 0 and b"aligned" in lib.seqpan_last_error()
    assert lib.seqpan_encode_videos(None, p, 4, p, p, 1 << 20, None) < 0 and b"handle" in lib.seqpan_last_error()

    def fwd(venc, vindex, U, B):
        return lib.seqpan_forward_encoded(None, p, p, venc, vindex, U, p, p, p, B, 8, 8, p, p, p, p, 1 << 20, None)

    assert fwd(None, p, 4, 2) < 0 and b"venc is NULL" in lib.seqpan_last_error()
    assert fwd(p, p, 0, 2) < 0 and b"U=0" in lib.seqpan_last_error()
    assert fwd(C.c_void_p(260), p, 4, 2) < 0 and b"aligned" in lib.seqpan_last_error()
    assert fwd(p, None, 3, 4) < 0 and b"U=3 < B=4" in lib.seqpan_last_error()
    assert fwd(p, None, 4, 4) < 0 and b"handle" in lib.seqpan_last_error()


def _cpu_model(cls=SeqPAN):
    w = synth.Workload("guards", 3, 4, 64, 10, 10, num_words=300)
    return w, cls(synth.make_configs(w), synth.make_word_vectors(w), precision="bf16").eval()


def _cpu_batch(w):
    b = synth.make_batch(w, 0)
    return b["words_ids"], b["char_ids"], b["vmasks"], b["tmasks"]


def test_python_guards_of_encoded_calls():
    w, m = _cpu_model()
    words, chars, vm, tm = _cpu_batch(w)
    enc = VideoEncodings(torch.zeros(6, w.vlen, 128), "bf16", m._VARIANT, None)
    with pytest.raises(_cabi.SeqpanError, match="vfeat_in=None"):
        m(words, chars, torch.zeros(4, w.vlen, w.vdim), vm, tm, video_encodings=enc)
    with pytest.raises(_cabi.SeqpanError, match="rows must be"):
        m(words, chars, None, vm, tm, video_encodings=VideoEncodings(torch.zeros(6, w.vlen, 64), "bf16", m._VARIANT, None))
    with pytest.raises(_cabi.SeqpanError, match="outside"):
        m(words, chars, None, vm, tm, video_index=torch.tensor([0, 1, 2, 6], dtype=torch.int32), video_encodings=enc)
    with pytest.raises(_cabi.SeqpanError, match="made by"):
        m(words, chars, None, vm, tm, video_encodings=VideoEncodings(enc.rows, "fp32", m._VARIANT, None))
    m.train()
    with pytest.raises(_cabi.SeqpanError, match="eval"):
        m(words, chars, None, vm, tm, video_encodings=enc)
    with pytest.raises(_cabi.SeqpanError, match="eval"):
        m.encode_videos(torch.zeros(2, w.vlen, w.vdim))
    m.eval()
    with pytest.raises(_cabi.SeqpanError, match="vfeats must be"):
        m.encode_videos(torch.zeros(2, w.vlen, 64))


def test_oneteacher_has_no_stored_encodings():
    w, m = _cpu_model(OneTeacher)
    words, chars, vm, tm = _cpu_batch(w)
    with pytest.raises(NotImplementedError):
        m.encode_videos(torch.zeros(2, w.vlen, w.vdim))
    with pytest.raises(NotImplementedError):
        m(words, chars, None, vm, tm, video_encodings=VideoEncodings(torch.zeros(4, w.vlen, 128), "bf16", 0, None))
