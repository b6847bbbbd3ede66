"""The training-mode forward as a torch autograd node: ``train.forward_differentiable`` and ``model(...)`` in ``train()``.

Any torch loss on the outputs backpropagates through the tape's adjoints on the training kernels.  CPU part: the node on the
kernel emulation (tests/cpu_train_backend.py) against the oracle's autograd for arbitrary output cotangents, the reference's
losses written in torch against ``tape_loss``, the sibling models, which tensors receive a gradient, and DistributedDataParallel
over gloo.  GPU part: the ``model(...)`` route on the device against the oracle, bit-identical values with and without a
graph, agreement with ``train_engine_SeqPAN`` in fp32 and bf16, and span decoding of outputs that require grad."""
import gc
import math
import os
import socket
import weakref
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cpu_train_backend import CpuEmuBackend
from oracle import seqpan_oracle as O
from test_train import DEAD, DEV, _case_model, _compare, _Masks, _oracle_train_engine, _setup
from test_train_bf16 import ORDER_GATES, _errors
from vmrframe_b200 import engine, synth, train
from vmrframe_b200.seqpan import SeqPAN


class EmuBackend(CpuEmuBackend):
    """The kernel emulation, whose LayerNorm and depthwise-conv adjoints are torch autograd calls of their own: an autograd
    node's backward runs with grad mode off, so they switch it back on."""

    def layernorm_bwd(self, *a):
        with torch.enable_grad():
            return super().layernorm_bwd(*a)

    def dwconv_bwd_w(self, *a):
        with torch.enable_grad():
            return super().dwconv_bwd_w(*a)


PAD_ROWS = ("text_encoder.char_emb.char_emb.weight", "text_encoder.word_emb.word_emb.weight")


def _cotangents(B, L, seed=9):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, L, generator=g), torch.randn(B, L, generator=g), torch.randn(B, L, 4, generator=g)


def _objective(W, sl, el, ms):
    """sum(ws * slogits) + sum(we * elogits) + sum(wm * match_score); a term whose weight is None is left out."""
    return sum((w.to(o.device) * o).sum() for w, o in zip(W, (sl, el, ms)) if w is not None)


def _replay_masks(be, masks, p, device="cpu"):
    """The backend's dropout draws replaced by the oracle's stream of keep-masks (same sites, same order, same shapes)."""
    be.dropout_mask = lambda shape, p_: masks.keep(shape).to(device) / (1.0 - p)
    return be


def _oracle(m, batch, g, W, drop=None):
    """Gradients of ``_objective`` over the oracle's autograd, for every parameter and for ``vfeats``."""
    sd = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in m.named_parameters()}
    full = dict(m.state_dict())
    full.update(sd)
    x = batch["vfeats"].clone().requires_grad_()
    O.DROP = drop
    try:
        out = O.forward(full, batch["words_ids"], batch["char_ids"], x, batch["vmasks"], batch["tmasks"], g)
    finally:
        O.DROP = None
    _objective(W, out["slogits"], out["elogits"], out["match_score"]).backward()
    want = {k: v.grad for k, v in sd.items() if v.grad is not None}
    want["vfeats"] = x.grad
    return want, out


def _node(m, batch, g, W, be, device="cpu"):
    """The same gradients through ``forward_differentiable``: ``p.grad`` and ``vfeats.grad`` after ``backward()``."""
    m.zero_grad(set_to_none=True)
    x = batch["vfeats"].to(device).clone().requires_grad_()
    bd = {k: v.to(device) for k, v in batch.items()}
    sl, el, ms = train.forward_differentiable(m, bd["words_ids"], bd["char_ids"], x, bd["vmasks"], bd["tmasks"],
                                              g.to(device), backend=be)
    _objective(W, sl, el, ms).backward()
    got = {k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None}
    got["vfeats"] = x.grad.cpu()
    return got, (sl, el, ms)


# ======================================================================================================================
# CPU
# ======================================================================================================================
@pytest.mark.parametrize("pretrained", [True, False])
@pytest.mark.parametrize("dropout", [0.0, 0.2])
def test_random_cotangents_match_oracle_autograd_cpu(dropout, pretrained):
    w, m, batch, g = _setup(droprate=dropout, pretrained=pretrained)
    m.train()
    W = _cotangents(*batch["vmasks"].shape)
    want, out_o = _oracle(m, batch, g, W, drop=_Masks(0.2).oracle_drop if dropout else None)
    be = _replay_masks(EmuBackend(), _Masks(0.2), dropout) if dropout else EmuBackend()
    got, (sl, el, ms) = _node(m, batch, g, W, be)
    assert torch.allclose(sl.detach(), out_o["slogits"].detach(), atol=1e-5)
    assert torch.allclose(ms.detach(), out_o["match_score"].detach(), atol=1e-5)
    for k in PAD_ROWS:            # the oracle's nn.Embedding(padding_idx=0) leaves row 0 at zero: so does the node
        if k in got:
            assert not bool(got[k][0].any())
    _compare(got, want)


def _reference_losses(sl, el, ms, label_embs, bd):
    return engine.lossfun_loc(sl, el, bd["label1ds"][:, 0, :], bd["label1ds"][:, 1, :], bd["vmasks"]) + \
        engine.lossfun_match(ms, label_embs, bd["NER_labels"], bd["vmasks"])


def test_reference_losses_on_the_outputs_equal_tape_loss_cpu():
    """engine.lossfun_loc + lossfun_match in torch on the node's outputs give the gradients of tape_loss, which builds the same
    losses on the tape.  The two differ only in where the loss is summed (torch's CPU reductions against the emulated ones-vector
    GEMMs in fp64): measured on this case at 1.4e-6 of a tensor's largest gradient, the loss equal to the last bit."""
    w, m, batch, g = _setup()
    m.train()
    m._train_step = train.TrainStep(m, backend=EmuBackend())
    loss_t, _ = train.tape_loss(m, batch, g)
    loss_t.backward()
    want = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    m.zero_grad(set_to_none=True)
    sl, el, ms = train.forward_differentiable(m, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"],
                                              batch["tmasks"], g, backend=EmuBackend())
    loss = _reference_losses(sl, el, ms, m.label_embs, batch)
    loss.backward()
    got = {k: p.grad for k, p in m.named_parameters() if p.grad is not None}
    assert math.isclose(float(loss.detach()), float(loss_t.detach()), rel_tol=1e-6)
    _compare(got, want, rtol=1e-4)


def _sibling_case(name, be, device="cpu"):
    """A sibling model's reference loss (the oracle's torch restatement of train_engine_<Model>) on the node's outputs, against
    the oracle's own autograd of the same loss."""
    variant, cfg, m, batch, g = _case_model(name)
    loss_o, want, _ = _oracle_train_engine(name)
    m.to(device).train()
    bd = {k: v.to(device) for k, v in batch.items()}
    sl, el, ms = train.forward_differentiable(m, bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"],
                                              g.to(device), backend=be)
    assert (ms is None) == (variant == "backbone")
    out = {"slogits": sl, "elogits": el, "match_score": ms}
    loss = O.train_engine_loss(variant, out, bd, cfg.loss, "train", getattr(m, "label_embs", None))
    loss.backward()
    got = {k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None}
    assert math.isclose(float(loss), float(loss_o), rel_tol=1e-4)
    _compare(got, want, rtol=1e-3)


@pytest.mark.parametrize("name", ["train_basefast", "train_multiteacher", "train_backbone"])
def test_sibling_models_backpropagate_reference_losses_cpu(name):
    _sibling_case(name, EmuBackend())


def test_which_tensors_receive_gradients_cpu():
    w, m, batch, g = _setup(pretrained=False)
    m.train()
    m.video_affine.video_conv1d.conv1d.bias.requires_grad_(False)         # a frozen parameter the forward uses
    be = EmuBackend()
    W = _cotangents(*batch["vmasks"].shape)
    args = (batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    sl, el, ms = train.forward_differentiable(m, *args, backend=be)
    _objective(W, sl, el, ms).backward()
    named = dict(m.named_parameters())
    dead = [k for k in named if any(d in k for d in DEAD)]
    assert len(dead) == 20 and all(named[k].grad is None for k in dead)
    assert named["video_affine.video_conv1d.conv1d.bias"].grad is None
    live = {k: p.grad for k, p in named.items() if p.grad is not None}
    assert len(live) == len(named) - 20 - 1
    for k in PAD_ROWS:
        assert not bool(live[k][0].any()) and bool(live[k][1:].any())
    ptrs = [p.untyped_storage().data_ptr() for p in live.values()]
    assert len(set(ptrs)) == len(ptrs)            # no two gradients share storage
    # AccumulateGrad adds a second backward's gradients into the first's in place: an aliased gradient would be added twice
    first = {k: v.clone() for k, v in live.items()}
    sl2, el2, ms2 = train.forward_differentiable(m, *args, backend=be)
    _objective(W, sl2, el2, ms2).backward()
    for k, v in first.items():
        assert torch.allclose(named[k].grad, 2 * v, rtol=1e-6, atol=1e-9), k
    # the tape is freed by its backward: a second one through the node raises, even with retain_graph; so does a double backward
    with pytest.raises(RuntimeError, match="tape is freed"):
        sl2.backward(W[0])
    sl3, _, _ = train.forward_differentiable(m, *args, backend=be)
    sl3.backward(W[0], retain_graph=True)
    with pytest.raises(RuntimeError, match="tape is freed"):
        sl3.backward(W[0])
    sl4, _, _ = train.forward_differentiable(m, *args, backend=be)
    (gs,) = torch.autograd.grad(sl4, [named["predictor.start_dense.conv1d.bias"]], W[0].clone().requires_grad_(), create_graph=True)
    with pytest.raises(RuntimeError, match="differentiate twice"):
        gs.sum().backward()


def test_tape_is_freed_when_the_outputs_are_dropped_cpu():
    """A forward whose outputs are dropped without a backward (a monitoring forward, a skipped step, an exception between
    forward and backward) frees its tape at once, by reference counting; so does one after its backward."""
    w, m, batch, g = _setup()
    m.train()
    args = (batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    was = gc.isenabled()
    gc.disable()
    try:
        for backward in (False, True):
            sl, el, ms = train.forward_differentiable(m, *args, backend=EmuBackend())
            tape, out = weakref.ref(sl.grad_fn.rec.tp), weakref.ref(sl._base)
            assert tape() is not None
            if backward:
                (sl.sum() + el.sum()).backward()
            del sl, el, ms
            assert tape() is None and out() is None, backward
    finally:
        if was:
            gc.enable()


def test_unused_outputs_get_no_cotangent_cpu():
    """Only slogits in the loss: elogits / match_score get no cotangent; the gradients equal the oracle's of the same loss."""
    w, m, batch, g = _setup()
    m.train()
    B, L = batch["vmasks"].shape
    W = (_cotangents(B, L)[0], None, None)
    want, _ = _oracle(m, batch, g, W)
    m.zero_grad(set_to_none=True)
    x = batch["vfeats"].clone().requires_grad_()
    sl, el, ms = train.forward_differentiable(m, batch["words_ids"], batch["char_ids"], x, batch["vmasks"], batch["tmasks"], g,
                                              backend=EmuBackend())
    (W[0] * sl).sum().backward()
    got = {k: p.grad for k, p in m.named_parameters() if p.grad is not None}
    got["vfeats"] = x.grad
    _compare(got, want)
    assert not any(k.startswith("predictor.end") for k in got)        # the end branch only feeds elogits


# ---- DistributedDataParallel over the node ---------------------------------------------------------------------------
class _Wrapped(torch.nn.Module):
    """A user's module around SeqPAN whose forward is the differentiable training forward on the kernel emulation."""

    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, bd, g):
        return train.forward_differentiable(self.m, bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"],
                                            g, backend=EmuBackend())


def _ddp_model():
    wm = synth.small_workload("ddp_ag", 2, 16, 6, 5, 710, num_words=40)
    m = SeqPAN(synth.make_configs(wm, droprate=0.0), synth.make_word_vectors(wm))
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=2))
    return m.train()


def _ddp_batch(rank):
    w = synth.small_workload("ddp_ag", 2, 16, 6, 5, 720 + rank, num_words=40)
    return synth.add_train_labels(synth.make_batch(w, 0)), synth.gumbel_noise(2, 16, seed=30 + rank)


def _ddp_loss(out, bd, label_embs):
    sl, el, ms = out
    return _reference_losses(sl, el, ms, label_embs, bd)


def _ddp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    m = _ddp_model()
    ddp = torch.nn.parallel.DistributedDataParallel(_Wrapped(m), find_unused_parameters=True)
    opt = torch.optim.SGD(ddp.parameters(), lr=0.1)
    bd, g = _ddp_batch(rank)
    _ddp_loss(ddp(bd, g), bd, m.label_embs).backward()
    opt.step()
    q.put((rank, {k: p.detach().numpy().copy() for k, p in m.named_parameters()}))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def test_distributed_data_parallel_over_the_node_cpu():
    """Two gloo ranks, different batches: after one backward and an SGD step the parameters are identical on both ranks and
    equal a single-process step on the mean of the two ranks' gradients."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, p0), (_, p1) = res
    grads = []
    for rank in range(2):
        m = _ddp_model()
        bd, g = _ddp_batch(rank)
        _ddp_loss(_Wrapped(m)(bd, g), bd, m.label_embs).backward()
        grads.append({k: p.grad for k, p in m.named_parameters() if p.grad is not None})
    assert set(grads[0]) == set(grads[1]) and not torch.allclose(grads[0]["label_embs"], grads[1]["label_embs"])
    m = _ddp_model()
    for k, p in m.named_parameters():
        assert np.array_equal(p0[k], p1[k]), f"{k} differs between the ranks"
        want = p.detach() - 0.1 * (grads[0][k] + grads[1][k]) / 2 if k in grads[0] else p.detach()
        assert np.allclose(p0[k], want.numpy(), rtol=1e-6, atol=1e-7), k


# ======================================================================================================================
# GPU: the model(...) route
# ======================================================================================================================
def _golden_model(name, droprate=0.0):
    from conftest import golden_case
    w, sd, batch, fx = golden_case(name)
    m = SeqPAN(synth.make_configs(w, droprate=droprate), synth.make_word_vectors(w))
    m.load_state_dict(sd)
    with torch.no_grad():      # off the orthogonal manifold: the norm term of lossfun_match has a kink at E^T E = I
        m.label_embs.add_(0.05 * torch.randn(m.label_embs.shape, generator=torch.Generator().manual_seed(1)))
    return m, synth.add_train_labels(batch), torch.from_numpy(fx["gumbel"])


def _module_grads(m, bd, g, W):
    m.zero_grad(set_to_none=True)
    x = bd["vfeats"].clone().requires_grad_()
    out = m(bd["words_ids"], bd["char_ids"], x, bd["vmasks"], bd["tmasks"], gumbel=g)
    assert out["slogits"].grad_fn is not None and out["label_embs"] is m.label_embs
    _objective(W, out["slogits"], out["elogits"], out["match_score"]).backward()
    dev = [p.grad for p in m.parameters() if p.grad is not None] + [x.grad]
    assert len({t.untyped_storage().data_ptr() for t in dev}) == len(dev)      # no two gradients share storage
    got = {k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None}
    got["vfeats"] = x.grad.cpu()
    return got, out


@pytest.mark.gpu
@pytest.mark.parametrize("dropout", [0.0, 0.2])
@pytest.mark.parametrize("case", ["charades_small", "anet_small"])
def test_module_route_matches_oracle_autograd(case, dropout):
    m, batch, g = _golden_model(case, droprate=dropout)
    W = _cotangents(*batch["vmasks"].shape)
    want, out_o = _oracle(m, batch, g, W, drop=_Masks(0.2).oracle_drop if dropout else None)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    masks = _Masks(0.2)
    orig = train.CudaBackend.dropout_mask
    if dropout:        # the oracle's draws through the backend the module builds
        train.CudaBackend.dropout_mask = lambda self, shape, p: masks.keep(shape).to(self.device) / (1.0 - p)
    try:
        got, out = _module_grads(m, bd, g.to(DEV), W)
    finally:
        train.CudaBackend.dropout_mask = orig
    assert torch.allclose(out["slogits"].detach().cpu(), out_o["slogits"].detach(), atol=1e-4)
    _compare(got, want, rtol=1e-3)


@pytest.mark.gpu
def test_forwards_without_backward_release_their_device_memory():
    """Training-mode forwards with a graph whose outputs are dropped without a backward hold no device memory afterwards."""
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7, droprate=0.2)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    args = (bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
    m(*args)                            # warm-up: whatever torch allocates once per process exists before the baseline
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    was = gc.isenabled()
    gc.disable()
    try:
        for _ in range(3):
            out = m(*args)
            assert out["slogits"].grad_fn is not None and torch.cuda.memory_allocated(DEV) > base
            del out
            assert torch.cuda.memory_allocated(DEV) == base
    finally:
        if was:
            gc.enable()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_values_are_bit_identical_with_and_without_a_graph(precision):
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7, droprate=0.2)
    m.configs.model.train_precision = precision
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    args = (bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
    torch.manual_seed(21)
    a = m(*args)
    torch.manual_seed(21)
    with torch.no_grad():
        b = m(*args)
    torch.manual_seed(21)
    with torch.inference_mode():
        c = m(*args)
    for k in ("slogits", "elogits", "match_score"):
        assert torch.equal(a[k].detach(), b[k]) and torch.equal(b[k], c[k]), k
    assert a["slogits"].grad_fn is not None and b["slogits"].grad_fn is None and c["slogits"].grad_fn is None
    for p in m.parameters():          # nothing requires grad: no graph either
        p.requires_grad_(False)
    torch.manual_seed(21)
    d = m(*args)
    assert d["slogits"].grad_fn is None and torch.equal(d["slogits"], b["slogits"])
    x = bd["vfeats"].clone().requires_grad_()      # ... unless the video features do
    torch.manual_seed(21)
    e = m(*args[:2], x, *args[3:])
    e["slogits"].sum().backward()
    assert torch.equal(e["slogits"].detach(), b["slogits"]) and x.grad is not None and bool(x.grad.any())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_module_route_agrees_with_train_engine(precision):
    """lossfun_loc + lossfun_match on model(...) then loss.backward() against train_engine_SeqPAN(...)[0].backward() under the
    same seed (dropout 0.2: the same draws).  fp32: rtol 1e-4 of each tensor's largest gradient.  bf16: ORDER_GATES."""
    from vmrframe_b200 import train_engine_SeqPAN
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7, droprate=0.2)
    m.configs.model.train_precision = precision
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    torch.manual_seed(5)
    loss_e, _ = train_engine_SeqPAN(m, batch, SimpleNamespace(device=DEV), "train")
    loss_e.backward()
    want = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters() if p.grad is not None}
    m.zero_grad(set_to_none=True)
    torch.manual_seed(5)
    out = m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
    loss = _reference_losses(out["slogits"], out["elogits"], out["match_score"], out["label_embs"], bd)
    loss.backward()
    got = {k: p.grad.detach().cpu() for k, p in m.named_parameters() if p.grad is not None}
    whole, cos, worst, name = _errors(got, want, floor=ORDER_GATES["floor"])
    print(f"\n{precision}: loss {float(loss):.7f} vs {float(loss_e):.7f}, whole-gradient rel {whole:.3e}, cos {cos:.8f}, "
          f"worst per-tensor rel {worst:.3e} ({name})")
    if precision == "fp32":
        assert math.isclose(float(loss), float(loss_e), rel_tol=1e-5)
        _compare(got, want, rtol=1e-4)
    else:
        assert abs(float(loss) - float(loss_e)) <= ORDER_GATES["loss"] * abs(float(loss_e))
        assert whole <= ORDER_GATES["whole"] and cos >= ORDER_GATES["cos"] and worst <= ORDER_GATES["per_tensor"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["train_basefast", "train_multiteacher", "train_backbone"])
def test_sibling_models_module_route_matches_oracle(name):
    variant, cfg, m, batch, g = _case_model(name)
    loss_o, want, _ = _oracle_train_engine(name)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    out = m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"], gumbel=g.to(DEV))
    assert set(out) == ({"slogits", "elogits", "vmask", "consume_time"} if variant == "backbone" else
                        {"slogits", "elogits", "vmask", "match_score", "label_embs", "consume_time"})
    loss = O.train_engine_loss(variant, out, bd, cfg.loss, "train", out.get("label_embs"))
    loss.backward()
    got = {k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None}
    assert math.isclose(float(loss), float(loss_o), rel_tol=1e-4)
    _compare(got, want, rtol=1e-3)


@pytest.mark.gpu
def test_decoding_accepts_outputs_that_require_grad():
    from vmrframe_b200.seqpan import extract_index, infer_basic_device, infer_SeqPAN
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    out = m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"], gumbel=g.to(DEV))
    assert out["slogits"].requires_grad and out["elogits"].requires_grad
    det = {k: (v.detach() if torch.is_tensor(v) else v) for k, v in out.items()}
    assert np.array_equal(infer_SeqPAN(out), infer_SeqPAN(det))
    for a, b in zip(extract_index(out["slogits"], out["elogits"]), extract_index(det["slogits"], det["elogits"])):
        assert torch.equal(a, b)
    assert torch.equal(infer_basic_device(out["slogits"], out["elogits"], out["vmask"]),
                       infer_basic_device(det["slogits"], det["elogits"], det["vmask"]))
