"""CUDA-graph replay of the drop-in training routes: ``train_engine_*`` (``train.tape_loss``) and ``model(...)`` in ``train()``
(``train.forward_differentiable``).

CPU part: the graph key, that nothing is captured on the kernel emulation or with injected dropout masks, and the LRU / in-flight
bookkeeping of the shared cache driven with fake graph entries.  GPU part: graph replay against the same routes forced eager
(bit-identical under ``torch.use_deterministic_algorithms``, order-noise gates otherwise), the correctness cases of the autograd
node, the sibling models, DistributedDataParallel and the memory bound."""
import gc
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import vmrframe_b200 as V
from cpu_train_backend import CpuEmuBackend
from test_train import DEV, _case_model, _compare, _setup
from test_train_autograd import _free_port, _reference_losses
from test_train_bf16 import ORDER_GATES, _errors
from vmrframe_b200 import train


@pytest.fixture
def flag():
    """``flag(on)`` sets torch's deterministic-algorithms flag for one test; restored afterwards."""
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield lambda on: torch.use_deterministic_algorithms(on)
    torch.use_deterministic_algorithms(was, warn_only=warn)


def _captured(m):
    return sum("graph" in e for e in m._train_step._graphs.values())


# ======================================================================================================================
# CPU
# ======================================================================================================================
def test_graph_key_covers_what_the_graph_bakes_in_cpu(flag):
    w, m, batch, g = _setup(droprate=0.2)
    m.train()
    ts = train.TrainStep(m, backend=CpuEmuBackend())
    key = lambda **kw: ts._graph_key(kw.get("route", "loss"), kw.get("data", batch), kw.get("gumbel", g),
                                     kw.get("precision", "fp32"), kw.get("runtype", "train"))
    k0 = key()
    assert key() == k0 and hash(key()) == hash(k0)
    short = dict(batch, vfeats=batch["vfeats"][:, :-1])
    ints = dict(batch, vmasks=batch["vmasks"].to(torch.int64))
    variants = [key(route="node"), key(data=short), key(data=ints), key(gumbel=None), key(precision="bf16"),
                key(runtype="valid")]
    flag(True)
    variants.append(key())
    flag(False)
    m.eval()
    variants.append(key())
    m.train()
    m.configs.model.droprate = 0.1
    variants.append(key())
    m.configs.model.droprate = 0.2
    p = m.predictor.start_dense.conv1d.weight
    p.requires_grad_(False)
    variants.append(key())
    p.requires_grad_(True)
    assert key() == k0
    m.predictor.start_dense.conv1d.weight = torch.nn.Parameter(p.detach().clone())    # same values, new storage
    ts.named = dict(m.named_parameters())
    variants.append(key())
    assert len(set(variants + [k0])) == len(variants) + 1


def test_nothing_is_captured_on_the_emulation_or_with_injected_masks_cpu():
    w, m, batch, g = _setup(droprate=0.2)
    m.train()
    m._train_step = train.TrainStep(m, backend=CpuEmuBackend())
    for _ in range(4):
        loss, _ = train.tape_loss(m, batch, g)
        loss.backward()
    assert not m._train_step._graphs
    assert not train._can_capture(CpuEmuBackend(), batch["vfeats"])

    class GraphSafeCpu(CpuEmuBackend):
        graph_safe = True
    assert not train._can_capture(GraphSafeCpu(), batch["vfeats"])              # a CPU tensor
    x = SimpleNamespace(is_cuda=True)
    assert not train._can_capture(GraphSafeCpu(), x, mask_fn=lambda s: None)
    assert train.CudaBackend.graph_safe


def test_lru_eviction_and_in_flight_bookkeeping_cpu():
    """The cache driven with fake graphs: two eager runs before a capture, at most ``max_graphs`` captured entries, the least
    recently used one without a forward in flight evicted (its eager count kept), and an eager run when all are in flight."""
    w, m, batch, g = _setup()
    ts = train.TrainStep(m, backend=CpuEmuBackend())
    ts.max_graphs = 2

    def run(key, busy=False):
        ent = ts._entry(key)
        if busy and ent.get("busy"):
            return ent, False
        if ts._use_graph(ent):
            ent.setdefault("graph", object())        # a capture
            ent.setdefault("pool", object())
            return ent, True
        ent["seen"] += 1
        return ent, False

    assert [run("a")[1] for _ in range(3)] == [False, False, True]
    assert [run("b")[1] for _ in range(3)] == [False, False, True]
    run("a")                                         # a is now the most recently used
    for _ in range(2):
        run("c")
    c, replayed = run("c")
    assert replayed and set(k for k, e in ts._graphs.items() if "graph" in e) == {"a", "c"}
    assert ts._graphs["b"] == {"seen": 2}            # evicted: graph and pool dropped, eager count kept
    assert run("b")[1]                               # ... so it is captured again at once, evicting a
    assert "graph" not in ts._graphs["a"]
    # a forward in flight pins its entry: with both captured entries in flight a new key runs eagerly
    flights = [train._InFlight(ts._graphs[k]) for k in ("b", "c")]
    assert ts._graphs["b"]["busy"] and run("b", busy=True) == (ts._graphs["b"], False)
    for _ in range(3):
        ent, replayed = run("d")
    assert not replayed and ent["seen"] == 3 and "graph" not in ent
    del flights[0]                                   # b's outputs dropped (or backpropagated): b may be evicted again
    assert not ts._graphs["b"]["busy"] and run("d")[1] and "graph" not in ts._graphs["b"]
    del flights


# ======================================================================================================================
# GPU
# ======================================================================================================================
CFG = SimpleNamespace(device=DEV)


def _model(precision="fp32", eager=False, droprate=0.2):
    """A model on the device; ``eager``: its drop-in routes never replay (a cache that holds no graph)."""
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7, droprate=droprate)
    m.configs.model.train_precision = precision
    m.to(DEV).train()
    if eager:
        m._train_step = train.TrainStep(m)
        m._train_step.max_graphs = 0
    return m, {k: v.to(DEV) for k, v in batch.items()}, batch


def _module_loss(m, bd, batch, x=None):
    """model(...) on the device; the reference's losses in torch on the CPU copies of the outputs (cuBLAS refuses to run under
    the deterministic flag without a workspace setting)."""
    out = m(bd["words_ids"], bd["char_ids"], bd["vfeats"] if x is None else x, bd["vmasks"], bd["tmasks"])
    return _reference_losses(out["slogits"].cpu(), out["elogits"].cpu(), out["match_score"].cpu(), out["label_embs"].cpu(),
                             batch), out


def _loop(route, precision, eager, steps=5):
    """``steps`` iterations of the reference loop: loss -> backward -> clip_grad_norm_ -> AdamW, from seed 11."""
    m, bd, batch = _model(precision, eager)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3)
    torch.manual_seed(11)
    rec = []
    for _ in range(steps):
        loss = V.train_engine_SeqPAN(m, bd, CFG, "train")[0] if route == "engine" else _module_loss(m, bd, batch)[0]
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        opt.step()
        rec.append({"loss": loss.detach().cpu(), **{"g." + k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None},
                    **{"p." + k: p.detach().cpu() for k, p in m.named_parameters()}})
    return rec, m


def _equal(a, b, what):
    assert set(a) == set(b), what
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, f"{what}: {len(bad)} tensors differ, e.g. {bad[:4]}"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("route", ["engine", "module"])
def test_graph_replay_is_bit_identical_to_eager_in_deterministic_mode(flag, route, precision):
    """Dropout 0.2 from one seed: torch's graph-safe generator gives the replayed steps the eager draws."""
    flag(True)
    graphed, mg = _loop(route, precision, eager=False)
    eager, me = _loop(route, precision, eager=True)
    assert _captured(mg) == 1 and _captured(me) == 0
    for s, (a, b) in enumerate(zip(graphed, eager)):
        _equal(a, b, f"{route} {precision} step {s + 1}")


def _grads(m):
    return {k: p.grad.detach().cpu() for k, p in m.named_parameters() if p.grad is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("route", ["engine", "module"])
def test_graph_replay_meets_the_order_noise_gates_in_default_mode(route, precision):
    """Four calls on fixed parameters, the same draws per call: the replayed third and fourth against eager calls."""
    res = []
    for eager in (False, True):
        m, bd, batch = _model(precision, eager)
        calls = []
        for i in range(4):
            m.zero_grad(set_to_none=True)
            torch.manual_seed(20 + i)
            loss = V.train_engine_SeqPAN(m, bd, CFG, "train")[0] if route == "engine" else _module_loss(m, bd, batch)[0]
            loss.backward()
            calls.append((float(loss.detach()), _grads(m)))
        res.append(calls)
    assert _captured(m) == 0
    for (lg, got), (le, want) in list(zip(*res))[2:]:
        if precision == "fp32":
            assert math.isclose(lg, le, rel_tol=1e-5)
            _compare(got, want, rtol=1e-4)
        else:
            whole, cos, worst, name = _errors(got, want, floor=ORDER_GATES["floor"])
            assert abs(lg - le) <= ORDER_GATES["loss"] * abs(le)
            assert whole <= ORDER_GATES["whole"] and cos >= ORDER_GATES["cos"] and worst <= ORDER_GATES["per_tensor"], name


def _both(scenario):
    """``scenario(m, bd, batch)`` on a replaying model and on an eager twin under the deterministic flag: every tensor it
    returns is bit-identical between the two.  Returns the replaying model."""
    res = []
    for eager in (False, True):
        m, bd, batch = _model(eager=eager)
        torch.manual_seed(7)
        res.append((scenario(m, bd, batch), m))
    (a, mg), (b, _) = res
    _equal(a, b, scenario.__name__)
    assert _captured(mg) >= 1
    return mg


def _warm(m, bd, batch, route, n=2, **kw):
    for _ in range(n):
        m.zero_grad(set_to_none=True)
        loss = V.train_engine_SeqPAN(m, bd, CFG, "train")[0] if route == "engine" else _module_loss(m, bd, batch, **kw)[0]
        loss.backward()
    m.zero_grad(set_to_none=True)


@pytest.mark.gpu
def test_correctness_cases_of_the_replayed_routes(flag):
    flag(True)

    def accumulate_two_engine_calls(m, bd, batch):
        _warm(m, bd, batch, "engine")
        l1, o1 = V.train_engine_SeqPAN(m, bd, CFG, "train")
        l2, o2 = V.train_engine_SeqPAN(m, dict(bd, vfeats=0.5 * bd["vfeats"]), CFG, "train")
        (l1 + l2).backward()
        return {"l1": l1.detach(), "l2": l2.detach(), "s1": o1["slogits"], "s2": o2["slogits"], **_grads(m)}
    _both(accumulate_two_engine_calls)

    def two_forwards_before_their_backwards(m, bd, batch):
        _warm(m, bd, batch, "module")
        l1, o1 = _module_loss(m, bd, batch)               # replayed: its entry is in flight ...
        l2, o2 = _module_loss(m, bd, batch, x=0.5 * bd["vfeats"])     # ... so this one runs on the eager tape
        l1.backward()
        l2.backward()
        return {"l1": l1.detach(), "l2": l2.detach(), "s1": o1["slogits"].detach(), "s2": o2["slogits"].detach(), **_grads(m)}
    _both(two_forwards_before_their_backwards)

    def unused_outputs(m, bd, batch):
        _warm(m, bd, batch, "module")
        out = m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])
        (out["slogits"].cpu() * torch.linspace(-1, 1, out["slogits"].shape[1])).sum().backward()   # elogits, match_score: None
        g = _grads(m)
        assert not any(k.startswith("predictor.end") for k in g)
        return g
    _both(unused_outputs)

    def video_features_require_grad(m, bd, batch):
        x = bd["vfeats"].clone().requires_grad_()
        _warm(m, bd, batch, "module", n=3, x=x)
        return {"x": x.grad.cpu(), **_grads(m)}
    _both(video_features_require_grad)

    def frozen_parameters(m, bd, batch):
        m.video_affine.video_conv1d.conv1d.bias.requires_grad_(False)
        out = {}
        for route in ("engine", "module"):
            _warm(m, bd, batch, route, n=3)
            assert m.video_affine.video_conv1d.conv1d.bias.grad is None
            m.zero_grad()
            loss = V.train_engine_SeqPAN(m, bd, CFG, "train")[0] if route == "engine" else _module_loss(m, bd, batch)[0]
            loss.backward()
            out.update({route + k: v for k, v in _grads(m).items()})
        return out
    _both(frozen_parameters)

    def replaced_parameter(m, bd, batch):
        _warm(m, bd, batch, "module", n=3)
        p = m.predictor.start_dense.conv1d.weight
        m.predictor.start_dense.conv1d.weight = torch.nn.Parameter(1.5 * p.detach())
        _warm(m, bd, batch, "module", n=1)
        loss, _ = _module_loss(m, bd, batch)
        loss.backward()
        return {"loss": loss.detach(), **_grads(m)}
    mg = _both(replaced_parameter)
    assert _captured(mg) == 1 and len(mg._train_step._graphs) == 2     # the old key's graph stays; the new key is not yet due

    m, bd, batch = _model()
    _warm(m, bd, batch, "module")
    loss, out = _module_loss(m, bd, batch)
    assert _captured(m) == 1
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="tape is freed"):
        loss.backward()


@pytest.mark.gpu
def test_toggling_the_mode_never_replays_a_graph_of_the_other_mode(flag):
    """Three calls per mode (the third captures), then a call in the first mode again: it replays that mode's graph and equals
    the eager twin bit for bit.  Deterministic flag on both routes; the precision on model(...), which reads it per call."""
    for route, modes, set_mode in (("engine", (True, False), lambda m, v: flag(v)),
                                   ("module", (True, False), lambda m, v: flag(v)),
                                   ("module", ("fp32", "bf16"), lambda m, v: setattr(m.configs.model, "train_precision", v))):
        flag(True)
        res = []
        for eager in (False, True):
            m, bd, batch = _model(eager=eager)
            for i, mode in enumerate([modes[0]] * 3 + [modes[1]] * 3 + [modes[0]]):
                set_mode(m, mode)
                m.zero_grad(set_to_none=True)
                torch.manual_seed(30 + i)
                loss = V.train_engine_SeqPAN(m, bd, CFG, "train")[0] if route == "engine" else _module_loss(m, bd, batch)[0]
                loss.backward()
            flag(True)
            res.append(({"loss": loss.detach().cpu(), **_grads(m)}, m))
        (a, mg), (b, _) = res
        assert _captured(mg) == 2
        _equal(a, b, f"{route} {modes}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["train_basefast", "train_multiteacher", "train_backbone"])
def test_sibling_engines_replay_their_eager_results(flag, name):
    flag(True)
    res = []
    for eager in (False, True):
        variant, cfg, m, batch, g = _case_model(name)
        m.to(DEV).train()
        cfg.device = DEV
        if eager:
            m._train_step = train.TrainStep(m)
            m._train_step.max_graphs = 0
        engine = {"basefast": V.train_engine_BaseFast, "multiteacher": V.train_engine_MultiTeacher,
                  "backbone": V.train_engine_BackBone}[variant]
        torch.manual_seed(3)
        losses = []
        for _ in range(4):
            m.zero_grad(set_to_none=True)
            loss, _ = engine(m, batch, cfg, "train")      # MultiTeacher: "train" carries the three teacher terms
            loss.backward()
            losses.append(loss.detach().cpu())
        res.append(({"loss": torch.stack(losses), **_grads(m)}, m))
    (a, mg), (b, _) = res
    assert _captured(mg) == 1
    _equal(a, b, name)


# ---- DistributedDataParallel over the replayed node -------------------------------------------------------------------
class _Wrapped(torch.nn.Module):
    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, bd):
        return self.m(bd["words_ids"], bd["char_ids"], bd["vfeats"], bd["vmasks"], bd["tmasks"])


def _ddp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    backend = "nccl" if dist.is_nccl_available() and torch.cuda.device_count() >= world else "gloo"
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    from vmrframe_b200 import synth
    from vmrframe_b200.seqpan import SeqPAN
    wm = synth.small_workload("ddp_graph", 4, 32, 9, 7, 740, num_words=60)
    m = SeqPAN(synth.make_configs(wm, droprate=0.2), synth.make_word_vectors(wm))
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=4))
    m.to(dev).train()
    ddp = torch.nn.parallel.DistributedDataParallel(_Wrapped(m), find_unused_parameters=True)
    opt = torch.optim.SGD(ddp.parameters(), lr=0.05)
    w = synth.small_workload("ddp_graph", 4, 32, 9 + 3 * rank, 7, 750 + rank, num_words=60)     # a batch shape per rank
    bd = {k: v.to(dev) for k, v in synth.add_train_labels(synth.make_batch(w, 0)).items()}
    torch.manual_seed(40 + rank)
    for _ in range(5):
        out = ddp(bd)
        loss = _reference_losses(out["slogits"], out["elogits"], out["match_score"], out["label_embs"], bd)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    torch.cuda.synchronize()
    q.put((rank, sum("graph" in e for e in m._train_step._graphs.values()),
           {k: p.detach().cpu().numpy().copy() for k, p in m.named_parameters()}))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_distributed_data_parallel_over_replayed_forwards():
    """Two ranks, different batch shapes, five steps (the third on each rank replays): the ranks end bit-identical."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in range(2)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, n0, p0), (_, n1, p1) = res
    assert n0 == 1 and n1 == 1
    for k in p0:
        assert np.array_equal(p0[k], p1[k]), f"{k} differs between the ranks"


@pytest.mark.gpu
def test_memory_stays_bounded_over_more_shapes_than_the_bound():
    """``max_graphs`` = 2 and a stream of five batch shapes, each three times (the third captures): never more than two
    captured entries, and the device memory after the stream is what two captures hold, not five."""
    from vmrframe_b200 import synth
    m, _, _ = _model()
    ts = train._train_step_of(m)
    ts.max_graphs = 2
    shapes = {}
    for tmax in range(5, 20):
        w = synth.small_workload("train", 4, 32, tmax, 7, 503, num_words=60)
        b = synth.add_train_labels(synth.make_batch(w, 0))
        shapes.setdefault(tuple(b["words_ids"].shape), {k: v.to(DEV) for k, v in b.items()})
    batches = list(shapes.values())[:5]
    assert len(batches) == 5

    def reserved():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.memory_reserved(DEV)

    base = reserved()
    pools = []
    for bd in batches:
        for _ in range(3):
            loss, _ = V.train_engine_SeqPAN(m, bd, CFG, "train")
            loss.backward()
            m.zero_grad(set_to_none=True)
        assert _captured(m) <= 2
        pools.append(reserved())
    grow = [b - a for a, b in zip([base] + pools, pools)]
    print(f"\nreserved after each shape (MB): {[round(p / 2 ** 20, 1) for p in pools]}")
    assert _captured(m) == 2
    assert pools[-1] - base <= 1.25 * (pools[1] - base) + (64 << 20), grow
