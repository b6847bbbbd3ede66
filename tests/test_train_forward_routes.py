"""The training forward is recorded in one place for every route: ``forward_only``, the autograd node's forward
(``forward_differentiable``) and the forward half of ``TrainStep.loss_and_grads`` issue the same kernel calls, in the same
order, with the same arguments and keywords, on the same inputs and seed (dropout 0.2, Gumbel noise drawn by the forward),
with torch's deterministic flag off and on, in fp32 and bf16.  CPU only: the calls are logged on the kernel emulation."""
import hashlib

import pytest
import torch

import vmrframe_b200 as V
from cpu_train_backend import CpuEmuBackend
from vmrframe_b200 import synth, train

KERNELS = ("gemm", "ewise", "softmax", "softmax_bwd", "layernorm", "layernorm_bwd", "dwconv", "dwconv_bwd_w", "gather_rows",
           "scatter_add_rows", "maxpool", "maxpool_bwd", "sumsq", "adamw", "dropout_mask", "gumbel")


def _desc(x):
    if torch.is_tensor(x):
        digest = hashlib.sha1(x.detach().contiguous().numpy().tobytes()).hexdigest()
        return ("tensor", tuple(x.shape), x.stride(), str(x.dtype), digest)
    if isinstance(x, (list, tuple)):
        return tuple(_desc(v) for v in x)
    if isinstance(x, dict):
        return tuple(sorted((k, _desc(v)) for k, v in x.items()))
    return x


def _logged(name):
    def call(self, *args, **kw):
        self.calls.append((name, _desc(args), _desc(kw)))
        kw.pop("mixed", None)                 # the emulation's products are fp32 in every mode
        kw.pop("deterministic", None)
        return getattr(CpuEmuBackend, name)(self, *args, **kw)
    return call


class RecordingBackend(CpuEmuBackend):
    """The kernel emulation, logging every kernel call: its name, its tensors by shape, strides, dtype and a digest of their
    values, and its other arguments and keywords by value."""

    def __init__(self):
        self.calls = []

    def empty(self, shape):                   # output buffers are logged too: no uninitialised memory in the log
        return torch.zeros(tuple(shape), dtype=torch.float32)


for _name in KERNELS:
    setattr(RecordingBackend, _name, _logged(_name))


@pytest.fixture
def flag():
    """``flag(on)`` sets torch's deterministic-algorithms flag for one test; restored afterwards."""
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield lambda on: torch.use_deterministic_algorithms(on)
    torch.use_deterministic_algorithms(was, warn_only=warn)


@pytest.fixture
def case():
    """A small model of each forward variant in ``train()`` with dropout 0.2, and a labelled batch."""
    w = synth.small_workload("train", 3, 24, 7, 6, 531, num_words=60)
    batch = synth.add_train_labels(synth.make_batch(w, 0))

    def make(variant, precision):
        m = getattr(V, variant)(synth.make_configs(w, droprate=0.2), synth.make_word_vectors(w))
        m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=6))
        m.configs.model.train_precision = precision
        return m.train()
    return make, batch


class _Stop(Exception):
    pass


def _trainstep_forward(m, batch, monkeypatch):
    be = RecordingBackend()

    def stop(*a, **k):
        raise _Stop
    with monkeypatch.context() as mp:
        mp.setattr(train, "compose_loss", stop)       # the losses come after the forward
        with pytest.raises(_Stop):
            train.TrainStep(m, backend=be).loss_and_grads(batch)
    return be.calls


def _node_forward(m, batch, monkeypatch):
    be = RecordingBackend()
    train.forward_differentiable(m, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"],
                                 backend=be)
    return be.calls


def _forward_only(m, batch, monkeypatch):
    be = RecordingBackend()
    with monkeypatch.context() as mp:
        mp.setattr(train, "CudaBackend", lambda device: be)
        with torch.no_grad():
            train.forward_only(m, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"])
    return be.calls


@pytest.mark.parametrize("variant", ["SeqPAN", "BackBone"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("det", [False, True])
def test_forward_routes_issue_the_same_kernel_calls_cpu(flag, monkeypatch, case, variant, precision, det):
    make, batch = case
    m = make(variant, precision)
    flag(det)
    logs = []
    for route in (_trainstep_forward, _node_forward, _forward_only):
        torch.manual_seed(17)
        logs.append(route(m, batch, monkeypatch))
    names = [c[0] for c in logs[0]]
    assert names.count("dropout_mask") > 10 and names.count("gumbel") == (variant == "SeqPAN")
    assert any(dict(c[2]).get("mixed") for c in logs[0] if c[0] == "gemm") == (precision == "bf16")
    for route, log in zip(("node forward", "forward_only"), logs[1:]):
        assert len(log) == len(logs[0]), route
        diff = next((i for i, (a, b) in enumerate(zip(logs[0], log)) if a != b), None)
        assert diff is None, f"{route}: call {diff} differs: {log[diff][0]} against TrainStep's {logs[0][diff][0]}"
