"""Training step of SeqPAN on the B200 kernels (SURVEY.md section 8 rows a19 / f4; BASELINE.json configs[4]).

Mirrors (reference file:line):
  * ``train_engine_SeqPAN``                    models/SeqPAN.py:171-182   forward (dropout active) + the two losses
  * ``lossfun_loc`` / ``lossfun_match``        models/loss.py:24-54
  * ``loss.backward()``                        main.py:94                 reverse-mode tape below
  * ``clip_grad_norm_(1.0)`` + ``AdamW.step``  main.py:95-96, utils/utils.py:87-97 (no-decay groups: names with
                                               ``bias`` / ``layer_norm`` / ``LayerNorm``)
  * linear warm-up / decay schedule            utils/utils.py:95-96 (transformers.get_linear_schedule_with_warmup)
  * gradient all-reduce (data parallel)        one flat fp32 bucket of the live gradients, NCCL sum / world size

How it is built.  The reference's backward is torch autograd over ~430 ATen operators.  Here ``SeqpanTape`` records the
training forward as a list of nodes, each a primitive with a forward rule and a hand-written vector-Jacobian rule, and
replays them in reverse.  Every rule is a call into ``libseqpan_b200.so`` (csrc/train_ops.cu: strided batched SGEMM,
broadcasting element-wise kernel, strided softmax, LayerNorm / depthwise-conv / embedding / max-pool adjoints, fused AdamW);
PyTorch supplies device memory, views (strides), the dropout / Gumbel random draws and ``torch.distributed``.  There is no
CPU path: the kernel backend refuses CPU tensors.  (tests/ substitute a torch-on-CPU emulation of the *kernels* to check the
tape and the adjoint rules against the oracle's autograd without a GPU; the product never does.)

The forward here is the reference's training forward restated primitive by primitive (same dropout sites, same order:
models/layers.py:48,67,119,146,284,291,294,296,352,357,431-432,570,631-638).  It deliberately does not reuse the fused
tcgen05 inference kernels yet: those keep no activations.  fp32 by default; ``precision="bf16"`` (``TrainStep`` /
``configs.model.train_precision``) runs the model's matrix products on the tensor cores (csrc/train_tc.cu) with bf16 operands
and fp32 accumulation, and keeps everything else fp32.
"""
from __future__ import annotations

import collections
import contextlib
import ctypes as C
import gc
import math

import torch

from . import _cabi

D, H, HD = 128, 4, 32
MASKV = -1e30
PRECISIONS = ("fp32", "bf16")      # training precision modes (see SeqpanTape)
# Input shapes a TrainStep keeps as CUDA graphs, least recently used evicted first; shared by TrainStep.step, the train engines
# and model(...) in train().  Each captured shape holds its activations in a graph pool (DESIGN.md section 10 gives the measured
# size per shape).
GRAPH_CACHE_SIZE = 16


@contextlib.contextmanager
def _capture(graph, pool=None):
    """``torch.cuda.graph`` with the cyclic garbage collector off.  A collection during a capture may destroy the graphs of a
    dead model (a model and its ``TrainStep`` form a cycle), a call that is illegal while a stream captures and that would
    invalidate the capture; so pending garbage is collected first."""
    was = gc.isenabled()
    torch.cuda.synchronize()
    gc.collect()
    gc.disable()
    try:
        with torch.cuda.graph(graph, pool=pool):
            yield
    finally:
        if was:
            gc.enable()


def _due(ent):
    """Whether a graph entry is due for capture (or holds its graph): after two eager runs of its key, when the lazy state of a
    run (Adam moments, the gradient bucket, the backend's caches) exists."""
    return ent["seen"] >= 2


def _replay(ent, fn, data, gumbel):
    """``fn(data, gumbel)`` replayed from the entry's CUDA graph, captured on first use.  The inputs (a dict of tensors) and the
    Gumbel draw are staged into static clones at the capture and copied in before every replay; the dropout draws stay fresh
    (torch's graph-safe generator).  Returns what ``fn`` returned at the capture, which the replay overwrites in place."""
    if "graph" not in ent:
        ent["in"] = {k: v.detach().clone() for k, v in data.items()}
        ent["gum"] = gumbel.clone() if gumbel is not None else None
        g = torch.cuda.CUDAGraph()
        with _capture(g):
            ent["out"] = fn(ent["in"], ent["gum"])
        ent["graph"] = g
    for k, v in data.items():
        ent["in"][k].copy_(v, non_blocking=True)
    if gumbel is not None:
        ent["gum"].copy_(gumbel, non_blocking=True)
    ent["graph"].replay()
    return ent["out"]


def _check_precision(precision):
    if precision not in PRECISIONS:
        raise ValueError(f"training precision {precision!r}: expected one of {PRECISIONS}")
    return precision


def train_precision(model, precision=None):
    """The training precision of ``model``: ``precision`` when given, else ``configs.model.train_precision`` (so the reference's
    own loop opts in from its YAML), else ``"fp32"``.  The module's inference ``precision=`` is a different setting and is not
    consulted."""
    if precision is None:
        precision = getattr(model.configs.model, "train_precision", "fp32")
    return _check_precision(precision)


def deterministic_mode():
    """True while ``torch.use_deterministic_algorithms(True)`` is in force (``warn_only=True`` included: the deterministic
    kernels exist, so there is nothing to warn about).  Then every tape reduces with the fixed-order ``seqpan_t_*_det`` kernels
    instead of float atomics, and two runs of a step on the same inputs and draws are bit-identical (DESIGN.md section 10).
    ``cudnn.deterministic`` is deliberately not consulted."""
    return torch.are_deterministic_algorithms_enabled()


# ---------------------------------------------------------------------------------------------------------------------
# kernel backend: torch tensors in, library kernels underneath
# ---------------------------------------------------------------------------------------------------------------------
def _pad4(vals, fill):
    vals = list(vals)
    return [fill] * (4 - len(vals)) + vals


class CudaBackend:
    """Thin tensor-level wrappers of the ``seqpan_t_*`` kernels.  Operands may be strided views (transposes, head splits
    and broadcasts are stride tricks, never copies)."""
    graph_safe = True       # every call is a stream-ordered launch with no host synchronisation: a tape on it can be captured

    def __init__(self, device):
        _cabi.require_device()
        self.device = torch.device(device)
        self.L = _cabi.lib()
        self._ones = {}

    # -- helpers --
    def _st(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _chk(self, rc):
        if rc < 0:
            raise _cabi.SeqpanError(f"training kernel failed ({rc}): {self.L.seqpan_t_last_error().decode()} / "
                                    f"{self.L.seqpan_last_error().decode()}")

    def _req(self, *ts):
        for t in ts:
            if t is not None and (not t.is_cuda or t.dtype != torch.float32):
                raise _cabi.SeqpanError("training kernels need float32 CUDA tensors (there is no CPU path)")

    def empty(self, shape):
        return torch.empty(tuple(shape), dtype=torch.float32, device=self.device)

    def _scratch(self, nbytes):
        """Device scratch of a deterministic kernel (fp32 elements; torch's allocator, so the graph's pool under capture)."""
        return self.empty(((nbytes + 7) // 8 * 2,))

    def zeros(self, shape):
        return torch.zeros(tuple(shape), dtype=torch.float32, device=self.device)

    def ones(self, n):
        if n not in self._ones:
            self._ones[n] = torch.ones(n, dtype=torch.float32, device=self.device)
        return self._ones[n]

    def dropout_mask(self, shape, p):
        """0 or 1/(1-p) per element, drawn by torch's own ``F.dropout`` (on a contiguous ones tensor of this shape) from torch's
        generator, at the reference's sites and in the reference's order.  Same distribution and generator, NOT bit-identical
        masks to a seeded reference run: torch's CUDA dropout kernel maps its Philox draws to elements differently for the
        non-contiguous tensors the reference feeds it at some sites (every ``Conv1D`` output is a transposed view).  Parity tests
        therefore inject the oracle's masks (``mask_fn``) instead of relying on seeds."""
        key = ("ones", tuple(shape))
        if key not in self._ones:
            self._ones[key] = torch.ones(tuple(shape), dtype=torch.float32, device=self.device)
        return torch.nn.functional.dropout(self._ones[key], p, True)

    def gumbel(self, shape):
        """The draw ``F.gumbel_softmax`` makes (models/SeqPAN.py:79; torch/nn/functional.py): -empty(shape).exponential_().log()."""
        return -torch.empty(tuple(shape), dtype=torch.float32, device=self.device).exponential_().log()

    # -- C[..., M, N] = alpha * A[..., M, K] @ B[..., K, N] + beta * C --
    def gemm(self, A, B, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None, mixed=False, deterministic=False):
        """``mixed=True``: bf16 operands (rounded to nearest even), fp32 accumulation, on the tensor cores
        (``seqpan_t_gemm_bf16``); otherwise the fp32 kernel.  ``deterministic=True``: a split-K product reduces its partial
        tiles in a fixed order (``seqpan_t_gemm_det`` / ``_bf16_det``) instead of with atomics."""
        self._req(A, B, out, bias)
        nb = A.dim() - 2
        assert B.dim() == A.dim() and 0 <= nb <= 2 and A.shape[-1] == B.shape[-2] and A.shape[:nb] == B.shape[:nb]
        M, K, N = A.shape[-2], A.shape[-1], B.shape[-1]
        if out is None:
            out = self.empty(tuple(A.shape[:nb]) + (M, N))
        assert tuple(out.shape) == tuple(A.shape[:nb]) + (M, N)
        g = _cabi.SeqpanGemm()
        g.M, g.N, g.K = M, N, K
        g.a_rs, g.a_cs, g.b_rs, g.b_cs, g.c_rs, g.c_cs = (A.stride(-2), A.stride(-1), B.stride(-2), B.stride(-1),
                                                          out.stride(-2), out.stride(-1))
        bs = _pad4(A.shape[:nb], 1)[2:]
        g.batch0, g.batch1 = bs
        sa, sb, sc = (_pad4(t.stride()[:nb], 0)[2:] for t in (A, B, out))
        g.a_b0, g.a_b1, g.b_b0, g.b_b1, g.c_b0, g.c_b1 = sa[0], sa[1], sb[0], sb[1], sc[0], sc[1]
        g.alpha, g.beta, g.splitk = alpha, beta, splitk if nb == 0 and out.stride(-1) == 1 else 1
        args = (A.data_ptr(), B.data_ptr(), out.data_ptr(), bias.data_ptr() if bias is not None else None, C.byref(g))
        if deterministic and g.splitk > 1:
            nbytes = self.L.seqpan_t_gemm_det_scratch_bytes(C.byref(g))
            fn = self.L.seqpan_t_gemm_bf16_det if mixed else self.L.seqpan_t_gemm_det
            scratch = self._scratch(nbytes)
            self._chk(fn(*args, scratch.data_ptr(), nbytes, self._st()))
        else:
            fn = self.L.seqpan_t_gemm_bf16 if mixed else self.L.seqpan_t_gemm
            self._chk(fn(*args, self._st()))
        return out

    # -- element-wise with broadcasting over <= 4 dims --
    def ewise(self, op, a, b=None, c=None, out=None, alpha=1.0, beta=0.0, accumulate=False):
        self._req(a, b, c, out)
        ops = [t for t in (a, b, c) if t is not None]
        shape = torch.broadcast_shapes(*[t.shape for t in ops])
        assert len(shape) <= 4
        if out is None:
            out = self.empty(shape)
        assert tuple(out.shape) == tuple(shape)
        e = _cabi.SeqpanEwise()
        e.op, e.accumulate, e.alpha, e.beta = _cabi.EW[op], int(accumulate), alpha, beta
        sh = _pad4(shape, 1)
        for i in range(4):
            e.shape[i] = sh[i]
        for name, t in (("so", out), ("sa", a), ("sb", b), ("sc", c)):
            st = _pad4(t.expand(shape).stride(), 0) if t is not None else [0, 0, 0, 0]
            arr = getattr(e, name)
            for i in range(4):
                arr[i] = st[i]
        self._chk(self.L.seqpan_t_ewise(out.data_ptr(), a.data_ptr(), b.data_ptr() if b is not None else None,
                                        c.data_ptr() if c is not None else None, C.byref(e), self._st()))
        return out

    def _softmax_desc(self, x, dim):
        assert x.is_contiguous()
        dim = dim % x.dim()
        inner = 1
        for s in x.shape[dim + 1:]:
            inner *= s
        outer = x.numel() // (inner * x.shape[dim])
        s = _cabi.SeqpanSoftmax()
        s.rows0, s.rows1, s.r0_stride, s.r1_stride, s.cols, s.c_stride = outer, inner, x.shape[dim] * inner, 1, x.shape[dim], inner
        return s

    def softmax(self, x, dim):
        self._req(x)
        y = torch.empty_like(x)
        self._chk(self.L.seqpan_t_softmax(y.data_ptr(), x.data_ptr(), C.byref(self._softmax_desc(x, dim)), self._st()))
        return y

    def softmax_bwd(self, y, dy, dim):
        self._req(y, dy)
        dy = dy if dy.is_contiguous() else self.ewise("COPY", dy)
        dx = torch.empty_like(y)
        self._chk(self.L.seqpan_t_softmax_bwd(dx.data_ptr(), y.data_ptr(), dy.data_ptr(), C.byref(self._softmax_desc(y, dim)), self._st()))
        return dx

    def layernorm(self, x, g, b, eps):
        self._req(x, g, b)
        assert x.is_contiguous() and x.shape[-1] == D
        y = torch.empty_like(x)
        _cabi.check(self.L.seqpan_op_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), C.c_float(eps), y.data_ptr(),
                                               x.numel() // D, self._st()))
        return y

    def layernorm_bwd(self, x, dy, g, eps, deterministic=False):
        self._req(x, dy, g)
        dy = dy if dy.is_contiguous() else self.ewise("COPY", dy)
        dx, dg, db = torch.empty_like(x), self.zeros((D,)), self.zeros((D,))
        args = (dx.data_ptr(), dg.data_ptr(), db.data_ptr(), x.data_ptr(), dy.data_ptr(), g.data_ptr(), C.c_float(eps), x.numel() // D)
        if deterministic:
            nb = self.L.seqpan_t_layernorm_bwd_det_scratch_bytes(x.numel() // D)
            scratch = self._scratch(nb)
            self._chk(self.L.seqpan_t_layernorm_bwd_det(*args, scratch.data_ptr(), nb, self._st()))
        else:
            self._chk(self.L.seqpan_t_layernorm_bwd(*args, self._st()))
        return dx, dg, db

    def dwconv(self, x, w, seg_len, flip=False):
        self._req(x, w)
        assert x.is_contiguous() and w.is_contiguous() and x.shape[-1] == D
        y = torch.empty_like(x)
        self._chk(self.L.seqpan_t_dwconv(y.data_ptr(), x.data_ptr(), w.data_ptr(), x.numel() // D, seg_len, int(flip), self._st()))
        return y

    def dwconv_bwd_w(self, x, dy, seg_len, deterministic=False):
        self._req(x, dy)
        dy = dy if dy.is_contiguous() else self.ewise("COPY", dy)
        dw = self.zeros((D, 1, 7))
        args = (dw.data_ptr(), x.data_ptr(), dy.data_ptr(), x.numel() // D, seg_len)
        if deterministic:
            nb = self.L.seqpan_t_dwconv_bwd_w_det_scratch_bytes(x.numel() // D)
            scratch = self._scratch(nb)
            self._chk(self.L.seqpan_t_dwconv_bwd_w_det(*args, scratch.data_ptr(), nb, self._st()))
        else:
            self._chk(self.L.seqpan_t_dwconv_bwd_w(*args, self._st()))
        return dw

    def gather_rows(self, table, ids):
        self._req(table)
        assert table.is_contiguous() and ids.dtype == torch.int64 and ids.is_contiguous()
        out = self.empty(tuple(ids.shape) + (table.shape[1],))
        self._chk(self.L.seqpan_t_gather_rows(out.data_ptr(), table.data_ptr(), ids.data_ptr(), ids.numel(), table.shape[1],
                                              table.shape[0], self._st()))
        return out

    def scatter_add_rows(self, dout, ids, rows, deterministic=False):
        self._req(dout)
        dout = dout if dout.is_contiguous() else self.ewise("COPY", dout)
        dt = self.zeros((rows, dout.shape[-1]))
        fn = self.L.seqpan_t_scatter_add_rows_det if deterministic else self.L.seqpan_t_scatter_add_rows
        self._chk(fn(dt.data_ptr(), dout.data_ptr(), ids.data_ptr(), ids.numel(), dout.shape[-1], rows, self._st()))
        return dt

    def maxpool(self, x):
        self._req(x)
        assert x.is_contiguous() and x.dim() == 3
        N, P, Cc = x.shape
        out = self.empty((N, Cc))
        idx = torch.empty((N, Cc), dtype=torch.int32, device=self.device)
        self._chk(self.L.seqpan_t_maxpool(out.data_ptr(), idx.data_ptr(), x.data_ptr(), N, P, Cc, self._st()))
        return out, idx

    def maxpool_bwd(self, dout, idx, P):
        self._req(dout)
        dout = dout if dout.is_contiguous() else self.ewise("COPY", dout)
        N, Cc = dout.shape
        dx = self.empty((N, P, Cc))
        self._chk(self.L.seqpan_t_maxpool_bwd(dx.data_ptr(), dout.data_ptr(), idx.data_ptr(), N, P, Cc, self._st()))
        return dx

    def sumsq(self, x, accum, deterministic=False):
        if deterministic:
            nb = self.L.seqpan_t_sumsq_det_scratch_bytes(x.numel())
            scratch = self._scratch(nb)
            self._chk(self.L.seqpan_t_sumsq_det(x.data_ptr(), x.numel(), accum.data_ptr(), scratch.data_ptr(), nb, self._st()))
        else:
            self._chk(self.L.seqpan_t_sumsq(x.data_ptr(), x.numel(), accum.data_ptr(), self._st()))

    def adamw(self, p, g, m, v, hp, sumsq, dyn=None):
        self._chk(self.L.seqpan_t_adamw(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), C.byref(hp),
                                        sumsq.data_ptr() if sumsq is not None else None,
                                        dyn.data_ptr() if dyn is not None else None, self._st()))


# ---------------------------------------------------------------------------------------------------------------------
# reverse-mode tape
# ---------------------------------------------------------------------------------------------------------------------
class Var:
    __slots__ = ("v", "g", "needs", "own")

    def __init__(self, v, needs=False):
        self.v, self.g, self.needs, self.own = v, None, needs, False


class SeqpanTape:
    """Records the training forward of SeqPAN; ``backward`` replays the adjoint rules in reverse order.

    ``precision="bf16"``: the model's matrix products (``linear`` y / dx / dW, the forward ``bmm``, the six products of
    ``attention``, the char-CNN window products) and their adjoints run with bf16 operands and fp32 accumulation; ones-vector
    reductions, bias gradients, the loss functions, LayerNorm, softmax, element-wise ops and the optimizer stay fp32 -- the
    autocast policy.  ``"fp32"`` calls ``backend.gemm`` exactly as before the mode existed (no ``mixed`` keyword).

    ``deterministic=True``: every reduction of the backward that the default kernels combine with float atomics (split-K
    products, LayerNorm dgamma / dbeta, depthwise-conv dw, embedding scatter-add) gets ``deterministic=True`` and runs on the
    fixed-order kernels; ``False`` passes no such keyword."""

    def __init__(self, backend, droprate=0.0, training=True, mask_fn=None, precision="fp32", deterministic=False):
        self.be = backend
        self.p = float(droprate) if training else 0.0
        self.mask_fn = mask_fn          # optional: (shape) -> keep-mask tensor of 0/1 (parity tests inject the oracle's draws)
        self.nodes = []
        self.mm = {"mixed": True} if _check_precision(precision) == "bf16" else {}    # keywords of a model product's be.gemm
        self.det = {"deterministic": True} if deterministic else {}                    # keywords of a reduction's backend call

    # -- bookkeeping --
    def leaf(self, t, needs=False):
        return Var(t, needs)

    def _rec(self, out_v, inputs, bwd):
        needs = any(i.needs for i in inputs)
        out = Var(out_v, needs)
        if needs:
            self.nodes.append((out, inputs, bwd))
        return out

    def _acc(self, var, g):
        if g is None or not var.needs:
            return
        if tuple(g.shape) != tuple(var.v.shape):
            g = g.reshape(var.v.shape)
        if var.g is None:
            var.g, var.own = g, False      # may alias the gradient of a sibling (a + b hands the same tensor to both)
        elif not var.own:
            var.g, var.own = self.be.ewise("AXPBY", var.g, g, alpha=1.0, beta=1.0), True      # first sum: a tensor of its own
        else:
            self.be.ewise("AXPBY", var.g, g, out=var.g, alpha=1.0, beta=1.0)

    def backward(self, out, gout=None):
        """Reverse sweep from ``out`` with cotangent ``gout``, or from several outputs at once: ``out`` a list of
        ``(Var, cotangent)`` pairs, where a pair whose cotangent is None contributes nothing.  Cotangents are only read."""
        for o, g in ([(out, gout)] if isinstance(out, Var) else out):
            self._acc(o, g)
        for o, inputs, bwd in reversed(self.nodes):
            if o.g is None:
                continue
            grads = bwd(o.g)
            for i, g in zip(inputs, grads):
                self._acc(i, g)
            o.g = None          # free interior gradients as soon as they are consumed
        self.nodes = []

    # -- primitives (forward rule + vector-Jacobian rule) --
    def linear(self, x, W, b=None):
        """``Conv1D`` with kernel 1 (models/layers.py:15-26): y = x W^T + b; W is the conv weight [N, K, 1] (or [N, K])."""
        be = self.be
        K, N = x.v.shape[-1], W.v.shape[0]
        x2, W2 = x.v.reshape(-1, K), W.v.reshape(N, K)
        M = x2.shape[0]
        y = be.gemm(x2, W2.t(), bias=b.v.reshape(N) if b is not None else None, **self.mm)
        sk = 1 if M < 1024 else min(64, max(1, M // 128))     # K-splits of the two long reductions (dW, db): fill the 148 SMs

        def bwd(g):
            g2 = g.reshape(M, N)
            dx = be.gemm(g2, W2, **self.mm).reshape(x.v.shape) if x.needs else None
            dW = be.gemm(g2.t(), x2, splitk=sk, **self.mm, **self.det).reshape(W.v.shape) if W.needs else None
            db = be.gemm(be.ones(M).reshape(1, M), g2, splitk=sk, **self.det).reshape(b.v.shape) if (b is not None and b.needs) else None
            return (dx, dW, db) if b is not None else (dx, dW)
        return self._rec(y.reshape(tuple(x.v.shape[:-1]) + (N,)), [x, W] + ([b] if b is not None else []), bwd)

    def layernorm(self, x, g, b, eps):
        be = self.be
        xc = x.v if x.v.is_contiguous() else be.ewise("COPY", x.v)
        y = be.layernorm(xc, g.v, b.v, eps)

        def bwd(gy):
            dx, dg, db = be.layernorm_bwd(xc, gy, g.v, eps, **self.det)
            return dx, dg, db
        return self._rec(y, [x, g, b], bwd)

    def add(self, a, b):
        """a + b with b broadcastable to a (bias / position-table adds); the adjoint of a broadcast is a sum."""
        be = self.be
        y = be.ewise("AXPBY", a.v, b.v, alpha=1.0, beta=1.0)

        def bwd(g):
            return g, self._sum_to(g, b.v.shape) if b.needs else None
        return self._rec(y, [a, b], bwd)

    def _sum_to(self, g, shape):
        """Sum ``g`` down to ``shape`` (leading dims dropped and/or size-1 dims kept): ones-vector GEMMs."""
        be = self.be
        shape = tuple(shape)
        if tuple(g.shape) == shape:
            return g
        g = g if g.is_contiguous() else be.ewise("COPY", g)
        lead = g.dim() - len(shape)
        if lead > 0:                                   # drop leading dims: [outer, inner] -> [inner]
            outer = 1
            for s in g.shape[:lead]:
                outer *= s
            inner = g.numel() // outer
            g = be.gemm(be.ones(outer).reshape(1, outer), g.reshape(outer, inner), splitk=min(64, max(1, outer // 128)),
                        **self.det).reshape(g.shape[lead:])
        for d, (gs, ss) in enumerate(zip(g.shape, shape)):
            if ss == 1 and gs != 1:                    # reduce dim d, keep it
                outer = 1
                for s in g.shape[:d]:
                    outer *= s
                inner = g.numel() // (outer * gs)
                g3 = g.reshape(outer, gs, inner)
                o = be.gemm(be.ones(gs).reshape(1, 1, gs).expand(outer, 1, gs), g3)      # [outer, 1, inner]
                g = o.reshape(tuple(g.shape[:d]) + (1,) + tuple(g.shape[d + 1:]))
        return g.reshape(shape)

    def mul(self, a, b):
        """a * b, b broadcastable to a."""
        be = self.be
        y = be.ewise("MUL", a.v, b.v)

        def bwd(g):
            da = be.ewise("MUL", g, b.v) if a.needs else None
            db = self._sum_to(be.ewise("MUL", g, a.v), b.v.shape) if b.needs else None
            return da, db
        return self._rec(y, [a, b], bwd)

    def mul_const(self, a, c):
        """a * c for a constant tensor c (masks, dropout keep-masks)."""
        be = self.be
        y = be.ewise("MUL", a.v, c)
        return self._rec(y, [a], lambda g: (be.ewise("MUL", g, c),))

    def scale(self, a, alpha, beta=0.0):
        be = self.be
        y = be.ewise("AFFINE", a.v, alpha=alpha, beta=beta)
        return self._rec(y, [a], lambda g: (be.ewise("AFFINE", g, alpha=alpha, beta=0.0),))

    def relu(self, a):
        be = self.be
        y = be.ewise("RELU", a.v)
        return self._rec(y, [a], lambda g: (be.ewise("RELU_BWD", g, y),))

    def sigmoid(self, a):
        be = self.be
        y = be.ewise("SIGMOID", a.v)
        return self._rec(y, [a], lambda g: (be.ewise("SIGMOID_BWD", g, y),))

    def mask_logits(self, a, mask):
        """models/layers.py:9-12: a + (1 - mask) * -1e30, mask a constant broadcastable tensor."""
        be = self.be
        y = be.ewise("MASK_LOGITS", a.v, mask)
        return self._rec(y, [a], lambda g: (g,))

    def add_const(self, a, c):
        be = self.be
        y = be.ewise("AXPBY", a.v, c, alpha=1.0, beta=1.0)
        return self._rec(y, [a], lambda g: (g,))

    def softmax(self, a, dim):
        be = self.be
        ac = a.v if a.v.is_contiguous() else be.ewise("COPY", a.v)
        y = be.softmax(ac, dim)
        return self._rec(y, [a], lambda g: (be.softmax_bwd(y, g, dim),))

    def bmm(self, a, b, ta=False, tb=False, keep_fp32=False):
        """Batched a @ b over <= 2 leading dims; ta / tb transpose the last two dims of an operand (a stride swap).  A ``b``
        with batch size 1 (a weight shared by the batch: w4C, w4Q, the pool weight) is broadcast; its gradient is the batch sum.
        ``keep_fp32``: a product of the loss functions, fp32 in every precision mode."""
        be = self.be
        mm = {} if keep_fp32 else self.mm
        if b.v.dim() == 3 and a.v.dim() == 3 and b.v.shape[0] == 1 and a.v.shape[0] != 1:
            b0 = b
            b = self._rec(b0.v.expand(a.v.shape[0], *b0.v.shape[1:]), [b0], lambda g: (self._sum_to(g, b0.v.shape),))
        A = a.v.transpose(-1, -2) if ta else a.v
        B = b.v.transpose(-1, -2) if tb else b.v
        y = be.gemm(A, B, **mm)

        def bwd(g):
            da = db = None
            if a.needs:
                da = be.gemm(B, g.transpose(-1, -2), **mm) if ta else be.gemm(g, B.transpose(-1, -2), **mm)
            if b.needs:
                db = be.gemm(g.transpose(-1, -2), A, **mm) if tb else be.gemm(A.transpose(-1, -2), g, **mm)
            return da, db
        return self._rec(y, [a, b], bwd)

    def dropout(self, a, channels_first=False):
        """``nn.Dropout(p)`` in training mode: keep-mask / (1 - p).  Identity when p == 0.  ``channels_first``: the reference
        applies this dropout to the ``[B, D, L]`` layout (conv block, models/layers.py:144-147): the mask is drawn in that
        element order and viewed back, so that an injected stream of draws lands on the same elements."""
        if self.p <= 0.0:
            return a
        shape = tuple(a.v.shape)
        if channels_first:
            shape = (shape[0], shape[2], shape[1])
        be = self.be
        if self.mask_fn is not None:      # a test injects the oracle's draws as a 0/1 keep-mask
            r = self.mask_fn(shape)
            if channels_first:
                r = r.transpose(1, 2)
            sc = 1.0 / (1.0 - self.p)
            y = be.ewise("DROPOUT", a.v, r, alpha=0.5, beta=sc)
            return self._rec(y, [a], lambda g: (be.ewise("DROPOUT", g, r, alpha=0.5, beta=sc),))
        m = be.dropout_mask(shape, self.p)
        if channels_first:
            m = m.transpose(1, 2)
        return self.mul_const(a, m)

    def dwconv(self, a, w, seg_len):
        be = self.be
        ac = a.v if a.v.is_contiguous() else be.ewise("COPY", a.v)
        y = be.dwconv(ac, w.v, seg_len, False)

        def bwd(g):
            gc = g if g.is_contiguous() else be.ewise("COPY", g)
            return (be.dwconv(gc, w.v, seg_len, True) if a.needs else None,
                    be.dwconv_bwd_w(ac, gc, seg_len, **self.det) if w.needs else None)
        return self._rec(y, [a, w], bwd)

    def cat_last(self, parts):
        be = self.be
        widths = [p.v.shape[-1] for p in parts]
        out = be.empty(tuple(parts[0].v.shape[:-1]) + (sum(widths),))
        off = 0
        for p, wd in zip(parts, widths):
            be.ewise("COPY", p.v, out=out[..., off:off + wd])
            off += wd

        def bwd(g):
            res, o = [], 0
            for p, wd in zip(parts, widths):
                res.append(g[..., o:o + wd] if p.needs else None)
                o += wd
            return res
        return self._rec(out, list(parts), bwd)

    def embedding(self, table, ids):
        be = self.be
        y = be.gather_rows(table.v, ids)
        return self._rec(y, [table], lambda g: (be.scatter_add_rows(g.reshape(-1, g.shape[-1]), ids, table.v.shape[0], **self.det),))

    def maxpool_mid(self, a):
        be = self.be
        P = a.v.shape[1]
        y, idx = be.maxpool(a.v if a.v.is_contiguous() else be.ewise("COPY", a.v))
        return self._rec(y, [a], lambda g: (be.maxpool_bwd(g, idx, P),))

    def reshape(self, a, shape):
        v = a.v.reshape(shape)
        return self._rec(v, [a], lambda g: (g.reshape(a.v.shape),))

    def transpose(self, a, d0, d1):
        v = a.v.transpose(d0, d1)
        return self._rec(v, [a], lambda g: (g.transpose(d0, d1),))

    def sum_all(self, a):
        be = self.be
        ac = a.v if a.v.is_contiguous() else be.ewise("COPY", a.v)
        n = ac.numel()
        y = be.gemm(be.ones(n).reshape(1, n), ac.reshape(n, 1), splitk=min(64, max(1, n // 2048)), **self.det).reshape(())
        return self._rec(y, [a], lambda g: (g.reshape((1,) * a.v.dim()).expand(a.v.shape),))

    def log(self, a):
        be = self.be
        y = be.ewise("LOG", a.v)
        return self._rec(y, [a], lambda g: (be.ewise("DIV", g, a.v),))

    def sqrt(self, a):
        be = self.be
        y = be.ewise("SQRT", a.v)
        return self._rec(y, [a], lambda g: (be.ewise("DIV", be.ewise("AFFINE", g, alpha=0.5), y),))

    def norm2(self, a):
        """Frobenius / 2-norm of all elements (torch.norm(x, p=2)); the adjoint is g x / ||x||, 0 at the origin."""
        be = self.be
        ac = a.v if a.v.is_contiguous() else be.ewise("COPY", a.v)
        n = ac.numel()
        sq = be.ewise("MUL", ac, ac)
        y = be.ewise("SQRT", be.gemm(be.ones(n).reshape(1, n), sq.reshape(n, 1))).reshape(())
        return self._rec(y, [a], lambda g: (be.ewise("MUL", be.ewise("DIV_SAFE", ac, y.reshape((1,) * ac.dim())), g.reshape((1,) * ac.dim())),))

    def div(self, a, b):
        """a / b, b broadcastable (used with scalars)."""
        be = self.be
        y = be.ewise("DIV", a.v, b.v)

        def bwd(g):
            da = be.ewise("DIV", g, b.v) if a.needs else None
            db = None
            if b.needs:
                t = be.ewise("DIV", be.ewise("MUL", g, y, alpha=-1.0), b.v)
                db = self._sum_to(t, b.v.shape)
            return da, db
        return self._rec(y, [a, b], bwd)

    # -- attention core shared by DualMultiAttention and TopSelfAttention2: softmax(q k^T * scale + mask) v, heads as strides --
    def attention(self, q, k, v, add_mask, scale, q_heads, k_heads, out_shape, out_heads):
        """q / k / v: Vars holding [*, 128]-wide rows; ``*_heads(t)`` returns the 4-D head view ``[b0, b1, rows, 32]`` of a
        tensor (a pure stride view); ``add_mask`` is an additive constant broadcastable to the scores ``[b0, b1, F, S]``.
        Dropout acts on the attention probabilities (models/layers.py:352,357; nn.MultiheadAttention's own dropout)."""
        be = self.be
        qh, kh, vh = q_heads(q.v), k_heads(k.v), k_heads(v.v)
        s = be.gemm(qh, kh.transpose(-1, -2), alpha=scale, **self.mm)
        s = be.ewise("AXPBY", s, add_mask, out=s, alpha=1.0, beta=1.0)
        p = be.softmax(s, -1)
        pd, r, thr, dsc = p, None, 0.5, 1.0
        if self.p > 0.0:
            if self.mask_fn is not None:
                r, dsc = self.mask_fn(p.shape), 1.0 / (1.0 - self.p)
            else:                           # the reference's own F.dropout call on the probabilities (0 or 1/(1-p) per element)
                r, thr, dsc = be.dropout_mask(p.shape, self.p), 0.5, 1.0
            pd = be.ewise("DROPOUT", p, r, alpha=thr, beta=dsc) if self.mask_fn is not None else be.ewise("MUL", p, r)
        out = be.empty(out_shape)
        be.gemm(pd, vh, out=out_heads(out), **self.mm)

        def bwd(g):
            gh = out_heads(g if g.is_contiguous() else be.ewise("COPY", g))
            dv = torch.zeros_like(v.v)
            be.gemm(pd.transpose(-1, -2), gh, out=k_heads(dv), **self.mm)
            dpd = be.gemm(gh, vh.transpose(-1, -2), **self.mm)
            if r is None:
                dp = dpd
            elif self.mask_fn is not None:
                dp = be.ewise("DROPOUT", dpd, r, alpha=thr, beta=dsc)
            else:
                dp = be.ewise("MUL", dpd, r)
            ds = be.softmax_bwd(p, dp, -1)
            dq, dk = torch.zeros_like(q.v), torch.zeros_like(k.v)
            be.gemm(ds, kh, out=q_heads(dq), alpha=scale, **self.mm)
            be.gemm(ds.transpose(-1, -2), qh, out=k_heads(dk), alpha=scale, **self.mm)
            return dq, dk, dv
        return self._rec(out, [q, k, v], bwd)


# ---------------------------------------------------------------------------------------------------------------------
# the model: reference forward in training mode, primitive by primitive
# ---------------------------------------------------------------------------------------------------------------------
class _Params:
    """Leaf Vars of the module's parameters by state_dict key (frozen ones: needs = False)."""

    def __init__(self, tape, named):
        self.vars = {k: tape.leaf(t.detach(), needs=bool(t.requires_grad)) for k, t in named.items()}

    def __getitem__(self, k):
        return self.vars[k]

    def has(self, k):
        return k in self.vars


def _conv1d(tp, P, prefix, x):
    return tp.linear(x, P[prefix + ".conv1d.weight"], P[prefix + ".conv1d.bias"])


def _ln(tp, P, prefix, x, eps):
    return tp.layernorm(x, P[prefix + ".weight"], P[prefix + ".bias"], eps)


def _text_embedding(tp, P, word_ids, char_ids):
    # models/layers.py:42-48, 65-75, 87-93
    be = tp.be
    B, T = word_ids.shape
    Cc = char_ids.shape[2]
    p = "text_encoder"
    if P.has(p + ".word_emb.glove_vec"):
        # cat[pad, unk, glove] rebuilt per call in the reference; only unk_vec is trainable: its gradient is the sum of the
        # output gradients of the words with id 1
        table = torch.cat([P[p + ".word_emb.pad_vec"].v, P[p + ".word_emb.unk_vec"].v, P[p + ".word_emb.glove_vec"].v], dim=0)
        wv = be.gather_rows(table, word_ids.reshape(-1).contiguous())
        unk = P[p + ".word_emb.unk_vec"]
        is_unk = (word_ids.reshape(-1) == 1).to(torch.float32)
        w = tp._rec(wv.reshape(B, T, -1), [unk], lambda g: (be.gemm(is_unk.reshape(1, -1), g.reshape(-1, g.shape[-1])),))
    else:
        w = tp.embedding(P[p + ".word_emb.word_emb.weight"], word_ids.reshape(-1).contiguous())
        w = tp.reshape(w, (B, T, -1))
        # nn.Embedding(padding_idx=0): row 0 receives no gradient -- the ids are never 0 for real words and the pad rows'
        # output gradient is scattered into row 0, which the optimizer step must ignore (_zero_pad_rows)
    w = tp.dropout(w)
    ce = tp.embedding(P[p + ".char_emb.char_emb.weight"], char_ids.reshape(-1).contiguous())     # [B*T*C, 100]
    ce = tp.dropout(ce)
    ce_c = ce.v if ce.v.is_contiguous() else be.ewise("COPY", ce.v)
    R = B * T * Cc
    outs = []
    for i, (k, ch) in enumerate(zip((1, 2, 3, 4), (10, 20, 30, 40))):
        Wk, bk = P[f"{p}.char_emb.char_convs.{i}.0.weight"], P[f"{p}.char_emb.char_convs.{i}.0.bias"]      # [ch,100,1,k]
        npos = Cc - k + 1
        # Conv2d(100 -> ch, (1,k)) over the characters of a word = one 2-D product over ALL character rows: window r is the
        # k*100 contiguous floats starting at row r (a stride view with row stride 100: rows overlap); windows that run into
        # the next word are computed and discarded (positions >= npos of every word), and get a zero gradient on the way back
        Rk = R - k + 1
        win = ce_c.as_strided((Rk, k * 100), (100, 1), ce_c.storage_offset())
        Wp2 = be.ewise("COPY", Wk.v.reshape(ch, 100, k).permute(0, 2, 1)).reshape(ch, k * 100)       # (o, j, i) order
        yfull = be.zeros((R, ch))
        be.gemm(win, Wp2.t(), out=yfull[:Rk], **tp.mm)
        y = be.ewise("AXPBY", yfull.reshape(B * T, Cc, ch)[:, :npos, :], bk.v.reshape(1, 1, ch), alpha=1.0, beta=1.0)   # [B*T, npos, ch]

        def bwd(g, win=win, Wp2=Wp2, Wk=Wk, k=k, ch=ch, npos=npos, Rk=Rk):
            gfull = be.zeros((B * T, Cc, ch))
            be.ewise("COPY", g, out=gfull[:, :npos, :])
            g2 = gfull.reshape(R, ch)
            dce = None
            if ce.needs:
                dwin = be.gemm(g2[:Rk], Wp2, **tp.mm)                                               # [Rk, k*100]
                dce = be.zeros((R, 100))
                for j in range(k):                       # overlapping windows add up: k shifted accumulations
                    be.ewise("AXPBY", dce[j:j + Rk], dwin[:, j * 100:(j + 1) * 100], out=dce[j:j + Rk], alpha=1.0, beta=1.0)
            dWp = be.gemm(g2[:Rk].t(), win, splitk=min(64, max(1, Rk // 128)), **tp.mm, **tp.det)   # [ch, k*100]
            dW = be.ewise("COPY", dWp.reshape(ch, k, 100).permute(0, 2, 1)).reshape(Wk.v.shape)
            db = be.gemm(be.ones(R).reshape(1, R), g2, splitk=min(64, max(1, R // 128)), **tp.det).reshape(ch)
            return dce, dW, db
        yk = tp._rec(y, [ce, Wk, bk], bwd)
        outs.append(tp.maxpool_mid(tp.relu(yk)))                       # [B*T, ch]
    cfeat = tp.reshape(tp.cat_last(outs), (B, T, 100))
    emb = tp.cat_last([w, cfeat])
    emb = _conv1d(tp, P, p + ".query_conv1d", emb)
    return _ln(tp, P, p + ".q_layer_norm", emb, 1e-6)


def _conv_block(tp, P, prefix, x):
    # models/layers.py:139-148
    out = x
    Lx = x.v.shape[1]
    i = 0
    while P.has(f"{prefix}.layer_norms.{i}.weight"):
        res = out
        out = _ln(tp, P, f"{prefix}.layer_norms.{i}", out, 1e-6)
        out = tp.dwconv(out, P[f"{prefix}.depthwise_separable_conv.{i}.0.weight"], Lx)
        out = tp.linear(out, P[f"{prefix}.depthwise_separable_conv.{i}.1.weight"], P[f"{prefix}.depthwise_separable_conv.{i}.1.bias"])
        out = tp.dropout(tp.relu(out), channels_first=True)
        out = tp.add(out, res)
        i += 1
    return out


def _feature_encoder(tp, P, prefix, x):
    # models/layers.py:396-399 (+ :102-107)
    X = x.v.shape[1]
    pos_full = P[prefix + ".pos_embedding.position_embeddings.weight"]
    pos = tp._rec(pos_full.v[:X], [pos_full], lambda g: (torch.cat([g, torch.zeros_like(pos_full.v[X:])], dim=0),))
    return _conv_block(tp, P, prefix + ".conv_block", tp.add(x, pos))


def _heads_bx(t):            # [B, X, 128] -> [B, 4, X, 32] (stride view)
    B, X, _ = t.shape
    return t.view(B, X, H, HD).permute(0, 2, 1, 3)


def _pair_mask(tp, m_a, m_b):
    """(1 - m_a[b,i] m_b[b,j]) * -1e30 as ``[B,1,Fa,Fb]``, built once per (mask pair) of a step by the element-wise kernel."""
    cache = tp.__dict__.setdefault("_pair_masks", {})
    key = (m_a.data_ptr(), m_b.data_ptr())
    if key not in cache:
        be = tp.be
        outer = be.ewise("MUL", m_a.unsqueeze(2), m_b.unsqueeze(1))
        cache[key] = be.ewise("AFFINE", outer, alpha=-MASKV, beta=MASKV).unsqueeze(1)
    return cache[key]


def _dual_multi_attention(tp, P, p, o, u, m_f, m_t):
    # models/layers.py:336-381 (BiLinear :257-263 applies dense_1 to both inputs)
    B, Fl, _ = o.v.shape
    q = _conv1d(tp, P, p + ".query", o)
    fk, fv = _conv1d(tp, P, p + ".f_key", o), _conv1d(tp, P, p + ".f_value", o)
    tk, tv = _conv1d(tp, P, p + ".t_key", u), _conv1d(tp, P, p + ".t_value", u)
    s_add = _pair_mask(tp, m_f, m_f)        # [B,1,F,F] additive constants: (1 - m_f (x) m_f) * -1e30 (create_attention_mask, :235-244)
    x_add = _pair_mask(tp, m_f, m_t)        # [B,1,F,S]
    sc = 1.0 / math.sqrt(float(HD))
    s = tp.attention(q, fk, fv, s_add, sc, _heads_bx, _heads_bx, (B, Fl, D), _heads_bx)
    x = tp.attention(q, tk, tv, x_add, sc, _heads_bx, _heads_bx, (B, Fl, D), _heads_bx)
    s = _conv1d(tp, P, p + ".s_dense", s)
    x = _conv1d(tp, P, p + ".x_dense", x)
    z = tp.add(tp.mul(_conv1d(tp, P, p + ".s_gate", s), x), tp.mul(_conv1d(tp, P, p + ".x_gate", x), s))
    z = _conv1d(tp, P, p + ".guided_dense", z)
    scores = tp.add(tp.add(_conv1d(tp, P, p + ".bilinear_1.dense_1", o), _conv1d(tp, P, p + ".bilinear_1.dense_1", z)),
                    P[p + ".bilinear_1.bias_value"])
    values = tp.add(tp.add(_conv1d(tp, P, p + ".bilinear_2.dense_1", o), _conv1d(tp, P, p + ".bilinear_2.dense_1", z)),
                    P[p + ".bilinear_2.bias_value"])
    return tp.mul(tp.sigmoid(tp.mask_logits(scores, m_f.unsqueeze(2))), values)


def _dual_attention_block(tp, P, p, f, g, m_f, m_g):
    # models/layers.py:281-297
    o = tp.dropout(_ln(tp, P, p + ".layer_norm_1", f, 1e-6))
    u = _ln(tp, P, p + ".layer_norm_t", g, 1e-6)
    y = _dual_multi_attention(tp, P, p + ".dual_multihead_attention", o, u, m_f, m_g)
    r = tp.add(tp.dropout(_conv1d(tp, P, p + ".dense_1", y)), f)
    out = tp.dropout(_ln(tp, P, p + ".layer_norm_2", r, 1e-6))
    return tp.add(tp.dropout(_conv1d(tp, P, p + ".dense_2", out)), r)


def _cq_attention(tp, P, p, c, q, m_c, m_q):
    # models/layers.py:417-437
    cd, qd = tp.dropout(c), tp.dropout(q)                                # trilinear_attention's dropout (:431-432)
    s0 = tp.bmm(cd, tp.reshape(P[p + ".w4C"], (1, D, 1)))                # [B,Lc,1]      (weight broadcast over the batch)
    s1 = tp.transpose(tp.bmm(qd, tp.reshape(P[p + ".w4Q"], (1, D, 1))), 1, 2)     # [B,1,Lq]
    s2 = tp.bmm(tp.mul(cd, tp.reshape(P[p + ".w4mlu"], (1, 1, D))), qd, tb=True)  # [B,Lc,Lq]
    score = tp.add(tp.add(s2, s0), s1)
    row = tp.softmax(tp.mask_logits(score, m_q.unsqueeze(1)), 2)
    col = tp.softmax(tp.mask_logits(score, m_c.unsqueeze(2)), 1)         # softmax over the context axis
    c2q = tp.bmm(row, q)
    q2c = tp.bmm(tp.bmm(row, col, tb=True), c)
    out = tp.cat_last([c, c2q, tp.mul(c, c2q), tp.mul(c, q2c)])
    return _conv1d(tp, P, p + ".cqa_linear", out)


def _cq_concatenate(tp, P, p, c, q, m_q):
    # models/layers.py:447-453, 462-468
    B, Lc, _ = c.v.shape
    alpha = tp.bmm(q, tp.reshape(P[p + ".weighted_pool.weight"], (1, D, 1)))          # [B,T,1]
    alpha = tp.softmax(tp.mask_logits(alpha, m_q.unsqueeze(2)), 1)
    pooled = tp.bmm(q, alpha, ta=True)                                                 # [B,128,1]
    pooled = tp.transpose(pooled, 1, 2)                                                # [B,1,128]
    tiled = tp._rec(pooled.v.expand(B, Lc, D), [pooled], lambda g: (tp._sum_to(g, pooled.v.shape),))
    return _conv1d(tp, P, p + ".conv1d", tp.cat_last([c, tiled]))


def _heads_lb(t):            # [B, L, 128] -> [L, 4, B, 32]: attention ACROSS the batch for every position (SURVEY.md section 0 #8)
    B, L, _ = t.shape
    return t.view(B, L, H, HD).permute(1, 2, 0, 3)


def _batch_axis_attention(tp, P, p, a, vmask):
    # TopSelfAttention2 (models/layers.py:567-574): nn.MultiheadAttention(batch_first=False) on [B,L,D]
    B, L, _ = a.v.shape
    Win, bin_ = P[p + ".in_proj_weight"], P[p + ".in_proj_bias"]
    qkv = tp.linear(a, Win, bin_)                                           # [B,L,384]
    parts = []
    for i in range(3):
        sl = tp._rec(qkv.v[..., i * D:(i + 1) * D], [qkv],
                     lambda g, i=i: (_embed_cols(tp.be, g, qkv.v.shape, i * D),))
        parts.append(sl)
    add = vmask.t().reshape(L, 1, 1, B)                                     # + vmask[b', l]: float key_padding_mask is ADDED
    o = tp.attention(parts[0], parts[1], parts[2], add, math.sqrt(1.0 / HD), _heads_lb, _heads_lb, (B, L, D), _heads_lb)
    return tp.linear(o, P[p + ".out_proj.weight"], P[p + ".out_proj.bias"])


def _embed_cols(be, g, shape, off):
    out = be.zeros(shape)
    be.ewise("COPY", g, out=out[..., off:off + g.shape[-1]])
    return out


def _feature_encoder_predict(tp, P, p, x, vmask):
    # models/layers.py:626-639 (layer_norm_1/2: default eps 1e-5)
    h = _feature_encoder(tp, P, p, x)
    a = tp.dropout(_ln(tp, P, p + ".layer_norm_1", h, 1e-5))
    r = tp.add(tp.dropout(_batch_axis_attention(tp, P, p + ".top_self_attention.selfattn", a, vmask)), h)
    out = tp.dropout(_ln(tp, P, p + ".layer_norm_2", r, 1e-5))
    return tp.add(tp.dropout(_conv1d(tp, P, p + ".dense", out)), r)


def _predictor(tp, P, x, vmask):
    # models/layers.py:659-671
    p = "predictor"
    s = _feature_encoder_predict(tp, P, p + ".feature_encoder", x, vmask)
    e = _feature_encoder_predict(tp, P, p + ".feature_encoder", s, vmask)
    s = _ln(tp, P, p + ".start_layer_norm", s, 1e-6)
    e = _ln(tp, P, p + ".end_layer_norm", e, 1e-6)
    s = _conv1d(tp, P, p + ".start_hidden", tp.cat_last([s, x]))
    e = _conv1d(tp, P, p + ".end_hidden", tp.cat_last([e, x]))
    B, L, _ = x.v.shape
    return (tp.reshape(_conv1d(tp, P, p + ".start_dense", s), (B, L)), tp.reshape(_conv1d(tp, P, p + ".end_dense", e), (B, L)))


def forward_train(tp, P, word_ids, char_ids, vfeat_in, vmask, tmask, gumbel, dual_blocks=True, text_encoder="vfeat_encoder",
                  match_head=True):
    """``SeqPAN.forward`` in training mode (models/SeqPAN.py:50-95) on the tape; returns Vars
    ``(slogits [B,L], elogits [B,L], match_score [B,L,4])``.  ``vfeat_in`` is a tensor (a constant of the tape) or a leaf Var
    (``tp.leaf(v, needs=True)``: its ``.g`` holds the gradient of the video features after ``backward``).
    ``dual_blocks=False``: ``BaseFast.forward`` (models/BaseFast.py:49-97: the two DualAttentionBlock passes are commented out
    there; its 2-layer encoder is read off the parameters -- so is MultiTeacher's, models/MultiTeacher.py:26).  ``text_encoder="tfeat_encoder"``, ``match_head=False``: ``BackBone.forward``
    (models/BackBone.py:40-75: the text has its own FeatureEncoder, the CQConcatenate output feeds the predictor directly and
    unmasked; ``match_score`` is None)."""
    t = _text_embedding(tp, P, word_ids, char_ids)                                   # :56
    v = tp.dropout(vfeat_in if isinstance(vfeat_in, Var) else tp.leaf(vfeat_in))      # VisualProjection.drop (:119)
    v = _ln(tp, P, "video_affine.v_layer_norm", _conv1d(tp, P, "video_affine.video_conv1d", v), 1e-6)   # :57
    v = _feature_encoder(tp, P, "vfeat_encoder", v)                                  # :59
    t = _feature_encoder(tp, P, text_encoder, t)                                     # :60 (shared weights; BackBone.py:49: its own)
    for blk in (("dual_attention_block_1", "dual_attention_block_2") if dual_blocks else ()):   # :64-70
        v_ = _dual_attention_block(tp, P, blk, v, t, vmask, tmask)
        t_ = _dual_attention_block(tp, P, blk, t, v, tmask, vmask)
        v, t = v_, t_
    t2v = _cq_attention(tp, P, "q2v_attn", v, t, vmask, tmask)                       # :73
    v2t = _cq_attention(tp, P, "v2q_attn", t, v, tmask, vmask)                       # :74
    fuse = _cq_concatenate(tp, P, "cq_cat", t2v, v2t, tmask)                         # :75
    if not match_head:                                                               # models/BackBone.py:62-63
        slogits, elogits = _predictor(tp, P, fuse, vmask)
        return slogits, elogits, None
    ml = _conv1d(tp, P, "match_conv1d", fuse)                                        # :78
    B, L = vmask.shape
    if gumbel is None:            # drawn HERE, where the reference draws it: after the encoder / attention dropouts, before the predictor's
        gumbel = tp.be.gumbel((B, L, 4))
    ms = tp.softmax(tp.scale(tp.add_const(ml, gumbel), 1.0 / 0.3), -1)               # :79 gumbel_softmax(tau = 0.3)
    soft = tp.reshape(tp.bmm(tp.reshape(ms, (1, B * L, 4)), tp.reshape(P["label_embs"], (1, D, 4)), tb=True), (B, L, D))   # :81
    fuse = tp.mul_const(tp.add(fuse, soft), vmask.unsqueeze(2))                      # :82
    slogits, elogits = _predictor(tp, P, fuse, vmask)                                # :83
    return slogits, elogits, ms


# What differs between the reference's train engines (forward variant + loss terms), by module class name:
#   SeqPAN       models/SeqPAN.py:171-182        location loss + match loss
#   BaseFast     models/BaseFast.py:113-127      no DualAttentionBlock passes; sigmoid(logits) into the location loss; + match loss
#   MultiTeacher models/MultiTeacher.py:165-195  sigmoid(logits) into the location loss, NO match loss (commented out, :175); runtype
#                                                "train" adds three teacher terms (lossfun_softloc weighted by calculate_adapt_cof)
#   BackBone     models/BackBone.py:94-107       own text encoder, no match head; location loss only
_TRAIN_SPECS = {
    "SeqPAN": dict(fwd=dict(dual_blocks=True), sigmoid_first=False, match_loss=True, teachers=False),
    "BaseFast": dict(fwd=dict(dual_blocks=False), sigmoid_first=True, match_loss=True, teachers=False),
    "MultiTeacher": dict(fwd=dict(dual_blocks=True), sigmoid_first=True, match_loss=False, teachers=True),
    "BackBone": dict(fwd=dict(dual_blocks=True, text_encoder="tfeat_encoder", match_head=False), sigmoid_first=False,
                     match_loss=False, teachers=False),
}


def train_spec(model):
    name = type(model).__name__
    if name not in _TRAIN_SPECS:
        raise NotImplementedError(f"no training step for {name} (SeqPAN, BaseFast, MultiTeacher, BackBone)")
    return _TRAIN_SPECS[name]


def _record_forward(model, be, named, inputs, gumbel, precision, training, mask_fn=None, needs_x=False):
    """The model's training forward recorded on a new tape: ``inputs`` are ``(word_ids, char_ids, vfeat_in, vmask, tmask)``,
    ``named`` the parameters by name (those that require grad receive a gradient), and ``vfeat_in`` receives one when
    ``needs_x``.  The tape reduces in a fixed order while :func:`deterministic_mode` is on.  Returns ``(tape, params, video
    leaf, (slogits, elogits, match_score or None))``."""
    tp = SeqpanTape(be, droprate=model.configs.model.droprate, training=training, mask_fn=mask_fn, precision=precision,
                    deterministic=deterministic_mode())
    P = _Params(tp, named)
    word_ids, char_ids, vfeat_in, vmask, tmask = inputs
    xv = tp.leaf(vfeat_in, needs=needs_x)
    return tp, P, xv, forward_train(tp, P, word_ids, char_ids, xv, vmask, tmask, gumbel, **train_spec(model)["fwd"])


_EMB_PAD_ROW = ("text_encoder.char_emb.char_emb.weight", "text_encoder.word_emb.word_emb.weight")


def _zero_pad_rows(P):
    """nn.Embedding(padding_idx=0): row 0 of the embedding tables gets no gradient."""
    for k in _EMB_PAD_ROW:
        if P.has(k) and P[k].g is not None:
            P[k].g[0].zero_()


# ---- losses (models/loss.py:24-54) -------------------------------------------------------------------------------------
def loss_loc(tp, slogits, elogits, s_labels, e_labels, sigmoid_first=False):
    """``nn.CrossEntropyLoss(reduction='mean')`` with soft ``[B,L]`` targets on the UNMASKED logits, start + end.
    ``sigmoid_first``: ``train_engine_BaseFast`` feeds ``torch.sigmoid(logits)`` to the loss (models/BaseFast.py:119-120)."""
    B = slogits.v.shape[0]
    total = None
    for lg, lab in ((slogits, s_labels), (elogits, e_labels)):
        if sigmoid_first:
            lg = tp.sigmoid(lg)
        lp = tp.log(tp.softmax(lg, 1))
        term = tp.scale(tp.sum_all(tp.mul_const(lp, lab)), -1.0 / B)
        total = term if total is None else tp.add(total, term)
    return total


def loss_match(tp, match_score, label_embs, ner_labels, vmask):
    """-sum(onehot * probs) masked mean + || offdiag(E^T E) ||_2 (models/loss.py:24-41)."""
    be = tp.be
    onehot = torch.nn.functional.one_hot(ner_labels, 4).to(torch.float32)             # constant
    w = be.ewise("MUL", onehot, vmask.unsqueeze(2))
    n = vmask.numel()
    denom = be.ewise("AFFINE", be.gemm(be.ones(n).reshape(1, n), vmask.reshape(n, 1)), alpha=1.0, beta=1e-12).reshape(())
    per = tp.scale(tp.div(tp.sum_all(tp.mul_const(match_score, w)), tp.leaf(denom)), -1.0)
    E = label_embs
    G = tp.bmm(tp.reshape(E, (1, D, 4)), tp.reshape(E, (1, D, 4)), ta=True, keep_fp32=True)   # [1,4,4] = E^T E
    off = tp.mul_const(G, (1.0 - torch.eye(4, device=vmask.device)).reshape(1, 4, 4))
    return tp.add(per, tp.norm2(off))


def _soft_dist(tp, x, temperature):
    """``softmax(F.normalize(x, p=2, dim=1) / temperature, dim=-1)`` of a ``[B,L]`` Var (models/loss.py:187-190)."""
    B, L = x.v.shape
    n = tp.sqrt(tp.bmm(tp.reshape(tp.mul(x, x), (1, B, L)), tp.leaf(tp.be.ones(L).reshape(1, L, 1)), keep_fp32=True))   # row norms [1,B,1]
    n = tp.scale(tp.relu(tp.scale(n, 1.0, -1e-12)), 1.0, 1e-12)                                          # F.normalize: clamp_min(eps)
    return tp.softmax(tp.scale(tp.div(x, tp.reshape(n, (B, 1))), 1.0 / temperature), 1)


def adapt_cof(t_label, gt_label):
    """``calculate_adapt_cof`` (models/MultiTeacher.py:151-159) + ``iou_batch`` (utils/utils.py:169-177): IoU of the teacher's
    argmax span with the ground truth's, one value per sample.  Label preprocessing ([B] integers), not part of the tape."""
    ts, te = t_label[:, 0].argmax(1), t_label[:, 1].argmax(1)
    gs, ge = gt_label[:, 0].argmax(1), gt_label[:, 1].argmax(1)
    inter = torch.minimum(te, ge) - torch.maximum(ts, gs)
    union = torch.maximum(te, ge) - torch.minimum(ts, gs)
    return torch.clamp(inter / union, min=0.0, max=1.0).to(torch.float32)


def loss_softloc(tp, s, e, s_lab, e_lab, vmask, temperature, row_weight):
    """``mean_b(row_weight[b] * lossfun_softloc(s, e, s_lab, e_lab, vmask, T)[b])`` (models/loss.py:180-199 as used by
    models/MultiTeacher.py:181-182): KL(teacher || student) of temperature softmaxes over L2-normalised rows.

    The reference normalises AFTER ``mask_logits``: a clip with padding carries a -1e30 entry, its fp32 row norm overflows to
    inf, both distributions collapse to uniform and the sample contributes exactly 0 -- value and gradient.  The same thing is
    stated here as a row weight (0 for clips with padding) instead of being left to inf arithmetic."""
    be = tp.be
    B, L = s.v.shape
    full = (vmask.sum(1) == L).to(torch.float32)
    w = (row_weight * full).reshape(B, 1)
    n = B * L
    total = None
    for x, lab in ((s, s_lab), (e, e_lab)):
        q = _soft_dist(tp, tp.leaf(lab.contiguous()), temperature).v              # teacher side: constants through the same kernels
        wq = be.ewise("MUL", q, w)
        lp = tp.log(_soft_dist(tp, x, temperature))
        # sum_l q (log q - log p): the first half is a constant of the batch
        c = be.gemm(be.ones(n).reshape(1, n), be.ewise("MUL", wq, be.ewise("LOG", q)).reshape(n, 1)).reshape(())
        term = tp.add_const(tp.scale(tp.sum_all(tp.mul_const(lp, wq)), -1.0 / B), be.ewise("AFFINE", c, alpha=1.0 / B))
        total = term if total is None else tp.add(total, term)
    return total


def compose_loss(tp, model, sl, el, ms, label_embs, data, vmask, runtype="train"):
    """The loss of the reference's ``train_engine_<Model>`` from the forward outputs (Vars), per ``_TRAIN_SPECS``."""
    spec = train_spec(model)
    lab = data["label1ds"].to(torch.float32)
    s_, e_ = (tp.sigmoid(sl), tp.sigmoid(el)) if spec["sigmoid_first"] else (sl, el)
    loss = loss_loc(tp, s_, e_, lab[:, 0, :], lab[:, 1, :])
    if spec["match_loss"]:
        loss = tp.add(loss, loss_match(tp, ms, label_embs, data["NER_labels"], vmask))
    if spec["teachers"] and runtype == "train":                            # models/MultiTeacher.py:179-193
        cfg = model.configs.loss
        for k in range(3):
            t = data[f"label1d_t{k}s"].to(torch.float32)
            kd = loss_softloc(tp, s_, e_, t[:, 0, :], t[:, 1, :], vmask, float(getattr(cfg, f"t{k}_temperature")), adapt_cof(t, lab))
            loss = tp.add(loss, tp.scale(kd, float(getattr(cfg, f"t{k}_cof"))))
    return loss


def loss_from_outputs(model, output, data, runtype="train", backend=None):
    """Loss VALUE (no graph) of a forward that already ran -- what the train engines return for a module in ``eval()``
    (main.py:112-127 logs it): the same loss kernels on the inference outputs."""
    vmask = data["vmasks"].to(torch.float32)
    tp = SeqpanTape(backend if backend is not None else CudaBackend(vmask.device), training=False)
    ms = tp.leaf(output["match_score"]) if "match_score" in output else None
    le = tp.leaf(output["label_embs"].detach()) if "label_embs" in output else None
    return compose_loss(tp, model, tp.leaf(output["slogits"]), tp.leaf(output["elogits"]), ms, le, data, vmask, runtype).v


# ---- one optimisation step ---------------------------------------------------------------------------------------------
class TrainStep:
    """``zero_grad(); loss.backward(); clip_grad_norm_(params, 1.0); optimizer.step(); scheduler.step()`` of main.py:93-97 for a
    ``vmrframe_b200.SeqPAN`` module, with the reference's AdamW groups and linear warm-up schedule (utils/utils.py:87-97).
    With an initialised process group the live gradients are summed over the ranks in ONE flat bucket and divided by the
    world size before clipping (data parallel, one batch of ``B`` pairs per rank)."""

    def __init__(self, model, lr=1e-4, warmup_proportion=0.0, num_train_steps=1, weight_decay=0.01, clip_norm=1.0, backend=None,
                 mask_fn=None, precision=None):
        self.model = model
        self.precision = train_precision(model, precision)      # "fp32" or "bf16" (mixed: bf16 products, fp32 everything else)
        self.named = {k: p for k, p in model.named_parameters()}
        dev = next(model.parameters()).device
        self.be = backend if backend is not None else CudaBackend(dev)
        self.live = None                     # names that received a gradient (the reference's 20 dead tensors never do)
        self.lr, self.wd, self.clip = lr, weight_decay, clip_norm
        self.warm, self.total = int(num_train_steps * warmup_proportion), int(num_train_steps)
        self.t = 0
        self.m, self.v = {}, {}
        self.mask_fn = mask_fn
        self.runtype = "train"                # MultiTeacher: the teacher terms enter the loss for runtype "train" only
        self.flat = None
        self.dyn = None                      # device float[3]: lr, 1 - beta1^t, sqrt(1 - beta2^t) of the current step
        self._graphs = collections.OrderedDict()     # graph key -> entry, least recently used first
        self.max_graphs = GRAPH_CACHE_SIZE           # captured entries kept (each holds its activations' memory pool)
        self._g2 = {}                        # deterministic mode -> the clip + AdamW half: {"seen", "graph", "out"}
        self.views = {}

    def _lr_now(self):
        # transformers.get_linear_schedule_with_warmup, stepped AFTER the optimizer (main.py:96-97): optimisation step n (1-based,
        # self.t while it runs) uses lr * lambda(n - 1)
        s = self.t - 1
        if s < self.warm:
            f = float(s) / float(max(1, self.warm))
        else:
            f = max(0.0, float(self.total - s) / float(max(1, self.total - self.warm)))
        return self.lr * f

    def loss_and_grads(self, data, gumbel=None):
        """Forward + both losses + backward.  Returns ``(loss tensor (device scalar), {name: grad}, outputs)``."""
        m = self.model
        vmask, tmask = data["vmasks"].to(torch.float32), data["tmasks"].to(torch.float32)
        tp, P, _, (sl, el, ms) = _record_forward(m, self.be, self.named, (data["words_ids"], data["char_ids"], data["vfeats"], vmask,
                                                                          tmask), gumbel, self.precision, m.training, self.mask_fn)
        loss = compose_loss(tp, m, sl, el, ms, P["label_embs"] if train_spec(m)["match_loss"] else None, data, vmask, self.runtype)
        tp.backward(loss, torch.ones((), dtype=torch.float32, device=vmask.device))
        _zero_pad_rows(P)
        grads = {k: v.g for k, v in P.vars.items() if v.g is not None}
        out = {"slogits": sl.v, "elogits": el.v, "vmask": data["vmasks"]}
        if ms is not None:
            out.update(match_score=ms.v, label_embs=m.label_embs)
        return loss.v, grads, out

    def _scalars(self):
        lr = self._lr_now() if self.total > 1 else self.lr
        return [lr, 1.0 - 0.9 ** self.t, math.sqrt(1.0 - 0.999 ** self.t)]

    def _part1(self, data, gumbel, relayout=False):
        """Forward + losses + backward; the live gradients land in ONE flat bucket (``self.flat``).  ``relayout``: a changed set
        of live gradients gets a new bucket instead of an error (the train engines, where parameters may be frozen between
        steps; every captured graph keeps the bucket it writes in its entry)."""
        be = self.be
        loss, grads, out = self.loss_and_grads(data, gumbel)
        names = sorted(grads)
        if self.live is None or (relayout and names != self.live):
            self.live, self.views = names, {}
            self.flat = be.zeros((sum(grads[k].numel() for k in names),))
            off = 0
            for k in names:
                n = grads[k].numel()
                self.views[k] = self.flat[off:off + n]
                off += n
        assert names == self.live, "the set of parameters that receive a gradient changed between steps"
        for k in names:
            g = grads[k]
            be.ewise("COPY", (g if g.is_contiguous() else be.ewise("COPY", g)).reshape(-1), out=self.views[k])
        return loss, out

    def _allreduce(self):
        """Data parallel: ONE all-reduce of the flat bucket per step.  Always issued eagerly, never from inside a captured
        graph: every rank then enqueues exactly one collective per step no matter which of its input shapes are already captured
        (ranks see different batch shapes, so their capture schedules differ)."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            return dist.get_world_size()
        return 1

    def _part2(self, world, det):
        """Mean over the ranks, squared norm for clip_grad_norm_, AdamW on every live tensor (scalars of the step from ``self.dyn``)."""
        be = self.be
        if world > 1:
            be.ewise("AFFINE", self.flat, out=self.flat, alpha=1.0 / world, beta=0.0)
        ss = torch.zeros((), dtype=torch.float64, device=self.flat.device)
        be.sumsq(self.flat, ss, **({"deterministic": True} if det else {}))
        for k in self.live:
            p = self.named[k]
            if k not in self.m:
                self.m[k], self.v[k] = torch.zeros_like(p.data), torch.zeros_like(p.data)
            hp = _cabi.SeqpanAdamW()
            no_decay = any(nd in k for nd in ("bias", "layer_norm", "LayerNorm"))
            hp.lr, hp.beta1, hp.beta2, hp.eps = self.lr, 0.9, 0.999, 1e-8
            hp.weight_decay = 0.0 if no_decay else self.wd
            hp.bias1, hp.bias2_sqrt = 1.0, 1.0
            hp.max_grad_norm = self.clip
            be.adamw(p.data, self.views[k], self.m[k], self.v[k], hp, ss, self.dyn)
        return ss

    # -- CUDA graphs of forward + losses + backward, one per graph key, least recently used evicted first --
    def _graph_key(self, route, data, gumbel, precision, *extra):
        """Everything a captured forward + backward bakes in: the route, the input shapes and dtypes, whether a Gumbel draw is
        given, the deterministic mode, the precision, ``model.training`` and its droprate, and for every parameter whether it
        requires grad and where its storage is (a re-created parameter must not replay a graph that reads the old one)."""
        m = self.model
        return ((route,) + tuple((k, tuple(v.shape), v.dtype) for k, v in sorted(data.items()))
                + (gumbel is not None, deterministic_mode(), precision, m.training, float(m.configs.model.droprate))
                + tuple((k, p.requires_grad, p.data_ptr()) for k, p in self.named.items()) + extra)

    def _entry(self, key):
        """The cache entry of ``key`` (``{"seen": eager runs}`` at first), moved to the most recently used end."""
        ent = self._graphs.pop(key, None)
        self._graphs[key] = ent = ent if ent is not None else {"seen": 0}
        return ent

    def _use_graph(self, ent):
        """Whether ``ent`` replays (and is captured first if need be): once :func:`_due`, and when a capture fits.  At most
        ``max_graphs`` entries hold graphs; the least recently used one without a forward in flight gives its graphs and pool
        up (its eager count stays).  When every capture holds a forward in flight the call runs eagerly."""
        if "graph" in ent:
            return True
        if not _due(ent):
            return False
        captured = [e for e in self._graphs.values() if "graph" in e]
        while len(captured) >= self.max_graphs:
            old = next((e for e in captured if not e.get("busy")), None)
            if old is None:
                return False
            captured.remove(old)
            for k in [k for k in old if k != "seen"]:
                del old[k]
        return True

    def _engine_loss_and_grads(self, data, gumbel):
        """``loss_and_grads`` of the train engines, replayed from a CUDA graph from the third call with the same key on.  A
        replay hands out views of a fresh copy of the entry's bucket and fresh copies of the outputs: they outlive the next
        replay, so gradients of two calls can be accumulated before one backward.  The entry keeps the bucket its graph
        writes (a later eager call may lay out a new one)."""
        ent = self._entry(self._graph_key("loss", data, gumbel, self.precision, self.runtype))
        if not self._use_graph(ent):
            ent["seen"] += 1
            return self.loss_and_grads(data, gumbel)
        loss, out, (flat, live) = _replay(ent, lambda d, g: (*self._part1(d, g, relayout=True), (self.flat, self.live)),
                                          data, gumbel)
        grads = dict(zip(live, flat.clone().split([self.named[k].numel() for k in live])))
        out = {k: (v.clone() if k in ("slogits", "elogits", "match_score") else v) for k, v in out.items()}
        out["vmask"] = data["vmasks"]
        return loss, grads, out

    def step(self, data, gumbel=None, graph=False):
        """One optimisation step.  ``graph=True`` replays the two device halves of the step (forward + backward into the bucket;
        clip + AdamW) as CUDA graphs after two eager steps per input shape: the tape issues ~1200 small launches from Python,
        which is host-bound; the graphs keep the same kernels and remove the host.  Inputs are copied into static buffers, the
        dropout / Gumbel draws stay fresh (torch's graph-safe generator), the gradient all-reduce stays an eager call between
        the two graphs.  Graphs are kept per key (:meth:`_graph_key`: shapes, deterministic mode, precision, parameters), at
        most ``max_graphs`` of them, least recently used evicted first."""
        be = self.be
        det = deterministic_mode()
        self.t += 1
        sc = self._scalars()
        if self.dyn is None:
            self.dyn = be.zeros((3,))
            self._dyn_host = torch.zeros(3, dtype=torch.float32)
            if self.dyn.is_cuda:
                self._dyn_host = self._dyn_host.pin_memory()
        self._dyn_host.copy_(torch.tensor(sc, dtype=torch.float32))
        self.dyn.copy_(self._dyn_host, non_blocking=True)
        world = 1
        if not graph:
            loss, out = self._part1(data, gumbel)
            world = self._allreduce()
            ss = self._part2(world, det)
        else:
            ent = self._entry(self._graph_key("step", data, gumbel, self.precision, self.runtype))
            if self._use_graph(ent):
                loss, out = _replay(ent, self._part1, data, gumbel)
            else:
                ent["seen"] += 1
                loss, out = self._part1(data, gumbel)
            world = self._allreduce()
            e2 = self._g2.setdefault(det, {"seen": 0})     # outside the LRU cache and never evicted: it holds no activations
            if _due(e2):
                ss = _replay(e2, lambda d, g: self._part2(world, det), {}, None)
            else:
                e2["seen"] += 1
                ss = self._part2(world, det)
        if hasattr(self.model, "repack"):
            self.model.repack()           # the inference handle's packed weights follow the update (p.data edits bump no version)
        return loss, out, ss              # ss: squared gradient norm before clipping (device fp64 scalar)


# ---- drop-in glue: the loss tensor the reference's loop calls .backward() on ----------------------------------------------
class _TapeLoss(torch.autograd.Function):
    """The tape has already run backward (d loss = 1) when this node is built; ``loss.backward()`` in the reference's loop
    (main.py:93-94) then only hands every parameter its finished gradient, so ``clip_grad_norm_`` and any torch optimizer work
    on the module unchanged."""

    @staticmethod
    def forward(ctx, loss_value, grads, *params):
        ctx.grads = grads
        return loss_value.clone()

    @staticmethod
    def backward(ctx, gout):
        return (None, None) + tuple(g * gout if g is not None else None for g in ctx.grads)


def tape_loss(model, data, gumbel=None, mask_fn=None, runtype="train"):
    """Training forward + the model's loss terms + backward on the kernels; returns ``(loss, output)`` where ``loss`` is a scalar
    tensor attached to the module's parameters (``loss.backward()`` fills ``p.grad``).  ``runtype`` is the train engines' fourth
    argument (only MultiTeacher reads it: its teacher terms exist for "train").

    From the third call with the same key (:meth:`TrainStep._graph_key`) on, forward, losses and backward replay as one CUDA
    graph from the model's ``TrainStep`` cache; never with ``mask_fn`` or off the CUDA kernels."""
    ts = _train_step_of(model)
    named = dict(model.named_parameters())
    ts.named, ts.mask_fn, ts.runtype = named, mask_fn, runtype
    if _can_capture(ts.be, data["vfeats"], mask_fn):
        value, grads, out = ts._engine_loss_and_grads(data, gumbel)
    else:
        value, grads, out = ts.loss_and_grads(data, gumbel)
    params = [p for p in named.values() if p.requires_grad]
    glist = [grads[k].reshape(p.shape) if k in grads else None for k, p in named.items() if p.requires_grad]
    return _TapeLoss.apply(value, glist, *params), out


def _train_step_of(model):
    """The ``TrainStep`` the drop-in routes share per model: its graph cache and bound serve both."""
    ts = getattr(model, "_train_step", None)
    if ts is None:
        ts = model._train_step = TrainStep(model)
    return ts


def _can_capture(be, x, mask_fn=None):
    """Whether a drop-in route may capture and replay: the CUDA kernels on a CUDA tensor, no injected dropout masks (a
    ``mask_fn`` hands in host-made draws) and no capture of the caller's already under way."""
    return (getattr(be, "graph_safe", False) and x.is_cuda and mask_fn is None
            and not torch.cuda.is_current_stream_capturing())


# ---- the training forward as one torch autograd node: any torch loss on its outputs backpropagates through the tape ----------
class _Recording:
    """What the node's backward needs: the tape, its nodes as the forward left them, its output Vars, the video leaf and the
    parameter Vars.  The tape's nodes are closures over the tape (a reference cycle); clearing them when the recording dies
    lets reference counting free a forward that is never backpropagated as soon as its outputs are dropped, as it frees
    :func:`forward_only`'s."""
    __slots__ = ("tp", "nodes", "outs", "xv", "P")

    def __init__(self, tp, P, xv, outs):
        self.tp, self.nodes, self.outs, self.xv, self.P = tp, tp.nodes, [o for o in outs if o is not None], xv, P

    def __del__(self):
        self.tp.nodes = []


class _InFlight:
    """Marks a graph entry's forward as in flight while the node that replayed it can still be backpropagated: a forward of
    the same key meanwhile runs on the eager tape, since a replay would overwrite the activations this backward reads."""
    __slots__ = ("ent",)

    def __init__(self, ent):
        self.ent = ent
        ent["busy"] = True

    def __del__(self):
        self.ent["busy"] = False


def _node_backward(rec, gouts, names):
    """The tape's adjoints from the node's outputs with cotangents ``gouts`` (None: unused); returns the gradients of
    ``vfeat_in`` and of the parameters ``names``, None where there is none.  A recording swept before (a graph entry's, whose
    backward is captured once per pattern of None cotangents) gets its nodes back and the gradient state that sweep left
    cleared."""
    if rec.tp.nodes is not rec.nodes:
        for o, inputs, _ in rec.nodes:
            for v in (o, *inputs):
                v.g, v.own = None, False
        rec.tp.nodes = rec.nodes
    rec.tp.backward(list(zip(rec.outs, gouts)))
    _zero_pad_rows(rec.P)
    return [rec.xv.g] + [rec.P[k].g for k in names]


def _graphed_node_backward(ent, gouts, names):
    """:func:`_node_backward` from a graph per pattern of cotangents (which are None): the backward issues different kernels
    for each.  A graph is captured from the entry's recording on first use, in the forward graph's pool.  Cotangents are
    copied into static buffers (which makes expanded views contiguous); the gradients handed back are fresh copies."""
    bwd = ent.setdefault("bwd", {})
    bkey = tuple(g is not None for g in gouts)
    if bkey not in bwd:
        static = [None if g is None else torch.empty(g.shape, dtype=torch.float32, device=g.device) for g in gouts]
        gb = torch.cuda.CUDAGraph()
        with _capture(gb, pool=ent["graph"].pool()):
            grads = _node_backward(ent["out"], static, names)
        bwd[bkey] = (gb, static, grads)
    gb, static, grads = bwd[bkey]
    for s, g in zip(static, gouts):
        if s is not None:
            s.copy_(g)
    gb.replay()
    return [g.clone() if g is not None else None for g in grads]


class _TapeForward(torch.autograd.Function):
    """Forward: the training forward recorded on a ``SeqpanTape`` (kept on ``ctx``).  Backward: the tape's adjoints from the
    cotangents of ``slogits`` / ``elogits`` / ``match_score`` that autograd hands in, one gradient per parameter and for
    ``vfeat_in``.  Once-differentiable, and the tape frees its nodes as it runs: a second backward raises.

    The outputs are fresh views of the tape's tensors, never the tensors the tape (and so ``ctx``) holds: a returned tensor
    reachable from ``ctx`` would close the cycle output -> grad_fn -> ctx -> output, and a forward dropped without a backward
    would keep its whole tape alive until a full garbage collection.

    ``slot``: None, or ``(entry, graphed)`` of the model's graph cache.  Graphed, the forward replays the entry's graph and
    returns copies of its outputs, and the backward replays a backward graph; eager, a completed backward counts towards the
    entry's capture."""

    @staticmethod
    def forward(ctx, model, be, slot, word_ids, char_ids, vmask, tmask, gumbel, vfeat_in, names, *params):
        ctx.set_materialize_grads(False)          # an output nobody used arrives as None and costs nothing
        ctx.names, ctx.shapes = names, [vfeat_in.shape] + [p.shape for p in params]
        ent, graphed = slot if slot is not None else (None, False)
        ctx.ent = ent
        data = {"words_ids": word_ids, "char_ids": char_ids, "vmasks": vmask, "tmasks": tmask, "vfeats": vfeat_in}

        def record(d, gum):
            inputs = (d["words_ids"], d["char_ids"], d["vfeats"], d["vmasks"], d["tmasks"])
            return _Recording(*_record_forward(model, be, dict(zip(names, params)), inputs, gum, train_precision(model),
                                               model.training, needs_x=ctx.needs_input_grad[8]))
        if graphed:
            rec = _replay(ent, record, data, gumbel)
            ctx.rec = _InFlight(ent)
            return tuple(o.v.clone() for o in rec.outs)
        ctx.rec = rec = record(data, gumbel)
        return tuple(o.v.view_as(o.v) for o in rec.outs)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gouts):
        rec = ctx.rec
        if rec is None:
            raise RuntimeError("backward through the SeqPAN training forward a second time: the tape is freed by the first "
                               "backward (retain_graph is not supported); run the forward again")
        ctx.rec = None
        if isinstance(rec, _InFlight):
            grads = _graphed_node_backward(rec.ent, gouts, ctx.names)
        else:
            be = rec.tp.be
            gouts = [g if g is None or g.is_contiguous() else be.ewise("COPY", g) for g in gouts]   # e.g. .sum()'s expanded views
            grads = _node_backward(rec, gouts, ctx.names)
            # Every returned gradient must be a tensor of its own: AccumulateGrad may adopt it as p.grad and later add into it
            # in place.  The tape lets siblings share one gradient tensor (a + b) and passes cotangents through untouched, so
            # a gradient whose storage is already taken by a cotangent or an earlier gradient is copied.
            taken = {g.untyped_storage().data_ptr() for g in gouts if g is not None}
            for i, g in enumerate(grads):
                if g is not None:
                    if g.untyped_storage().data_ptr() in taken:
                        grads[i] = g = be.ewise("COPY", g)
                    taken.add(g.untyped_storage().data_ptr())
            if ctx.ent is not None:
                ctx.ent["seen"] += 1                  # one more eager forward + backward of this key
        res = [g.reshape(shape) if g is not None else None for g, shape in zip(grads, ctx.shapes)]
        return (None,) * 8 + tuple(res[:1]) + (None,) + tuple(res[1:])


def forward_differentiable(model, word_ids, char_ids, vfeat_in, vmask, tmask, gumbel=None, backend=None):
    """``SeqPAN.forward`` in training mode on the tape, as one torch autograd node: returns ``(slogits, elogits, match_score or
    None)`` attached to every parameter that requires grad and to ``vfeat_in`` when it does, so that ``loss.backward()`` of any
    torch loss on them fills ``p.grad`` / ``vfeat_in.grad`` through the training kernels.  The same kernels, in the same order,
    with the same dropout and Gumbel draws as :func:`forward_only`: the values are bit-identical.  ``backend`` defaults to the
    CUDA kernels of ``vfeat_in``'s device.

    With the default backend the node replays CUDA graphs from the model's ``TrainStep`` cache once its key (shapes, modes,
    parameters, whether ``vfeat_in`` requires grad) has completed forward and backward eagerly twice: one forward graph, and a
    backward graph per pattern of unused outputs.  While a replayed forward awaits its backward, the same key runs eagerly."""
    be = backend if backend is not None else CudaBackend(vfeat_in.device)
    named = dict(model.named_parameters())
    vm, tm, x = vmask.to(torch.float32), tmask.to(torch.float32), vfeat_in.to(torch.float32)
    slot = None
    if backend is None and _can_capture(be, x):
        ts = _train_step_of(model)
        ts.named = named
        data = {"words_ids": word_ids, "char_ids": char_ids, "vmasks": vm, "tmasks": tm, "vfeats": x}
        ent = ts._entry(ts._graph_key("node", data, gumbel, train_precision(model), x.requires_grad and torch.is_grad_enabled()))
        slot = (ent, not ent.get("busy") and ts._use_graph(ent))
    outs = _TapeForward.apply(model, be, slot, word_ids, char_ids, vm, tm, gumbel, x, tuple(named), *named.values())
    return outs if len(outs) == 3 else (outs[0], outs[1], None)


def forward_only(model, word_ids, char_ids, vfeat_in, vmask, tmask, gumbel=None):
    """``SeqPAN.forward`` in TRAINING mode (dropout active) without recording a tape: what ``model(...)`` returns when the
    module is in ``train()`` and no gradient is wanted (``torch.no_grad()`` / ``inference_mode()``, or nothing requires grad).
    :func:`forward_differentiable` is the same forward with a graph; :func:`tape_loss` / :class:`TrainStep` run forward, the
    reference's losses and backward in one call."""
    named = {k: p.detach() for k, p in model.named_parameters()}        # leaves that need no gradient: no node is recorded
    inputs = (word_ids, char_ids, vfeat_in.to(torch.float32), vmask.to(torch.float32), tmask.to(torch.float32))
    _, _, _, (sl, el, ms) = _record_forward(model, CudaBackend(vfeat_in.device), named, inputs, gumbel, train_precision(model), True)
    return sl.v, el.v, (ms.v if ms is not None else None)
