"""bf16 mixed-precision training step: ``TrainStep(precision="bf16")`` / ``configs.model.train_precision``.

The model's matrix products run on the tensor cores with bf16 operands and fp32 accumulation (csrc/train_tc.cu,
``seqpan_t_gemm_bf16``); reductions, losses, LayerNorm, softmax, element-wise ops and AdamW stay fp32.

CPU part: which GEMM calls the tape marks ``mixed``, how the mode is chosen, and the numerical effect of bf16 products
(a bf16-rounding subclass of the kernel emulation against the oracle's fp32 autograd).  GPU part: the kernel against an fp64
product of the bf16-rounded operands, the device tape against the bf16 emulation and against the oracle, the training loop,
the drop-in route, and that the fp32 step never calls the bf16 kernel."""
import ctypes as C
import math
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from cpu_train_backend import CpuEmuBackend
from test_train import DEV, _case_model, _Masks, _oracle_grads, _setup
from vmrframe_b200 import _cabi, synth, train
from vmrframe_b200.seqpan import SeqPAN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden_train import LOOP_SEED, LOOP_STEPS, LOOP_TRAIN_CFG  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TRAIN_PY = os.path.abspath(train.__file__)
# tape sites whose GEMMs are model products (forward rule and vector-Jacobian rule)
PRODUCT_SITES = {"SeqpanTape.linear", "SeqpanTape.linear.<locals>.bwd", "SeqpanTape.bmm", "SeqpanTape.bmm.<locals>.bwd",
                 "SeqpanTape.attention", "SeqpanTape.attention.<locals>.bwd", "_text_embedding", "_text_embedding.<locals>.bwd"}
LOSS_FNS = {"loss_loc", "loss_match", "loss_softloc", "_soft_dist", "compose_loss"}


def _rb(t):
    return t.to(torch.bfloat16).to(torch.float32)


class Bf16EmuBackend(CpuEmuBackend):
    """The kernel emulation with ``seqpan_t_gemm_bf16``'s semantics for ``mixed=True``: operands rounded to bf16 (nearest
    even), products summed in fp64 here.  Records every GEMM call: (keywords, caller site, tape phase, indicator operand)."""

    def __init__(self):
        self.calls = []
        self.phase = "model"

    def gemm(self, A, B, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None, **kw):
        site, phase = None, self.phase
        f = sys._getframe(1)
        while f is not None:
            if os.path.abspath(f.f_code.co_filename) == TRAIN_PY:
                site = site or f.f_code.co_qualname                 # innermost tape frame: the call site
                if f.f_code.co_name in LOSS_FNS:
                    phase = "loss"                                  # forward rule of a node of a loss function
            f = f.f_back
        indicator = A.shape[-2] == 1 and bool(((A == 0) | (A == 1)).all())       # ones / 0-1 row vectors: reductions
        self.calls.append(dict(kw=dict(kw), site=site, phase=phase, indicator=indicator))
        if kw.get("mixed"):
            A, B = _rb(A), _rb(B)
        return super().gemm(A, B, out, alpha, beta, splitk, bias)


class Bf16Fp32SumEmuBackend(Bf16EmuBackend):
    """The same bf16-rounded operands, products summed in fp32 (torch's CPU sgemm) instead of fp64: a second correct
    implementation of ``seqpan_t_gemm_bf16`` that differs from ``Bf16EmuBackend`` only in the order and width of its sums."""

    def gemm(self, A, B, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None, **kw):
        if not kw.get("mixed"):
            return super().gemm(A, B, out, alpha, beta, splitk, bias, **kw)
        y = alpha * torch.matmul(_rb(A), _rb(B))
        if bias is not None:
            y = y + bias
        if out is None:
            return y
        out.copy_(y + (beta * out if beta != 0.0 else 0.0))
        return out


# Whole-step gates between two correct bf16 implementations that differ only in the order of their fp32 sums (the device
# kernel against the fp64-sum emulation).  bf16 rounds every product operand, so a last-bit difference in an activation now and
# then moves an operand to the neighbouring bf16 value (2^-8 relative), and those flips compound through the 40-odd layers of
# forward and backward.  Two emulations on the CPU, fp32 sums against fp64 sums, differ on charades_small by 4.6e-5 in the loss,
# 1.5e-2 (1.8e-2 with dropout) in the whole gradient, cosine 0.99985, and up to 0.16 in the relative error of a tensor whose
# gradient norm exceeds 1e-3 of the largest (0.8 for predictor.start_hidden's bias at 1.1e-4 of it: a sum that cancels to a
# remainder of the size of the noise).  The gates leave about 2x of that; test_bf16_summation_order_noise_cpu pins the
# measurement, test_bf16_tape_gemms_on_device_equal_their_emulation pins every product of the step call by call.
ORDER_GATES = dict(loss=1e-4, whole=4e-2, cos=0.9995, per_tensor=0.3, floor=1e-3)


def _check_order_gates(val, grads, val_ref, ref, what):
    whole, cos, worst, name = _errors(grads, ref, floor=ORDER_GATES["floor"])
    print(f"\n{what}: loss rel {abs(val - val_ref) / abs(val_ref):.3e}, whole-gradient rel {whole:.3e}, cos {cos:.8f}, "
          f"worst per-tensor rel {worst:.3e} ({name})")
    assert abs(val - val_ref) <= ORDER_GATES["loss"] * abs(val_ref)
    assert whole <= ORDER_GATES["whole"] and cos >= ORDER_GATES["cos"], (whole, cos)
    assert worst <= ORDER_GATES["per_tensor"], (worst, name)


def _tag_phases(tp, be):
    """Tags every tape node with the phase it was recorded in ('loss' when a loss function is on the stack) and makes the
    backend see that phase while the node's vector-Jacobian rule runs (the loss functions are no longer on the stack then)."""
    rec = tp._rec

    def _rec(out_v, inputs, bwd):
        f, phase = sys._getframe(1), "model"
        while f is not None:
            if os.path.abspath(f.f_code.co_filename) == TRAIN_PY and f.f_code.co_name in LOSS_FNS:
                phase = "loss"
                break
            f = f.f_back

        def tagged(g):
            be.phase = phase
            try:
                return bwd(g)
            finally:
                be.phase = "model"
        return rec(out_v, inputs, tagged)
    tp._rec = _rec


def _tape_grads(m, batch, g, be, precision, p=0.0, mask_fn=None):
    """Loss (location + match) and gradients of the tape in ``precision`` (the objective of test_train's ``loss`` runs)."""
    tp = train.SeqpanTape(be, droprate=p, training=True, mask_fn=mask_fn, precision=precision)
    P = train._Params(tp, dict(m.named_parameters()))
    sl, el, ms = train.forward_train(tp, P, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    val = tp.add(train.loss_loc(tp, sl, el, batch["label1ds"][:, 0].contiguous(), batch["label1ds"][:, 1].contiguous()),
                 train.loss_match(tp, ms, P["label_embs"], batch["NER_labels"], batch["vmasks"]))
    tp.backward(val, torch.ones((), device=val.v.device))
    grads = {k: v.g.detach().cpu() for k, v in P.vars.items() if v.g is not None}
    grads["text_encoder.char_emb.char_emb.weight"][0] = 0        # nn.Embedding(padding_idx=0), as TrainStep does
    return float(val.v), grads


def _errors(got, want, floor=1e-4):
    """(whole-gradient relative error, cosine, worst per-tensor relative Frobenius error, its name) over the tensors whose
    reference gradient norm exceeds ``floor`` of the largest.  The others (key biases behind the shift-invariant softmax, LN and
    hidden biases of the predictor) have a true gradient that is rounding noise: a relative error means nothing for them."""
    assert set(got) == set(want)
    ks = sorted(want)
    a = torch.cat([got[k].double().reshape(-1) for k in ks])
    b = torch.cat([want[k].double().reshape(-1) for k in ks])
    norms = {k: float(want[k].double().norm()) for k in ks}
    top = max(norms.values())
    per = [(float((got[k].double() - want[k].double()).norm()) / norms[k], k) for k in ks if norms[k] > floor * top]
    worst = max(per)
    return float((a - b).norm() / b.norm()), float(a @ b / (a.norm() * b.norm())), worst[0], worst[1]


def _golden_model(name):
    from conftest import golden_case
    w, sd, batch, fx = golden_case(name)
    m = SeqPAN(synth.make_configs(w, droprate=0.0), synth.make_word_vectors(w))
    m.load_state_dict(sd)
    with torch.no_grad():      # off the orthogonal manifold: the norm term of lossfun_match has a kink at E^T E = I
        m.label_embs.add_(0.05 * torch.randn(m.label_embs.shape, generator=torch.Generator().manual_seed(1)))
    return m, synth.add_train_labels(batch), torch.from_numpy(fx["gumbel"])


# ======================================================================================================================
# CPU
# ======================================================================================================================
def test_bf16_tape_marks_exactly_the_model_products_cpu():
    w, m, batch, g = _setup()
    be = Bf16EmuBackend()
    tp = train.SeqpanTape(be, precision="bf16")
    _tag_phases(tp, be)
    counts = dict(linear=0, bmm=0, attention=0)
    for name in counts:                  # forward products of the model: one per linear / bmm node, two per attention
        orig = getattr(tp, name)

        def counted(*a, name=name, orig=orig, **kw):
            if not kw.get("keep_fp32"):
                counts[name] += 1
            return orig(*a, **kw)
        setattr(tp, name, counted)
    P = train._Params(tp, dict(m.named_parameters()))
    sl, el, ms = train.forward_train(tp, P, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    nfwd = len(be.calls)
    loss = train.compose_loss(tp, m, sl, el, ms, P["label_embs"], batch, batch["vmasks"].to(torch.float32))
    tp.backward(loss, torch.ones(()))
    marked = [c for c in be.calls if c["kw"].get("mixed")]
    assert all(c["kw"] in ({}, {"mixed": True}) for c in be.calls)
    # the marked calls are exactly the product sites of the model, and nothing from a reduction or a loss function
    for c in be.calls:
        product = c["site"] in PRODUCT_SITES and c["phase"] == "model" and not c["indicator"]
        assert bool(c["kw"].get("mixed")) == product, c
    assert not any(c["indicator"] or c["phase"] == "loss" for c in marked)
    fwd_marked = sum(1 for c in be.calls[:nfwd] if c["kw"].get("mixed"))
    assert fwd_marked == counts["linear"] + counts["bmm"] + 2 * counts["attention"] + 4       # + the 4 char-CNN window products
    assert counts["attention"] == 2 * 2 * 2 + 2              # 2 blocks x 2 directions x 2 attentions + the predictor's 2 passes
    assert any(c["phase"] == "loss" for c in be.calls) and any(c["indicator"] for c in be.calls)
    # fp32: the same tape calls be.gemm without the keyword
    be32 = Bf16EmuBackend()
    _tape_grads(m, batch, g, be32, "fp32")
    assert len(be32.calls) == len(be.calls) and all(c["kw"] == {} for c in be32.calls)


def test_training_precision_is_chosen_by_argument_then_config_cpu(monkeypatch):
    w, m, batch, g = _setup()
    assert train.TrainStep(m, backend=CpuEmuBackend()).precision == "fp32"
    m.configs.model.train_precision = "bf16"
    assert train.TrainStep(m, backend=CpuEmuBackend()).precision == "bf16"
    assert train.TrainStep(m, backend=CpuEmuBackend(), precision="fp32").precision == "fp32"
    for bad in ("tf32", "fp16"):
        with pytest.raises(ValueError):
            train.TrainStep(m, backend=CpuEmuBackend(), precision=bad)
        m.configs.model.train_precision = bad
        with pytest.raises(ValueError):
            train.TrainStep(m, backend=CpuEmuBackend())
    del m.configs.model.train_precision
    with pytest.raises(ValueError):
        train.SeqpanTape(CpuEmuBackend(), precision="tf32")
    # the drop-in route: train_engine_SeqPAN -> tape_loss -> TrainStep(model) inherits the config's mode
    from vmrframe_b200 import train_engine_SeqPAN
    backends = []
    monkeypatch.setattr(train, "CudaBackend", lambda dev: backends.append(Bf16EmuBackend()) or backends[-1])
    m.train()
    m.configs.model.train_precision = "bf16"
    loss, _ = train_engine_SeqPAN(m, batch, SimpleNamespace(device="cpu"), "train")
    assert m._train_step.precision == "bf16" and any(c["kw"].get("mixed") for c in backends[0].calls)
    loss.backward()
    assert all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)


@pytest.mark.parametrize("case", ["charades_small", "anet_small"])
def test_bf16_products_keep_loss_and_gradient_close_to_fp32_cpu(case):
    """The numerical effect of bf16 products, on the bf16-rounding emulation against the oracle's fp32 autograd."""
    m, batch, g = _golden_model(case)
    val_o, want, _ = _oracle_grads(m, batch, g, "loss")
    val_t, got = _tape_grads(m, batch, g, Bf16EmuBackend(), "bf16")
    whole, cos, worst, name = _errors(got, want)
    assert abs(val_t - val_o) <= 1e-3 * abs(val_o)
    assert whole <= 5e-2 and cos >= 0.999, (whole, cos)
    assert worst <= 0.2, (worst, name)


# ======================================================================================================================
# GPU
# ======================================================================================================================
def _r(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed + sum(shape))) * scale


def _check_bf16_gemm(be, A, B, name, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None):
    """One seqpan_t_gemm_bf16 call against an fp64 product of the bf16-rounded operands:
    |C - ref| <= 2e-5 * |alpha| * (|A_bf16| . |B_bf16|) + 1e-6, elementwise."""
    a, b = _rb(A.cpu()).double(), _rb(B.cpu()).double()
    want = alpha * torch.matmul(a, b)
    if bias is not None:
        want = want + bias.double()
    if out is not None and beta != 0.0:
        want = want + beta * out.double()
    bound = 2e-5 * abs(alpha) * torch.matmul(a.abs(), b.abs()) + 1e-6
    got = be.gemm(A.to(DEV), B.to(DEV), out=out.to(DEV) if out is not None else None, alpha=alpha, beta=beta, splitk=splitk,
                  bias=bias.to(DEV) if bias is not None else None, mixed=True)
    err = (got.cpu().double() - want).abs()
    assert bool((err <= bound).all()), f"{name}: worst excess {float((err - bound).max()):.3e}"


def _layouts(M, N, K, seed):
    """(A, B) in the four operand layouts: A K-major or M-major, B K-major or N-major."""
    for am in ("K", "M"):
        for bm in ("K", "N"):
            A = _r(M, K, seed=seed) if am == "K" else _r(K, M, seed=seed).t()
            B = _r(N, K, seed=seed + 1).t() if bm == "K" else _r(K, N, seed=seed + 1)
            yield f"{M}x{N}x{K} A:{am} B:{bm}", A, B


@pytest.mark.gpu
def test_bf16_gemm_kernel_contract():
    be = train.CudaBackend(DEV)
    # every case of test_train.py::test_gemm_kernel_strides_batches_splitk
    A, B = _r(70, 33), _r(33, 130)
    cases = [(A, B, {}), (_r(33, 70).t(), _r(130, 33).t(), {}), (_r(5000, 40, seed=1).t(), _r(5000, 24, seed=2), {"splitk": 16}),
             (_r(1, 3000, seed=3), _r(3000, 50, seed=4), {"splitk": 8}), (_r(3, 4, 20, 32), _r(3, 4, 25, 32).transpose(-1, -2), {})]
    x = _r(3, 20, 128, seed=5)
    cases.append((_r(3, 4, 17, 20, seed=6), x.view(3, 20, 4, 32).permute(0, 2, 1, 3), {}))
    cases.append((_r(6, 9, 5, seed=7), _r(1, 5, 1, seed=8).expand(6, 5, 1), {}))
    for i, (a, b, kw) in enumerate(cases):
        _check_bf16_gemm(be, a, b, f"case {i}", **kw)
    p, v = _r(3, 4, 20, 25, seed=9), _r(3, 25, 128, seed=10)
    hv = lambda t: t.view(t.shape[0], t.shape[1], 4, 32).permute(0, 2, 1, 3)
    out = torch.zeros(3, 20, 128, device=DEV)
    be.gemm(p.to(DEV), hv(v.to(DEV)), out=hv(out), alpha=0.5, mixed=True)
    want = 0.5 * (_rb(p).double() @ hv(_rb(v)).double())
    assert torch.allclose(hv(out).cpu().double(), want, rtol=1e-5, atol=1e-5)
    _check_bf16_gemm(be, A, B, "beta", out=_r(70, 130, seed=11), beta=1.0)
    # four operand layouts over edge sizes (sparse crossing of 1, 25, 30, 100, 127, 129, 6400), K = 19197 with split-K
    shapes = [(1, 25, 30, 1), (25, 30, 100, 1), (30, 100, 127, 1), (100, 127, 129, 1), (127, 129, 1, 1), (129, 1, 25, 1),
              (6400, 128, 128, 1), (6400, 30, 25, 1), (25, 6400, 100, 1), (128, 128, 6400, 50), (100, 100, 32, 1),
              (40, 30, 19197, 16), (129, 127, 19197, 1)]
    for i, (M, N, K, sk) in enumerate(shapes):
        for name, a, b in _layouts(M, N, K, seed=20 + i):
            _check_bf16_gemm(be, a, b, name + f" splitk {sk}", splitk=sk)
    # operands off the 16-byte grid (the element-wise load path): an odd row stride, and a base pointer 4 bytes off
    big = _r(100 * 129 + 1, seed=40).to(DEV)
    _check_bf16_gemm(be, big[1:].view(100, 129), _r(129, 96, seed=41), "row stride 129")
    _check_bf16_gemm(be, big[1:1 + 100 * 128].view(100, 128), big[1:1 + 96 * 128].view(96, 128).t(), "base pointer off by 4 bytes")
    # batch strides of 0 (a weight broadcast over the batch), in both batch dims
    _check_bf16_gemm(be, _r(6, 100, 30, seed=42), _r(1, 30, 40, seed=43).expand(6, 30, 40), "batch stride 0")
    _check_bf16_gemm(be, _r(2, 3, 50, 64, seed=44), _r(1, 1, 64, 33, seed=45).expand(2, 3, 64, 33), "two batch dims, stride 0")
    # alpha != 1, beta = 1 and a bias, with split-K; bias without split-K
    _check_bf16_gemm(be, _r(70, 5000, seed=46), _r(5000, 130, seed=47), "alpha beta bias splitk", out=_r(70, 130, seed=48),
                     alpha=0.5, beta=1.0, splitk=8, bias=_r(130, seed=49))
    _check_bf16_gemm(be, _r(300, 128, seed=50), _r(200, 128, seed=51).t(), "bias", bias=_r(200, seed=52), alpha=-1.5)


@pytest.mark.gpu
def test_bf16_gemm_writes_only_its_output_view():
    be = train.CudaBackend(DEV)
    # attention heads into a slice of a wider buffer: [3, 4 heads, 20, 32] views of columns 100..227 of [3, 20, 300]
    p, v = _r(3, 4, 20, 25, seed=60), _r(3, 25, 128, seed=61)
    hv = lambda t: t.view(t.shape[0], t.shape[1], 4, 32).permute(0, 2, 1, 3)
    buf = torch.full((3, 20, 300), float("nan"), device=DEV)
    view = buf[..., 100:228]
    be.gemm(p.to(DEV), hv(v.to(DEV)), out=view.unflatten(-1, (4, 32)).permute(0, 2, 1, 3), mixed=True)
    outside = torch.cat([buf[..., :100].reshape(-1), buf[..., 228:].reshape(-1)])
    assert bool(torch.isnan(outside).all())
    want = (_rb(p).double() @ hv(_rb(v)).double()).permute(0, 2, 1, 3).reshape(3, 20, 128)
    assert torch.allclose(view.cpu().double(), want, rtol=1e-5, atol=1e-5)
    # split-K (zeroed view, atomics) into the middle columns of a row-major buffer
    buf = torch.full((70, 300), float("nan"), device=DEV)
    a, b = _r(70, 3000, seed=62), _r(3000, 130, seed=63)
    be.gemm(a.to(DEV), b.to(DEV), out=buf[:, 50:180], splitk=8, mixed=True)
    assert bool(torch.isnan(buf[:, :50]).all() and torch.isnan(buf[:, 180:]).all())
    assert torch.allclose(buf[:, 50:180].cpu().double(), _rb(a).double() @ _rb(b).double(), rtol=1e-4, atol=1e-4)


@pytest.mark.gpu
def test_bf16_gemm_rounds_to_nearest_even():
    """1 + 2^-8 + 2^-10 lies above the midpoint between the bf16 neighbours 1 and 1 + 2^-7: round-to-nearest gives
    1 + 2^-7, truncation 1.  64 such products: 64.5 against 64."""
    be = train.CudaBackend(DEV)
    A = torch.full((128, 64), 1.0 + 2.0 ** -8 + 2.0 ** -10, device=DEV)
    C_ = be.gemm(A, torch.ones(64, 16, device=DEV), mixed=True)
    assert bool((C_ == 64.5).all()), C_.unique()
    # the exact midpoint 1 + 2^-8 goes to the even neighbour 1
    C_ = be.gemm(torch.full((128, 64), 1.0 + 2.0 ** -8, device=DEV), torch.ones(64, 16, device=DEV), mixed=True)
    assert bool((C_ == 64.0).all()), C_.unique()


@pytest.mark.gpu
def test_bf16_gemm_rejects_what_the_fp32_gemm_rejects():
    L = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    a, b, c = (torch.zeros(64, device=DEV) for _ in range(3))

    def desc(**kw):
        g = _cabi.SeqpanGemm()
        g.M = g.N = g.K = 4
        g.a_rs = g.b_rs = g.c_rs = 4
        g.a_cs = g.b_cs = g.c_cs = 1
        g.batch0 = g.batch1 = 1
        g.alpha, g.beta, g.splitk = 1.0, 0.0, 1
        for k, v in kw.items():
            setattr(g, k, v)
        return g
    pa, pb, pc = a.data_ptr(), b.data_ptr(), c.data_ptr()
    bad = [(None, pb, pc, desc()), (pa, None, pc, desc()), (pa, pb, None, desc()), (pa, pb, pc, None),
           (pa, pb, pc, desc(M=-1)), (pa, pb, pc, desc(K=-2)), (pa, pb, pc, desc(batch0=0)), (pa, pb, pc, desc(batch1=0)),
           (pa, pb, pc, desc(splitk=4, beta=0.5)), (pa, pb, pc, desc(splitk=4, batch0=2)), (pa, pb, pc, desc(splitk=4, c_cs=2)),
           (pa, pb, pc, desc(batch0=300, batch1=300))]
    for i, (A, B, C_, g) in enumerate(bad):
        args = (A, B, C_, None, C.byref(g) if g is not None else None, st)
        rc32 = L.seqpan_t_gemm(*args)
        e32 = L.seqpan_t_last_error()
        rc16 = L.seqpan_t_gemm_bf16(*args)
        e16 = L.seqpan_t_last_error()
        assert rc32 < 0 and rc16 == rc32 and e16 == e32, (i, rc32, rc16, e32, e16)
    # M == 0 / N == 0: nothing to do, success
    for g in (desc(M=0), desc(N=0)):
        assert L.seqpan_t_gemm(a.data_ptr(), b.data_ptr(), c.data_ptr(), None, C.byref(g), st) == 0
        assert L.seqpan_t_gemm_bf16(a.data_ptr(), b.data_ptr(), c.data_ptr(), None, C.byref(g), st) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("dropout", [False, True])
def test_bf16_summation_order_noise_cpu(dropout):
    """Two correct bf16 tapes that differ only in how their products are summed (fp32 against fp64) stay inside the gates the
    device tape is held to against the emulation -- and are further apart than a bf16 tape could ever be held to (5e-3)."""
    m, batch, g = _golden_model("charades_small")
    p = 0.2 if dropout else 0.0
    val64, g64 = _tape_grads(m, batch, g, Bf16EmuBackend(), "bf16", p=p, mask_fn=_Masks(0.2).keep if dropout else None)
    val32, g32 = _tape_grads(m, batch, g, Bf16Fp32SumEmuBackend(), "bf16", p=p, mask_fn=_Masks(0.2).keep if dropout else None)
    _check_order_gates(val32, g32, val64, g64, f"bf16 fp32-sum vs fp64-sum emulation (dropout={dropout})")
    assert _errors(g32, g64)[0] > 5e-3


class _CheckingCudaBackend(train.CudaBackend):
    """The device backend with every ``mixed`` GEMM checked, as it runs, against an fp64 product of its bf16-rounded operands."""

    def __init__(self, device):
        super().__init__(device)
        self.checked, self.worst = 0, 0.0

    def gemm(self, A, B, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None, mixed=False):
        if not mixed:
            return super().gemm(A, B, out, alpha, beta, splitk, bias)
        a, b = _rb(A.cpu()).double(), _rb(B.cpu()).double()
        want = alpha * torch.matmul(a, b)
        if bias is not None:
            want = want + bias.cpu().double()
        if out is not None and beta != 0.0:
            want = want + beta * out.cpu().double()
        bound = 2e-5 * abs(alpha) * torch.matmul(a.abs(), b.abs()) + 1e-6
        res = super().gemm(A, B, out, alpha, beta, splitk, bias, mixed=True)
        err = (res.cpu().double() - want).abs()
        assert bool((err <= bound).all()), (tuple(A.shape), tuple(B.shape), A.stride(), B.stride(), float((err - bound).max()))
        self.checked += 1
        self.worst = max(self.worst, float((err / bound).max()))
        return res


@pytest.mark.gpu
def test_bf16_tape_gemms_on_device_equal_their_emulation():
    """Every product of a bf16 training step on the device (all shapes, strides, batch broadcasts, strided outputs and
    split-K of the real tape, charades_small with dropout) equals the fp64 product of its bf16-rounded operands within the
    kernel bound -- what the emulation computes from the same operands."""
    m, batch, g = _golden_model("charades_small")
    emu = Bf16EmuBackend()
    _tape_grads(m, batch, g, emu, "bf16", p=0.2, mask_fn=_Masks(0.2).keep)
    m.to(DEV)
    bd = {k: v.to(DEV) for k, v in batch.items()}
    mg = _Masks(0.2)
    be = _CheckingCudaBackend(DEV)
    _tape_grads(m, bd, g.to(DEV), be, "bf16", p=0.2, mask_fn=lambda shape: mg.keep(shape).to(DEV))
    print(f"\n{be.checked} bf16 GEMMs of one step checked, worst error {be.worst:.3f} of the bound")
    assert be.checked == sum(1 for c in emu.calls if c["kw"].get("mixed")) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dropout", [False, True])
def test_bf16_tape_on_device_matches_the_bf16_emulation(dropout):
    """The whole step: rounding is the same on both sides, only the order of the fp32 sums differs, so the two are held to
    ORDER_GATES, the distance between two correct implementations (test_bf16_summation_order_noise_cpu)."""
    m, batch, g = _golden_model("charades_small")
    p = 0.2 if dropout else 0.0
    mc, mg = _Masks(0.2), _Masks(0.2)
    val_c, want = _tape_grads(m, batch, g, Bf16EmuBackend(), "bf16", p=p, mask_fn=mc.keep if dropout else None)
    m.to(DEV)
    bd = {k: v.to(DEV) for k, v in batch.items()}
    val_g, got = _tape_grads(m, bd, g.to(DEV), train.CudaBackend(DEV), "bf16", p=p,
                             mask_fn=(lambda shape: mg.keep(shape).to(DEV)) if dropout else None)
    _check_order_gates(val_g, got, val_c, want, f"bf16 device vs bf16 emulation (dropout={dropout})")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["charades_small", "anet_small"])
def test_bf16_tape_on_device_stays_close_to_the_fp32_oracle(case):
    m, batch, g = _golden_model(case)
    val_o, want, _ = _oracle_grads(m, batch, g, "loss")
    m.to(DEV)
    bd = {k: v.to(DEV) for k, v in batch.items()}
    val_t, got = _tape_grads(m, bd, g.to(DEV), train.CudaBackend(DEV), "bf16")
    whole, cos, worst, name = _errors(got, want)
    print(f"\nbf16 device vs fp32 oracle ({case}): loss rel {abs(val_t - val_o) / abs(val_o):.3e}, whole-gradient rel {whole:.3e}, "
          f"cos {cos:.8f}, worst per-tensor rel {worst:.3e} ({name})")
    assert abs(val_t - val_o) <= 1e-3 * abs(val_o)
    assert whole <= 5e-2 and cos >= 0.999, (whole, cos)
    assert worst <= 0.2, (worst, name)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_bf16_train_loop_on_device_follows_the_reference_loop(graph):
    """LOOP_STEPS bf16 optimisation steps against the fixture of the reference's own fp32 loop: the same learning rates, the
    loss within 1e-2 per step, and the loss falls."""
    fx = np.load(os.path.join(GOLDEN, "train_loop_seqpan.npz"))
    _, cfg, m, batch, _ = _case_model("train_seqpan")
    m.to(DEV).train()
    m.repack = lambda: None
    ts = train.TrainStep(m, weight_decay=0.01, precision="bf16", **LOOP_TRAIN_CFG)
    bd = {k: v.to(DEV) for k, v in batch.items()}
    B, L = batch["vmasks"].shape
    losses = []
    for k in range(LOOP_STEPS):
        loss, _, _ = ts.step(bd, synth.gumbel_noise(B, L, seed=LOOP_SEED + k).to(DEV), graph=graph)
        losses.append(float(loss))
        assert math.isclose(ts._lr_now(), float(fx["lrs"][k]), rel_tol=1e-6, abs_tol=1e-12)
        assert math.isclose(losses[-1], float(fx["losses"][k]), rel_tol=1e-2), (k, losses[-1], float(fx["losses"][k]))
    print(f"\nbf16 loop (graph={graph}): losses {losses}, reference {fx['losses'].tolist()}")
    assert losses[-1] < losses[0]


@pytest.mark.gpu
def test_bf16_drop_in_route_on_device():
    """train_engine_SeqPAN with configs.model.train_precision = "bf16", then loss.backward() and torch.optim.AdamW; and
    train_engine_MultiTeacher in bf16 (its teacher terms are loss functions: fp32)."""
    import vmrframe_b200 as V
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7)
    m.configs.model.train_precision = "bf16"
    m.to(DEV).train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3)
    cfg = SimpleNamespace(device=DEV)
    loss, out = V.train_engine_SeqPAN(m, batch, cfg, "train")
    assert m._train_step.precision == "bf16"
    opt.zero_grad()
    loss.backward()
    live = [k for k, p in m.named_parameters() if p.grad is not None]
    assert len(live) == 170 and all(bool(torch.isfinite(p.grad).all()) for p in m.parameters() if p.grad is not None)
    opt.step()
    variant, cfg_t, mt, batch_t, g_t = _case_model("train_multiteacher")
    mt.configs.model.train_precision = "bf16"
    mt.to(DEV).train()
    cfg_t.device = DEV
    loss_t, _ = V.train_engine_MultiTeacher(mt, batch_t, cfg_t, "train")
    assert mt._train_step.precision == "bf16" and math.isfinite(float(loss_t.detach()))
    loss_t.backward()
    assert all(bool(torch.isfinite(p.grad).all()) for p in mt.parameters() if p.grad is not None)


class _CountingLib:
    """The library handle with a call counter per entry point."""

    def __init__(self, lib):
        self._lib, self.n = lib, {}

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.n[name] = self.n.get(name, 0) + 1
            return fn(*a)
        return call


@pytest.mark.gpu
def test_fp32_step_never_calls_the_bf16_gemm():
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7)
    m.to(DEV).train()
    m.repack = lambda: None
    bd = {k: v.to(DEV) for k, v in batch.items()}
    counts = {}
    for precision in (None, "bf16"):
        be = train.CudaBackend(DEV)
        be.L = _CountingLib(be.L)
        train.TrainStep(m, backend=be, precision=precision).step(bd, g.to(DEV))
        torch.cuda.synchronize()
        counts[precision] = be.L.n
    assert counts[None].get("seqpan_t_gemm_bf16", 0) == 0 and counts[None]["seqpan_t_gemm"] > 0
    assert counts["bf16"]["seqpan_t_gemm_bf16"] > 0
