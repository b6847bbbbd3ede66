"""Deterministic training mode: ``torch.use_deterministic_algorithms(True)`` routes every reduction of a training step to the
fixed-order ``seqpan_t_*_det`` kernels (split-K GEMM in fp32 and bf16, LayerNorm dgamma / dbeta, depthwise-conv dw, embedding
scatter-add, the clipping norm) instead of float atomics.

CPU part: the routing of ``TrainStep``, the train engines and the autograd node with the flag on, off and on with
``warn_only``, and the deterministic emulation's gradients against the oracle's autograd.  GPU part: each new kernel against
its emulation (bit for bit where the order is pinned), bit-identical whole steps, eager against graph replay, the autograd
node, toggling the flag between graph-replayed steps, and accuracy against the oracle.

While the flag is on, torch fills ``torch.empty`` with NaN: scratch a kernel reads without having written shows up as NaN.
cuBLAS raises under the flag unless ``CUBLAS_WORKSPACE_CONFIG`` is set, so every torch reference here runs on the CPU."""
import ctypes as C
from types import SimpleNamespace

import pytest
import torch

from cpu_train_backend import CpuEmuBackend
from test_train import DEV, _compare, _Masks, _oracle_grads, _setup
from test_train_autograd import _golden_model, _reference_losses
from test_train_bf16 import Bf16EmuBackend, _check_order_gates, _rb
from test_train_bf16 import _tape_grads as _bf16_tape_grads
from vmrframe_b200 import _cabi, train

GT, TB_K = 16, 64          # K granularity of a K-split: seqpan_t_gemm (fp32) / seqpan_t_gemm_bf16


@pytest.fixture
def flag():
    """Sets torch's deterministic-algorithms flag for one test: ``flag(on, warn_only=False)``; restored afterwards."""
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield lambda on, warn_only=False: torch.use_deterministic_algorithms(on, warn_only=warn_only)
    torch.use_deterministic_algorithms(was, warn_only=warn)


# ---- emulation of the deterministic kernels (their ordering contracts, include/seqpan_b200.h) -------------------------------
def ordered_splitk(A, B, split, kstep, alpha=1.0, bias=None):
    """alpha * (((p0 + p1) + p2) + ...) + bias over the K ranges of seqpan_t_gemm's splits, partials summed in fp32."""
    K = A.shape[-1]
    kc = ((K + split - 1) // split + kstep - 1) // kstep * kstep
    s = None
    for k in range(split):
        p = torch.matmul(A[:, k * kc:(k + 1) * kc].double(), B[k * kc:(k + 1) * kc].double()).float()
        s = p if s is None else s + p
    y = alpha * s
    return y + bias if bias is not None else y


def ordered_scatter(dtable, dout, ids, rows):
    """seqpan_t_scatter_add_rows_det: per row, 0 + the rows of dout whose clamped id hits it in ascending n, added once."""
    acc = torch.zeros(rows, dout.shape[-1])
    hit = torch.zeros(rows, dtype=torch.bool)
    for n, r in enumerate(ids.clamp(0, rows - 1).tolist()):
        acc[r] += dout[n]
        hit[r] = True
    dtable[hit] += acc[hit]
    return dtable


class DetEmuBackend(CpuEmuBackend):
    """The kernel emulation with the deterministic keywords: ordered split-K partials and the ordered scatter-add.  Records
    every reduction-capable call as (method, effective split-K, keywords)."""

    def __init__(self):
        self.calls = []

    def gemm(self, A, B, out=None, alpha=1.0, beta=0.0, splitk=1, bias=None, **kw):
        sk = splitk if A.dim() == 2 and (out is None or out.stride(-1) == 1) else 1      # CudaBackend.gemm's rule
        self.calls.append(("gemm", sk, dict(kw)))
        if kw.get("mixed"):
            A, B = _rb(A), _rb(B)
        if not (kw.get("deterministic") and sk > 1):
            return super().gemm(A, B, out, alpha, beta, splitk, bias)
        y = ordered_splitk(A, B, sk, TB_K if kw.get("mixed") else GT, alpha, bias)
        if out is None:
            return y
        out.copy_(y + (beta * out if beta != 0.0 else 0.0))
        return out

    def layernorm_bwd(self, x, dy, g, eps, **kw):
        self.calls.append(("layernorm_bwd", 1, dict(kw)))
        with torch.enable_grad():            # also inside the autograd node's backward
            return super().layernorm_bwd(x, dy, g, eps)

    def dwconv_bwd_w(self, x, dy, seg_len, **kw):
        self.calls.append(("dwconv_bwd_w", 1, dict(kw)))
        with torch.enable_grad():
            return super().dwconv_bwd_w(x, dy, seg_len)

    def scatter_add_rows(self, dout, ids, rows, **kw):
        self.calls.append(("scatter_add_rows", 1, dict(kw)))
        if kw.get("deterministic"):
            return ordered_scatter(torch.zeros(rows, dout.shape[-1]), dout.reshape(-1, dout.shape[-1]), ids.reshape(-1), rows)
        return super().scatter_add_rows(dout, ids, rows)

    def sumsq(self, x, accum, **kw):
        self.calls.append(("sumsq", 1, dict(kw)))
        super().sumsq(x, accum)


def _check_routing(calls, det, step):
    """det: no split-K > 1 product and no atomic LayerNorm / dwconv / scatter / sumsq call; off: no deterministic keyword."""
    names = {c[0] for c in calls}
    assert {"layernorm_bwd", "dwconv_bwd_w", "scatter_add_rows"} <= names and ("sumsq" in names) == step
    assert any(c[0] == "gemm" and c[1] > 1 for c in calls)          # the step has split-K products to route
    for name, sk, kw in calls:
        if not det:
            assert "deterministic" not in kw, (name, sk, kw)
        elif name != "gemm" or sk > 1:
            assert kw.get("deterministic") is True, (name, sk, kw)


# ======================================================================================================================
# CPU
# ======================================================================================================================
@pytest.mark.parametrize("mode", ["off", "on", "warn_only"])
def test_mode_follows_the_torch_flag_cpu(flag, mode):
    flag(mode != "off", warn_only=mode == "warn_only")
    assert train.deterministic_mode() is (mode != "off")


@pytest.mark.parametrize("entry", ["train_step", "train_engine", "autograd_node"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["off", "on", "warn_only"])
def test_reductions_are_routed_by_the_flag_cpu(flag, monkeypatch, mode, precision, entry):
    w, m, batch, g = _setup(B=4, L=256, T=7, Cc=6, droprate=0.2)      # B * L = 1024 rows: the linear layers' dW use split-K
    m.configs.model.train_precision = precision
    m.train()
    be = DetEmuBackend()
    flag(mode != "off", warn_only=mode == "warn_only")
    if entry == "train_step":
        train.TrainStep(m, backend=be).step(batch, g)
    elif entry == "train_engine":            # train_engine_SeqPAN -> tape_loss -> TrainStep(model)
        from vmrframe_b200 import train_engine_SeqPAN
        monkeypatch.setattr(train, "CudaBackend", lambda dev: be)
        loss, _ = train_engine_SeqPAN(m, batch, SimpleNamespace(device="cpu"), "train")
        loss.backward()
    else:
        sl, el, ms = train.forward_differentiable(m, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"],
                                                  batch["tmasks"], g, backend=be)
        (sl.sum() + el.sum() + ms.sum()).backward()
    _check_routing(be.calls, mode != "off", entry == "train_step")
    assert any(c[2].get("mixed") for c in be.calls) == (precision == "bf16")


def _det_tape_grads(m, batch, g, be, precision="fp32", p=0.0, mask_fn=None):
    """Loss (location + match) and gradients of a deterministic tape."""
    tp = train.SeqpanTape(be, droprate=p, training=True, mask_fn=mask_fn, precision=precision, deterministic=True)
    P = train._Params(tp, dict(m.named_parameters()))
    sl, el, ms = train.forward_train(tp, P, batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"], g)
    val = tp.add(train.loss_loc(tp, sl, el, batch["label1ds"][:, 0].contiguous(), batch["label1ds"][:, 1].contiguous()),
                 train.loss_match(tp, ms, P["label_embs"], batch["NER_labels"], batch["vmasks"]))
    tp.backward(val, torch.ones((), device=val.v.device))
    grads = {k: v.g.detach().cpu() for k, v in P.vars.items() if v.g is not None}
    grads["text_encoder.char_emb.char_emb.weight"][0] = 0        # nn.Embedding(padding_idx=0), as TrainStep does
    return float(val.v), grads


@pytest.mark.parametrize("dropout", [0.0, 0.2])
def test_deterministic_emulation_matches_oracle_autograd_cpu(dropout):
    m, batch, g = _golden_model("charades_small")
    drop = _Masks(0.2).oracle_drop if dropout else None
    val_o, want, _ = _oracle_grads(m, batch, g, "loss", drop=drop)
    be = DetEmuBackend()
    val_t, got = _det_tape_grads(m, batch, g, be, p=dropout, mask_fn=_Masks(0.2).keep if dropout else None)
    assert any(c[0] == "gemm" and c[1] > 1 and c[2].get("deterministic") for c in be.calls)
    assert abs(val_t - val_o) <= 1e-5 * abs(val_o)
    _compare(got, want, rtol=1e-3)


def test_ordered_scatter_emulation_sums_in_ascending_order_cpu():
    """The pinned order is visible: 1 + 2^-24 + 2^-24 is 1 in fp32 summed left to right, 1 + 2^-23 when the small terms go first."""
    dout = torch.tensor([[1.0], [2.0 ** -24], [2.0 ** -24]])
    assert float(ordered_scatter(torch.zeros(1, 1), dout, torch.zeros(3, dtype=torch.int64), 1)) == 1.0
    assert float(ordered_scatter(torch.zeros(1, 1), dout.flip(0), torch.zeros(3, dtype=torch.int64), 1)) == 1.0 + 2.0 ** -23


# ======================================================================================================================
# GPU
# ======================================================================================================================
def _r(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed + sum(shape))) * scale


def _gemm_cases():
    """The split-K cases of test_train.py::test_gemm_kernel_strides_batches_splitk and test_train_bf16.py's contract test."""
    yield "dW 5000", _r(5000, 40, seed=1).t(), _r(5000, 24, seed=2), dict(splitk=16)
    yield "ones-vector", _r(1, 3000, seed=3), _r(3000, 50, seed=4), dict(splitk=8)
    for i, (M, N, K, sk) in enumerate([(128, 128, 6400, 50), (40, 30, 19197, 16)]):
        seed = 28 + i if K == 6400 else 31
        for am in ("K", "M"):
            for bm in ("K", "N"):
                A = _r(M, K, seed=seed) if am == "K" else _r(K, M, seed=seed).t()
                B = _r(N, K, seed=seed + 1).t() if bm == "K" else _r(K, N, seed=seed + 1)
                yield f"{M}x{N}x{K} A:{am} B:{bm}", A, B, dict(splitk=sk)
    yield "alpha beta bias", _r(70, 5000, seed=46), _r(5000, 130, seed=47), dict(splitk=8, alpha=0.5, beta=1.0, bias=_r(130, seed=49),
                                                                              out=_r(70, 130, seed=48))


def _want(A, B, mixed, alpha=1.0, beta=0.0, bias=None, out=None, **_):
    a, b = (_rb(A).double(), _rb(B).double()) if mixed else (A.double(), B.double())
    y = alpha * torch.matmul(a, b)
    if bias is not None:
        y = y + bias.double()
    if out is not None and beta != 0.0:
        y = y + beta * out.double()
    return y, abs(alpha) * torch.matmul(a.abs(), b.abs())


def _dev(kw):
    return {k: (v.to(DEV) if isinstance(v, torch.Tensor) else v) for k, v in kw.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", [False, True])
def test_deterministic_splitk_gemm_is_accurate_and_bit_identical(flag, mixed):
    """Within the existing bounds against an fp64 product (of the bf16-rounded operands for bf16): fp32 5e-5 of the largest
    element (test_train.py), bf16 2e-5 * |A||B| + 1e-6 per element (test_train_bf16.py); repeated launches, and launches next to
    unrelated split-K work on another stream, are bit-identical."""
    flag(True)
    be = train.CudaBackend(DEV)
    side = torch.cuda.Stream(DEV)
    noise_a, noise_b = torch.randn(2048, 8192, device=DEV), torch.randn(8192, 512, device=DEV)
    for name, A, B, kw in _gemm_cases():
        want, mag = _want(A, B, mixed, **kw)
        runs = []
        for r in range(3):
            k = _dev(kw)
            if r == 2:                        # unrelated atomic split-K products on another stream, overlapping this launch
                side.wait_stream(torch.cuda.current_stream(DEV))
                with torch.cuda.stream(side):
                    for _ in range(4):
                        be.gemm(noise_a, noise_b, splitk=32, mixed=mixed)
            runs.append(be.gemm(A.to(DEV), B.to(DEV), mixed=mixed, deterministic=True, **k).cpu())
        torch.cuda.synchronize()
        err = (runs[0].double() - want).abs()
        if mixed:
            assert bool((err <= 2e-5 * mag + 1e-6).all()), f"{name}: worst excess {float((err - 2e-5 * mag - 1e-6).max()):.3e}"
        else:
            assert float(err.max()) <= 5e-5 * max(1.0, float(want.abs().max())), name
        assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2]), name


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", [False, True])
def test_deterministic_gemm_writes_only_its_view_and_rejects_what_the_gemm_rejects(flag, mixed):
    flag(True)
    be = train.CudaBackend(DEV)
    a, b = _r(70, 3000, seed=62), _r(3000, 130, seed=63)
    want, _ = _want(a, b, mixed)
    for beta in (0.0, 1.0):
        buf = torch.full((70, 300), float("nan"), device=DEV)
        buf[:, 50:180] = 0.25
        be.gemm(a.to(DEV), b.to(DEV), out=buf[:, 50:180], beta=beta, splitk=8, mixed=mixed, deterministic=True)
        assert bool(torch.isnan(buf[:, :50]).all() and torch.isnan(buf[:, 180:]).all())
        assert torch.allclose(buf[:, 50:180].cpu().double(), want + 0.25 * beta, rtol=1e-4, atol=1e-4)
    L = _cabi.lib()
    det = L.seqpan_t_gemm_bf16_det if mixed else L.seqpan_t_gemm_det
    st = torch.cuda.current_stream().cuda_stream
    x = torch.zeros(64, device=DEV)
    scratch = torch.empty(1 << 20, device=DEV)

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
    p = x.data_ptr()
    bad = [(None, p, p, desc()), (p, None, p, desc()), (p, p, None, desc()), (p, p, p, None), (p, p, p, desc(M=-1)),
           (p, p, p, desc(K=-2)), (p, p, p, desc(batch0=0)), (p, p, p, desc(batch1=0)), (p, p, p, desc(splitk=4, beta=0.5)),
           (p, p, p, desc(splitk=4, batch0=2)), (p, p, p, desc(splitk=4, c_cs=2)), (p, p, p, desc(batch0=300, batch1=300))]
    for i, (A, B, C_, g) in enumerate(bad):
        gp = C.byref(g) if g is not None else None
        rc = L.seqpan_t_gemm(A, B, C_, None, gp, st)
        e = L.seqpan_t_last_error()
        rcd = det(A, B, C_, None, gp, scratch.data_ptr(), scratch.numel() * 4, st)
        assert rc < 0 and rcd == rc and L.seqpan_t_last_error() == e, (i, rc, rcd)
    g = desc(splitk=4)
    assert L.seqpan_t_gemm_det_scratch_bytes(C.byref(g)) == 4 * 4 * 4 * 4
    assert det(p, p, p, None, C.byref(g), None, 0, st) == -3
    assert det(p, p, p, None, C.byref(g), scratch.data_ptr(), 255, st) == -3
    for g in (desc(M=0, splitk=4), desc(N=0, splitk=4)):
        assert det(p, p, p, None, C.byref(g), None, 0, st) == 0
    torch.cuda.synchronize()


def _st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.gpu
def test_deterministic_scatter_add_equals_the_ordered_emulation_bit_for_bit(flag):
    flag(True)
    L = _cabi.lib()
    g = torch.Generator().manual_seed(3)
    cases = [("char table", 70, 100, torch.randint(0, 70, (19200,), generator=g)),
             ("word table", 200, 300, torch.randint(0, 200, (1600,), generator=g)),
             ("one repeated id", 50, 300, torch.full((700,), 5, dtype=torch.int64)),
             ("clamped ids", 70, 100, torch.tensor([-3, 69, 70, 1000, -1, 0, 68, 5000, 3] * 40))]
    for name, rows, dim, ids in cases:
        dout = torch.randn(ids.numel(), dim, generator=g)
        base = torch.randn(rows, dim, generator=g)
        want = ordered_scatter(base.clone(), dout, ids, rows)
        outs = []
        dd, ii = dout.to(DEV), ids.to(DEV)       # held: a freed temporary's block can be reused before the kernel runs
        for _ in range(2):
            dt = base.to(DEV)
            _cabi.check(L.seqpan_t_scatter_add_rows_det(dt.data_ptr(), dd.data_ptr(), ii.data_ptr(), ids.numel(), dim, rows, _st()))
            outs.append(dt.cpu())
        assert torch.equal(outs[0], want) and torch.equal(outs[1], want), name


def _scratch(nbytes):
    return torch.empty((nbytes + 7) // 8 * 2, device=DEV)      # NaN-filled under the flag


@pytest.mark.gpu
def test_deterministic_layernorm_dwconv_sumsq_match_emulation_and_repeat(flag):
    """Within fp32 order noise of the emulation, ACCUMULATED into what the output held, and bit-identical across launches; the
    LayerNorm dx equals the atomic kernel's."""
    flag(True)
    L, cb = _cabi.lib(), CpuEmuBackend()
    M = 6400
    x, dy, gam = _r(M, 128, seed=1), _r(M, 128, seed=2), _r(128, seed=3)
    dx_e, dg_e, db_e = cb.layernorm_bwd(x, dy, gam, 1e-6)
    g0, b0 = _r(128, seed=4), _r(128, seed=5)
    nb = L.seqpan_t_layernorm_bwd_det_scratch_bytes(M)
    outs = []
    xd, dyd, gd = x.to(DEV), dy.to(DEV), gam.to(DEV)     # device operands (and scratch) are held across every call
    for det in (True, True, False):
        dx, dg, db = torch.empty(M, 128, device=DEV), g0.to(DEV), b0.to(DEV)
        args = [t.data_ptr() for t in (dx, dg, db, xd, dyd, gd)] + [C.c_float(1e-6), M]
        if det:
            scratch = _scratch(nb)
            _cabi.check(L.seqpan_t_layernorm_bwd_det(*args, scratch.data_ptr(), nb, _st()))
        else:
            _cabi.check(L.seqpan_t_layernorm_bwd(*args, _st()))
        outs.append((dx.cpu(), dg.cpu(), db.cpu()))
    (dx, dg, db), again, atomic = outs
    assert all(torch.equal(u, v) for u, v in zip(outs[0], again)) and torch.equal(dx, atomic[0])
    for got, want, name in ((dx, dx_e, "dx"), (dg, g0 + dg_e, "dgamma"), (db, b0 + db_e, "dbeta")):
        assert float((got - want).abs().max()) <= 2e-5 * float(want.abs().max()), name
    # depthwise-conv weight gradient: 64 segments of 100 rows
    rows, seg = 6400, 100
    xc, dyc, w0 = _r(rows, 128, seed=6), _r(rows, 128, seed=7), _r(128, 1, 7, seed=8)
    want = w0 + cb.dwconv_bwd_w(xc, dyc, seg)
    nb = L.seqpan_t_dwconv_bwd_w_det_scratch_bytes(rows)
    res = []
    xd, dyd = xc.to(DEV), dyc.to(DEV)
    for _ in range(2):
        dw, scratch = w0.to(DEV), _scratch(nb)
        _cabi.check(L.seqpan_t_dwconv_bwd_w_det(dw.data_ptr(), xd.data_ptr(), dyd.data_ptr(), rows, seg, scratch.data_ptr(), nb, _st()))
        res.append(dw.cpu())
    assert torch.equal(res[0], res[1]) and float((res[0] - want).abs().max()) <= 2e-5 * float(want.abs().max())
    # squared norm: 5M elements, fp64 partials
    v = _r(5_000_000, seed=9)
    nb = L.seqpan_t_sumsq_det_scratch_bytes(v.numel())
    res = []
    vd = v.to(DEV)
    for _ in range(2):
        acc, scratch = torch.full((), 3.0, dtype=torch.float64, device=DEV), _scratch(nb)
        _cabi.check(L.seqpan_t_sumsq_det(vd.data_ptr(), v.numel(), acc.data_ptr(), scratch.data_ptr(), nb, _st()))
        res.append(float(acc))
    want = 3.0 + float((v.double() ** 2).sum())
    assert res[0] == res[1] and abs(res[0] - want) <= 1e-6 * want


class _CountingLib:
    """The library handle, recording every entry point called and the split-K of every GEMM descriptor."""

    def __init__(self, lib):
        self._lib, self.names, self.splitk = lib, set(), set()

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            self.names.add(name)
            if name in ("seqpan_t_gemm", "seqpan_t_gemm_bf16"):
                self.splitk.add(a[4]._obj.splitk)
            return fn(*a)
        return call


def _steps(case, precision, graph, n=4, backend=None):
    """``n`` TrainSteps of a fresh model from the golden weights, dropout 0.2, fresh draws from seed 11: per step the loss, the
    gradient bucket, the squared norm, the parameters and the AdamW moments."""
    m, batch, _ = _golden_model(case, droprate=0.2)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    ts = train.TrainStep(m, lr=1e-3, num_train_steps=1, precision=precision, backend=backend)
    torch.manual_seed(11)
    rec = []
    for _ in range(n):
        loss, _, ss = ts.step(bd, graph=graph)
        rec.append(dict(loss=loss.clone(), grad=ts.flat.clone(), ss=ss.clone(),
                        **{"p." + k: p.detach().clone() for k, p in m.named_parameters()},
                        **{"m." + k: t.clone() for k, t in ts.m.items()}, **{"v." + k: t.clone() for k, t in ts.v.items()}))
    return rec


def _equal(r1, r2, what):
    for s, (a, b) in enumerate(zip(r1, r2)):
        assert set(a) == set(b)
        bad = [k for k in a if not torch.equal(a[k], b[k])]
        assert not bad, f"{what}, step {s + 1}: {len(bad)} tensors differ, e.g. {bad[:4]}"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", ["charades_small", "anet_small"])
def test_whole_steps_are_bit_identical(flag, case, precision):
    """Two fresh runs of four steps agree bit for bit, eager and graph-replayed, and the eager run equals the replayed one.  The
    device backend calls no atomic entry point and no split-K product of the atomic GEMMs."""
    flag(True)
    be = train.CudaBackend(DEV)
    be.L = _CountingLib(be.L)
    eager = _steps(case, precision, False, backend=be)
    assert not be.L.names & {"seqpan_t_layernorm_bwd", "seqpan_t_dwconv_bwd_w", "seqpan_t_scatter_add_rows", "seqpan_t_sumsq"}
    assert be.L.splitk == {1} and "seqpan_t_sumsq_det" in be.L.names
    assert ("seqpan_t_gemm_bf16_det" if precision == "bf16" else "seqpan_t_gemm_det") in be.L.names
    _equal(eager, _steps(case, precision, False), "eager vs eager")
    graphed = _steps(case, precision, True)
    _equal(graphed, _steps(case, precision, True), "graph vs graph")
    _equal(eager, graphed, "eager vs graph")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_autograd_node_backward_is_bit_identical(flag, precision):
    """model(...) + lossfun_loc + lossfun_match (in torch, on the CPU) + backward(), twice under one seed."""
    flag(True)
    w, m, batch, g = _setup(B=4, L=32, T=9, Cc=7, droprate=0.2)
    m.configs.model.train_precision = precision
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    res = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        x = bd["vfeats"].clone().requires_grad_()
        torch.manual_seed(5)
        out = m(bd["words_ids"], bd["char_ids"], x, bd["vmasks"], bd["tmasks"])
        loss = _reference_losses(out["slogits"].cpu(), out["elogits"].cpu(), out["match_score"].cpu(), out["label_embs"].cpu(), batch)
        loss.backward()
        got = {k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None}
        got["vfeats"] = x.grad.cpu()
        res.append(got)
    assert set(res[0]) == set(res[1])
    assert all(torch.equal(res[0][k], res[1][k]) for k in res[0]), [k for k in res[0] if not torch.equal(res[0][k], res[1][k])]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_toggling_the_flag_between_graph_steps_selects_the_mode(flag, precision):
    """Deterministic steps 1-3 (graph captured at 3), default steps 4-6 (captured at 6), deterministic step 7 replays the
    deterministic graphs: its loss, gradients and squared norm equal a fresh deterministic step from the same parameters and
    draws bit for bit."""
    m, batch, _ = _golden_model("charades_small", droprate=0.2)
    m.to(DEV).train()
    bd = {k: v.to(DEV) for k, v in batch.items()}
    ts = train.TrainStep(m, lr=1e-3, num_train_steps=1, precision=precision)
    torch.manual_seed(11)
    for i in range(6):
        flag(i < 3)
        ts.step(bd, graph=True)
    flag(True)
    params = {k: p.detach().clone() for k, p in m.named_parameters()}
    rng = torch.cuda.get_rng_state(DEV)
    loss, _, ss = ts.step(bd, graph=True)
    got = {k: ts.views[k].clone() for k in ts.live}
    assert sum("graph" in e for e in ts._graphs.values()) == 2 and set(ts._g2) == {True, False}
    m2, _, _ = _golden_model("charades_small", droprate=0.2)
    m2.load_state_dict(params, strict=False)
    m2.to(DEV).train()
    fresh = train.TrainStep(m2, lr=1e-3, num_train_steps=1, precision=precision)
    torch.cuda.set_rng_state(rng, DEV)
    loss2, grads, _ = fresh.loss_and_grads(bd)
    flat = torch.cat([grads[k].reshape(-1) for k in sorted(grads)])
    ss2 = torch.zeros((), dtype=torch.float64, device=DEV)
    fresh.be.sumsq(flat, ss2, deterministic=True)
    assert sorted(grads) == ts.live and torch.equal(loss, loss2) and torch.equal(ss, ss2)
    assert all(torch.equal(got[k], grads[k].reshape(-1)) for k in ts.live)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deterministic_tape_on_device_stays_within_the_accuracy_gates(flag, precision):
    """fp32: the oracle's autograd at rtol 1e-3 (test_train.py); bf16: ORDER_GATES against the bf16 emulation (test_train_bf16.py)."""
    flag(True)
    m, batch, g = _golden_model("charades_small")
    if precision == "fp32":
        val_o, want, _ = _oracle_grads(m, batch, g, "loss")
    else:
        val_o, want = _bf16_tape_grads(m, batch, g, Bf16EmuBackend(), "bf16")
    m.to(DEV)
    bd = {k: v.to(DEV) for k, v in batch.items()}
    val, got = _det_tape_grads(m, bd, g.to(DEV), train.CudaBackend(DEV), precision)
    if precision == "fp32":
        assert abs(val - val_o) <= 1e-5 * abs(val_o)
        _compare(got, want, rtol=1e-3)
    else:
        _check_order_gates(val, got, val_o, want, "deterministic bf16 tape vs bf16 emulation")
