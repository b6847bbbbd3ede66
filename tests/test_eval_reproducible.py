"""Reproducible evaluation sweeps (DESIGN.md section 13): seeded per-batch Gumbel noise (``seqpan_gumbel_noise``,
``gumbel_noise``) and order-independent IoU counters (``seqpan_iou_counters_exact``, ``IouCounters(exact=True)``) behind
``evaluate(seed=, batch_ids=)``.

CPU: a numpy port of Philox4x32-10 against the Random123 known answers, its Gumbel transform against the Gumbel law, the
exactness argument of the rounded sums, the argument checks of ``evaluate`` / ``gumbel_noise`` / the C ABI, and the batch ids
through ``shard_batches`` and ``draw_chunks``.  B200: the kernel against the port, bit for bit (Philox words and uniforms,
read back by a probe kernel compiled from the same header) and within 4 ulp (noise); the exact counters; and seeded sweeps
that return the same bits however they are split."""
import ctypes as C
import math
import os
import socket
import threading

import numpy as np
import pytest
import torch

from vmrframe_b200 import SeqPAN, _cabi, engine, gumbel_noise, infer_SeqPAN, synth

DEV = "cuda:0"

# ---- numpy port of the definition ---------------------------------------------------------------------------------------
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 of uint32 counters ``[..., 4]`` under uint32 keys ``[..., 2]`` (broadcast)."""
    c = [ctr[..., i].astype(np.uint64) for i in range(4)]
    k0, k1 = key[..., 0].astype(np.uint64), key[..., 1].astype(np.uint64)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _MASK, (k1 + np.uint64(0xBB67AE85)) & _MASK
    return np.stack(c, -1).astype(np.uint32)


def port_words(seed, batch_id, B, L):
    """The ``[B, L, 4]`` Philox words of batch ``batch_id`` of a sweep seeded with ``seed``."""
    rows = np.arange(B * L, dtype=np.uint64)
    ctr = np.stack([rows, np.full_like(rows, batch_id), np.zeros_like(rows), np.zeros_like(rows)], -1)
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64)
    return philox4x32_10(ctr, key).reshape(B, L, 4)


def port_uniform(x):
    return ((x >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)


def port_gumbel(u):
    """-log(-log(u)) with each logarithm correctly rounded to fp32 (computed in fp64, then rounded)."""
    v = (-np.log(u.astype(np.float64))).astype(np.float32)
    return (-np.log(v.astype(np.float64))).astype(np.float32)


def span_iou(gt, fr):
    """``span_iou`` of kernels_f32.cu: fp32 min / max / differences, fp64 division, clamped at 0."""
    g0, g1, p0, p1 = (a.astype(np.float32) for a in (gt[:, 0], gt[:, 1], fr[:, 0], fr[:, 1]))
    uni = np.maximum(g1, p1) - np.minimum(g0, p0)
    inter = np.minimum(g1, p1) - np.maximum(g0, p0)
    with np.errstate(divide="ignore", invalid="ignore"):
        iou = np.where(uni != 0, inter.astype(np.float64) / uni.astype(np.float64), 0.0)
    return np.maximum(iou, 0.0)


def exact_counters(gt, fr):
    """What ``seqpan_iou_counters_exact`` adds for one call."""
    iou = span_iou(gt, fr)
    return np.array([len(iou), np.sum(np.rint(iou * 2.0 ** 28) * 2.0 ** -28), np.sum(iou >= 0.3), np.sum(iou >= 0.5),
                     np.sum(iou >= 0.7)], dtype=np.float64)


# ---- CPU ------------------------------------------------------------------------------------------------------------------
def test_philox_port_known_answers():
    # Random123's kat_vectors for philox4x32_10 (also what curand_Philox4x32_10 returns)
    for ctr, key, want in [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
                           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
                           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
                            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]:
        got = philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
        assert got.tolist() == list(want)
    # the definition's key and counter layout: seed 0, batch 0, row 0 is the first known answer
    assert port_words(0, 0, 1, 1)[0, 0].tolist() == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


def test_port_gumbel_follows_the_gumbel_law():
    from scipy import stats
    u = port_uniform(port_words(12345, 3, 4096, 256)).reshape(-1)           # 2^22 samples
    assert u.size == 1 << 22 and u.min() > 0 and u.max() < 1
    assert np.all(u == (np.floor(u.astype(np.float64) * 2 ** 23) + 0.5) * 2.0 ** -23)   # the open grid, exactly
    g = port_gumbel(u).astype(np.float64)
    assert np.all(np.isfinite(g))
    assert abs(g.mean() - np.euler_gamma) < 3e-3                              # standard error 6.3e-4
    assert abs(g.var() - np.pi ** 2 / 6) < 1e-2                               # standard error 1.7e-3
    assert stats.kstest(g, stats.gumbel_r.cdf).pvalue > 1e-3


def test_rounded_iou_sums_do_not_depend_on_order():
    rng = np.random.default_rng(0)
    iou = rng.random(1 << 16)
    iou[:100] = 0.0
    iou[100:200] = 1.0
    q = np.rint(iou * 2.0 ** 28) * 2.0 ** -28
    assert np.all(np.abs(q - iou) <= 2.0 ** -29)
    exact = math.fsum(q)

    def seq(x):
        s = 0.0
        for v in x.tolist():
            s += v
        return s

    sums = [seq(q), seq(q[::-1]), float(np.sum(q)), sum(seq(c) for c in np.array_split(q, 37))]
    for _ in range(3):
        p = rng.permutation(q)
        sums += [seq(p), float(np.add.reduce(p)), seq(np.array([seq(c) for c in np.array_split(p, 148)]))]
    assert all(s == exact for s in sums)
    # the unrounded values do depend on the order
    raw = [seq(iou), seq(iou[::-1]), float(np.sum(iou))] + [seq(rng.permutation(iou)) for _ in range(3)]
    assert len(set(raw)) > 1
    # the bound: n <= 2^25 values <= 1 sum to at most 2^25 = 2^53 units of 2^-28, all representable
    top = 2.0 ** 25 - 2.0 ** -28
    assert top + 2.0 ** -28 == 2.0 ** 25 and top - 2.0 ** -28 != top
    assert 2.0 ** 25 + 2.0 ** -28 == 2.0 ** 25                                # one past the bound is lost


def _fake_batches(n, B=4):
    return [{"vmasks": torch.ones(B, 8)} for _ in range(n)]


def test_evaluate_argument_checks():
    bt = _fake_batches(3)
    bad = [dict(seed=-1), dict(seed=1 << 64), dict(seed=1.5), dict(seed="7"), dict(seed=True), dict(seed=np.float64(2)),
           dict(seed=1, batch_ids=[0, 1]), dict(seed=1, batch_ids=[0, 1, 2, 3]), dict(seed=1, batch_ids=[0, 1, 1]),
           dict(seed=1, batch_ids=[0, -1, 2]), dict(seed=1, batch_ids=[0, 1, 1 << 32]), dict(seed=1, batch_ids=[0, 1.0, 2]),
           dict(seed=1, batch_ids=[0, True, 2]), dict(batch_ids=[0, 1, 2])]
    for kw in bad:
        with pytest.raises(ValueError):
            engine.evaluate(None, bt, **kw)
    huge = [{"vmasks": torch.empty(1 << 24, 0)} for _ in range(2)] + [{"vmasks": torch.empty(1, 0)}]   # 2^25 + 1 samples
    with pytest.raises(ValueError, match="2\\^25"):
        engine.evaluate(None, huge, seed=0)
    assert engine._sweep_ids(huge[:2], 0, None) == (0, [0, 1])                 # 2^25 exactly is allowed
    assert engine._sweep_ids(bt, None, None) == (None, None)
    assert engine._sweep_ids(bt, (1 << 64) - 1, np.array([7, 0, (1 << 32) - 1])) == ((1 << 64) - 1, [7, 0, (1 << 32) - 1])
    assert engine._sweep_ids(bt, np.uint64(5), range(10, 13)) == (5, [10, 11, 12])
    assert engine._sweep_ids([], 3, None) == (3, [])
    for kw in (dict(seed=-1, batch_id=0), dict(seed=1 << 64, batch_id=0), dict(seed=0, batch_id=1 << 32),
               dict(seed=0, batch_id=-1), dict(seed=0.0, batch_id=0), dict(seed=0, batch_id=0.5)):
        with pytest.raises(ValueError):
            gumbel_noise(2, 8, **kw)
    with pytest.raises(ValueError):
        gumbel_noise(-1, 8, 0, 0)


def test_c_abi_argument_checks():
    lib = _cabi.lib()
    p = C.c_void_p(256)      # never dereferenced: every call below fails its argument checks first
    for args, msg in [((0, 0, 2, 8, None), b"out is NULL"), ((0, 0, 2, 8, C.c_void_p(260)), b"aligned"),
                      ((0, 0, -1, 8, p), b"B=-1"), ((0, 0, 2, 0, p), b"L=0"), ((0, 0, 2, 257, p), b"L=257"),
                      ((0, 0, (1 << 31) - 1, 256, p), b"32-bit")]:
        assert lib.seqpan_gumbel_noise(*args, None) == -1 and msg in lib.seqpan_last_error(), (args, lib.seqpan_last_error())
    for args, msg in [((None, p, 2, p), b"fracs is NULL"), ((p, None, 2, p), b"gt_fracs is NULL"),
                      ((p, p, 2, None), b"counters is NULL"), ((p, p, -1, p), b"B=-1")]:
        assert lib.seqpan_iou_counters_exact(*args, None) == -1 and msg in lib.seqpan_last_error(), args


class _FakeStore:
    """``TCPStore.add`` semantics (atomic add, returns the new value) for single-process checks."""

    def __init__(self):
        self.v, self.lock = {}, threading.Lock()

    def add(self, key, n):
        with self.lock:
            self.v[key] = self.v.get(key, 0) + n
            return self.v[key]


def _fake_spans(n, B, seed=4):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        s, p = rng.random(B) * 0.6, rng.random(B) * 0.6
        out.append((np.stack([s, s + 0.05 + rng.random(B) * 0.35], 1).astype(np.float32),
                    np.stack([p, p + 0.05 + rng.random(B) * 0.35], 1).astype(np.float32)))
    return out


def test_batch_ids_through_shards_and_the_work_queue():
    """Every batch reaches exactly one rank with its global id, and the ranks' exact counters sum to the single-process bits
    in any order."""
    n, B, seed = 97, 6, 2 ** 40 + 17
    spans = _fake_spans(n, B)
    batches = _fake_batches(n, B)
    _, ids = engine._sweep_ids(batches, seed, None)
    want = np.sum([exact_counters(*spans[i]) for i in ids], axis=0)

    def rank_part(ids):
        s, got = engine._sweep_ids([batches[k] for k in ids], seed, ids)
        assert s == seed and got == list(ids)
        return np.sum([exact_counters(*spans[k]) for k in got], axis=0)

    for world in (2, 3, 8):
        parts = [rank_part(engine.shard_batches(n, r, world)) for r in range(world)]
        for order in (parts, parts[::-1]):
            assert np.sum(order, axis=0).tobytes() == want.tobytes()
    for world, chunk in ((2, 8), (4, 8), (3, 16)):
        store, parts, seen = _FakeStore(), [], []
        lock = threading.Lock()

        def rank_loop():
            for ids in engine.draw_chunks(store, n, world, chunk):
                c = rank_part(ids)                    # one evaluate(allreduce=False) per chunk
                with lock:
                    parts.append(c)
                    seen.extend(ids)

        ts = [threading.Thread(target=rank_loop) for _ in range(world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        assert sorted(seen) == list(range(n))
        total = np.zeros(5)
        for c in parts:                               # completion order of the threads
            total += c
        assert total.tobytes() == want.tobytes()


# ---- B200: kernels ----------------------------------------------------------------------------------------------------------
PROBE_CASES = [(0, 0, 1, 256), (1, 7, 3, 100), ((1 << 32) + 5, (1 << 32) - 1, 2, 64), ((1 << 64) - 1, 123, 256, 100),
               (0x243F6A8885A308D3, 1 << 31, 5, 33)]

# The stages of seqpan_gumbel_noise read back on the device: the same inline functions (csrc/gumbel.cuh) compiled with the
# library's flags.
PROBE_SRC = r"""
#include "gumbel.cuh"
__global__ void probe(uint64_t seed, uint32_t batch_id, uint32_t rows, uint4* words, float4* uniforms, float4* noise) {
  const uint32_t r = blockIdx.x * 256u + threadIdx.x;
  if (r >= rows) return;
  const uint4 x = sq::gumbel_words(seed, batch_id, r);
  words[r] = x;
  uniforms[r] = make_float4(sq::open_uniform(x.x), sq::open_uniform(x.y), sq::open_uniform(x.z), sq::open_uniform(x.w));
  noise[r] = make_float4(sq::gumbel_of(x.x), sq::gumbel_of(x.y), sq::gumbel_of(x.z), sq::gumbel_of(x.w));
}
extern "C" int philox_probe(uint64_t seed, uint32_t batch_id, int rows, void* words, void* uniforms, void* noise) {
  probe<<<(rows + 255) / 256, 256>>>(seed, batch_id, rows, (uint4*)words, (float4*)uniforms, (float4*)noise);
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    import subprocess
    from vmrframe_b200 import build
    d = tmp_path_factory.mktemp("philox_probe")
    src, so = d / "probe.cu", d / "probe.so"
    src.write_text(PROBE_SRC)
    cmd = [os.environ.get("NVCC", "nvcc")] + build.CFLAGS + ["-I", build.CSRC, "-shared", "-cudart", "static", "-o", str(so),
                                                            str(src)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = C.CDLL(str(so))
    lib.philox_probe.restype = C.c_int
    lib.philox_probe.argtypes = [C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]

    def run(seed, batch_id, B, L):
        words = torch.empty(B, L, 4, dtype=torch.int32, device=DEV)
        uni, noise = torch.empty(B, L, 4, device=DEV), torch.empty(B, L, 4, device=DEV)
        torch.cuda.synchronize()
        assert lib.philox_probe(seed, batch_id, B * L, words.data_ptr(), uni.data_ptr(), noise.data_ptr()) == 0
        return words.cpu().numpy().view(np.uint32), uni.cpu().numpy(), noise.cpu().numpy()
    return run


@pytest.mark.gpu
def test_device_philox_and_uniforms_equal_the_port(probe):
    w, _, _ = probe(0, 0, 1, 1)
    assert w[0, 0].tolist() == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]   # curand's Philox on the device
    for seed, bid, B, L in PROBE_CASES:
        w, u, g = probe(seed, bid, B, L)
        pw = port_words(seed, bid, B, L)
        assert np.array_equal(w, pw), (seed, bid, B, L)
        assert np.array_equal(u.view(np.uint32), port_uniform(pw).view(np.uint32)), (seed, bid, B, L)
        # and the library's kernel computes the probe's noise from them, bit for bit
        assert np.array_equal(gumbel_noise(B, L, seed, bid, device=DEV).cpu().numpy().view(np.uint32), g.view(np.uint32))


@pytest.mark.gpu
def test_device_noise_within_4_ulp_of_the_port():
    """4 ulp of max(|g|, 1): one rounding of the inner logarithm moves g by up to 2^-23 absolutely, which near g = 0 is many
    ulp of g itself."""
    for seed, bid, B, L in PROBE_CASES:
        g = gumbel_noise(B, L, seed, bid, device=DEV)
        assert g.shape == (B, L, 4) and g.dtype == torch.float32 and g.device == torch.device(DEV)
        g = g.cpu().numpy()
        want = port_gumbel(port_uniform(port_words(seed, bid, B, L)))
        assert np.all(np.isfinite(g))
        scale = np.spacing(np.maximum(np.abs(want), np.float32(1)))
        assert np.all(np.abs(g.astype(np.float64) - want) <= 4 * scale.astype(np.float64)), (seed, bid, B, L)
    assert gumbel_noise(0, 8, 1, 2, device=DEV).shape == (0, 8, 4)
    with torch.cuda.device(DEV):
        assert gumbel_noise(2, 8, 1, 2).device == torch.device(DEV)           # default: the current device


@pytest.mark.gpu
def test_noise_repeats_and_replays_bit_for_bit():
    B, L = 256, 100
    out = torch.empty(B, L, 4, device=DEV)

    def launch():
        _cabi.check(_cabi.lib().seqpan_gumbel_noise(99, 5, B, L, out.data_ptr(), torch.cuda.current_stream().cuda_stream))

    launch()
    first = out.clone()
    for _ in range(3):
        out.fill_(float("nan"))
        launch()
        assert torch.equal(out, first)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        launch()
    out.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, first)
    assert torch.equal(gumbel_noise(B, L, 99, 5, device=DEV), first)


@pytest.mark.gpu
def test_streams_of_other_seeds_and_batches_are_uncorrelated():
    B, L = 256, 100
    n = B * L * 4
    base = gumbel_noise(B, L, 7, 11, device=DEV).reshape(-1).double()
    others = [(7, 12), (8, 11), (7 + (1 << 32), 11), (7, 11 + (1 << 31)), ((1 << 64) - 1, (1 << 32) - 1), (0, 0)]
    for seed, bid in others:
        o = gumbel_noise(B, L, seed, bid, device=DEV).reshape(-1).double()
        assert not torch.equal(o, base)
        corr = float(torch.corrcoef(torch.stack([base, o]))[0, 1])
        assert abs(corr) < 4 / math.sqrt(n), (seed, bid, corr)
    # neighbouring rows and the four labels of a row are not correlated either
    g = base.reshape(B * L, 4)
    assert abs(float(torch.corrcoef(torch.stack([g[:-1, 0], g[1:, 0]]))[0, 1])) < 4 / math.sqrt(B * L)
    assert abs(float(torch.corrcoef(torch.stack([g[:, 0], g[:, 3]]))[0, 1])) < 4 / math.sqrt(B * L)


def _spans(n, seed):
    rng = np.random.default_rng(seed)
    s, p = rng.random(n) * 0.6, rng.random(n) * 0.6
    gt = np.stack([s, s + 0.05 + rng.random(n) * 0.35], 1).astype(np.float32)
    fr = np.stack([p, p + rng.random(n) * 0.35], 1).astype(np.float32)
    fr[:7] = gt[:7]                             # IoU exactly 1
    fr[20:25] = [[0.2, 0.2]] * 5
    gt[20:25] = [[0.2, 0.2]] * 5                # empty union: IoU 0
    gt[30], fr[30] = [0.0, 0.4], [0.2, 0.4]     # IoU 0.5 exactly
    gt[31], fr[31] = [0.0, 0.1], [0.5, 0.6]     # disjoint: clamped at 0
    return gt, fr


@pytest.mark.gpu
def test_exact_counters():
    n = 70001
    gt, fr = _spans(n, 3)
    ex = engine.IouCounters(DEV, exact=True)
    ex.update(torch.from_numpy(fr), torch.from_numpy(gt))
    plain = engine.IouCounters(DEV)
    plain.update(torch.from_numpy(fr), torch.from_numpy(gt))
    c, cp = ex.buf.cpu().numpy(), plain.buf.cpu().numpy()
    assert c[0] == cp[0] == n and np.array_equal(c[2:], cp[2:])
    iou = span_iou(gt, fr)
    assert abs(c[1] - math.fsum(iou)) <= n * 2.0 ** -29
    assert c.tobytes() == exact_counters(gt, fr).tobytes()                    # the host emulation, bit for bit
    # get_i345_mi of the same IoUs: the R1 entries exactly, the mean IoU within 1e-9 (1e-7 percentage points)
    host = engine.get_i345_mi(iou.tolist())
    assert ex.result()[:4] == host[:4] and abs(ex.result()[4] - host[4]) <= 1e-7
    rng = np.random.default_rng(5)
    for trial in range(3):
        perm = rng.permutation(n)
        other = engine.IouCounters(DEV, exact=True)
        streams = [torch.cuda.Stream() for _ in range(3)]
        ev = torch.cuda.Event()
        ev.record()
        cuts = np.sort(rng.choice(np.arange(1, n), size=9 + trial, replace=False))
        pieces = [(torch.from_numpy(gt[idx]).to(DEV), torch.from_numpy(fr[idx]).to(DEV)) for idx in np.split(perm, cuts)]
        torch.cuda.synchronize()
        for k, (g, f) in enumerate(pieces):                                   # several calls on several streams, one buffer
            st = streams[k % 3]
            st.wait_event(ev)
            with torch.cuda.stream(st):
                _cabi.check(_cabi.lib().seqpan_iou_counters_exact(f.data_ptr(), g.data_ptr(), g.shape[0], other.buf.data_ptr(),
                                                                  st.cuda_stream))
        torch.cuda.synchronize()
        assert other.buf.cpu().numpy().tobytes() == c.tobytes(), trial
        bufs = []                                                             # separate buffers summed afterwards
        for g, f in pieces:
            b = engine.IouCounters(DEV, exact=True)
            b.update(f, g)
            bufs.append(b.buf)
        assert torch.stack(bufs).sum(0).cpu().numpy().tobytes() == c.tobytes()


# ---- B200: sweeps -----------------------------------------------------------------------------------------------------------
def _model(w, precision="fp32", seed=5, device=DEV):
    m = SeqPAN(synth.make_configs(w), synth.make_word_vectors(w), precision=precision).eval()
    m.load_state_dict(synth.randomize_state_dict(m.state_dict(), seed=seed))
    return m.to(device)


SWEEP = synth.small_workload("reproducible", 8, 64, 10, 10, 83)


def _sweep_batches(n=7):
    return [synth.make_batch(SWEEP, i, pin=True) for i in range(n)]


def _bits(t):
    return t.detach().cpu().numpy().tobytes()


def _same(a, b):
    (ma, ca, ia), (mb, cb, ib) = a, b
    assert ma == mb and _bits(ca) == _bits(cb)
    assert len(ia["fracs"]) == len(ib["fracs"]) and all(np.array_equal(x, y) for x, y in zip(ia["fracs"], ib["fracs"]))


@pytest.mark.gpu
@pytest.mark.parametrize("topk", [None, 5])
def test_seeded_sweep_is_the_same_however_it_is_split(topk):
    m = _model(SWEEP)
    batches = _sweep_batches()
    n = len(batches)
    seed = 2 ** 33 + 9
    kw = dict(return_fracs=True, topk=topk, seed=seed)
    ref = engine.evaluate(m, batches, DEV, streams=1, depth=2, **kw)
    assert ref[2]["seed"] == seed and ref[1].dtype == torch.float64

    def check(res):
        _same(ref, res)
        if topk:
            assert _bits(res[2]["topk"]["counters"]) == _bits(ref[2]["topk"]["counters"])
            assert res[2]["topk"]["recall"] == ref[2]["topk"]["recall"]
            assert all(np.array_equal(x, y) for x, y in zip(res[2]["topk_fracs"], ref[2]["topk_fracs"]))

    for streams in (2, 3):
        check(engine.evaluate(m, batches, DEV, streams=streams, **kw))
    check(engine.evaluate(m, batches, DEV, streams=2, depth=1, **kw))
    check(engine.evaluate(m, batches, DEV, streams=2, ragged_h2d=False, **kw))
    check(engine.evaluate(m, batches, DEV, streams=3, ragged_h2d=True, h2d_ctas=0, **kw))
    check(engine.evaluate(m, batches, **kw))                                  # default device and lanes
    # chunked calls with allreduce=False, summed
    parts = [engine.evaluate(m, batches[lo:hi], DEV, streams=2, allreduce=False, batch_ids=range(lo, hi), **kw)
             for lo, hi in ((0, 2), (2, 3), (3, n))]
    total = sum(p[1] for p in parts)
    assert _bits(total) == _bits(ref[1])
    assert engine.metrics_from_counters(total.cpu().tolist()) == ref[0]
    assert all(np.array_equal(x, y) for x, y in zip([f for p in parts for f in p[2]["fracs"]], ref[2]["fracs"]))
    if topk:
        assert _bits(sum(p[2]["topk"]["counters"] for p in parts)) == _bits(ref[2]["topk"]["counters"])
    # permuted batches with their ids
    perm = [4, 0, 6, 2, 5, 1, 3]
    res = engine.evaluate(m, [batches[k] for k in perm], DEV, streams=3, batch_ids=perm, **kw)
    assert res[0] == ref[0] and _bits(res[1]) == _bits(ref[1])
    assert all(np.array_equal(res[2]["fracs"][j], ref[2]["fracs"][k]) for j, k in enumerate(perm))
    if topk:
        assert _bits(res[2]["topk"]["counters"]) == _bits(ref[2]["topk"]["counters"])
    else:
        # top-k leaves the IoU part alone
        tk = engine.evaluate(m, batches, DEV, streams=2, return_fracs=True, topk=5, seed=seed)
        _same(ref, tk)


@pytest.mark.gpu
def test_seeded_sweep_equals_batchwise_calls_and_repeats():
    m = _model(SWEEP)
    batches = _sweep_batches()
    seed = 31
    ref = engine.evaluate(m, batches, DEV, return_fracs=True, streams=2, seed=seed)
    _same(ref, engine.evaluate(m, batches, DEV, return_fracs=True, streams=2, seed=seed))     # the same seed twice
    ic = engine.IouCounters(DEV, exact=True)
    for i, (hb, fr) in enumerate(zip(batches, ref[2]["fracs"])):
        b = {k: v.to(DEV) for k, v in hb.items()}
        B, L = hb["vmasks"].shape
        g = gumbel_noise(B, L, seed, i, device=DEV)
        out = m(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], gumbel=g)
        assert np.array_equal(infer_SeqPAN(out), fr), i
        ic.update(torch.from_numpy(fr), hb["se_fracs"])
        g2 = gumbel_noise(B, L, seed + 1, i, device=DEV)                     # another seed: other noise, other logits
        assert not torch.equal(g, g2)
        out2 = m(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], gumbel=g2)
        assert not torch.equal(out["slogits"], out2["slogits"])
    assert _bits(ic.buf) == _bits(ref[1])
    other = engine.evaluate(m, batches, DEV, return_fracs=True, streams=2, seed=seed + 1)
    assert other[2]["seed"] == seed + 1


@pytest.mark.gpu
def test_unseeded_sweep_is_unchanged():
    """seed=None: torch's draw on the lane and the plain counters, as before (one lane: the draws in batch order)."""
    m = _model(SWEEP)
    batches = _sweep_batches(5)
    torch.manual_seed(21)
    metrics, counters, info = engine.evaluate(m, batches, DEV, return_fracs=True, streams=1)
    assert "seed" not in info
    torch.manual_seed(21)
    ic = engine.IouCounters(DEV)
    for hb, fr in zip(batches, info["fracs"]):
        b = {k: v.to(DEV) for k, v in hb.items()}
        B, L = hb["vmasks"].shape
        g = -torch.empty(B, L, 4, device=DEV).exponential_().log()
        out = m(b["words_ids"], b["char_ids"], b["vfeats"], b["vmasks"], b["tmasks"], gumbel=g)
        fd = infer_SeqPAN(out)
        assert np.array_equal(fd, fr)
        ic.update(torch.from_numpy(fd), hb["se_fracs"])
    assert _bits(ic.buf) == _bits(counters) and ic.result() == metrics


@pytest.mark.gpu
@pytest.mark.parametrize("topk", [None, 5])
def test_seeded_sweep_from_encodings_equals_raw_clips(topk):
    w = synth.Workload("reproducible_encoded", 62, 16, 64, 10, 10, num_words=300, group=8)
    m = _model(w, "bf16", seed=9)
    batches = [synth.share_clips(synth.make_batch(w, i, pin=True), w.group) for i in range(4)]
    enc = m.encode_videos(torch.cat([bt["vfeats"] for bt in batches]).to(DEV))
    enc_batches = []
    for i, bt in enumerate(batches):
        e = {k: v for k, v in bt.items() if k != "vfeats"}
        e["video_index"] = (bt["video_index"] + 2 * i).to(torch.int32)
        enc_batches.append(e)
    kw = dict(return_fracs=True, topk=topk, seed=1 << 63)
    raw = engine.evaluate(m, batches, DEV, streams=2, **kw)
    for streams in (1, 3):
        res = engine.evaluate(m, enc_batches, DEV, streams=streams, video_encodings=enc, **kw)
        _same(raw, res)
        if topk:
            assert _bits(res[2]["topk"]["counters"]) == _bits(raw[2]["topk"]["counters"])
    rev = engine.evaluate(m, enc_batches[::-1], DEV, streams=2, video_encodings=enc, batch_ids=[3, 2, 1, 0], **kw)
    assert _bits(rev[1]) == _bits(raw[1]) and rev[0] == raw[0]


# ---- B200: two ranks --------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


N_RANK_BATCHES, RANK_SEED = 21, 1234567


def _rank_worker(rank, world, port, port2, q):
    import datetime

    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
    m = _model(SWEEP, device=dev)
    batches = _sweep_batches(N_RANK_BATCHES)
    mine = engine.shard_batches(len(batches), rank, world)
    _, static, _ = engine.evaluate(m, [batches[k] for k in mine], dev, seed=RANK_SEED, batch_ids=mine)
    store = dist.TCPStore("127.0.0.1", port2, world, rank == 0)
    total = torch.zeros(5, dtype=torch.float64, device=dev)
    drawn = []
    for ids in engine.draw_chunks(store, len(batches), world, chunk=8):
        _, c, _ = engine.evaluate(m, [batches[k] for k in ids], dev, seed=RANK_SEED, batch_ids=ids, allreduce=False)
        total += c
        drawn.extend(ids)
    dist.all_reduce(total)
    q.put((rank, static.cpu().numpy().tobytes(), total.cpu().numpy().tobytes(), drawn))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_nccl_ranks_return_the_single_process_counters():
    import torch.multiprocessing as mp
    m = _model(SWEEP)
    _, want, _ = engine.evaluate(m, _sweep_batches(N_RANK_BATCHES), DEV, seed=RANK_SEED)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port, port2 = _free_port(), _free_port()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, port2, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda r: r[0])
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(timeout=30)
    assert sorted(k for r in res for k in r[3]) == list(range(N_RANK_BATCHES))
    for _, static, queued, _ in res:
        assert static == _bits(want)
        assert queued == _bits(want)
