"""Host-side pieces of the measurement: the parity statistics bench.py prints (oracle/parity.py), the roofline bound selection
and the workload label both bench arms must share."""
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import parity
from oracle import seqpan_oracle as O


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_parity_stats_on_known_perturbations():
    g = torch.Generator().manual_seed(0)
    B, L = 64, 40
    want = {"slogits": torch.randn(B, L, generator=g) * 0.3, "elogits": torch.randn(B, L, generator=g) * 0.3,
            "match_score": torch.softmax(torch.randn(B, L, 4, generator=g), -1)}
    vm = torch.ones(B, L)
    fr = O.infer_basic(want["slogits"], want["elogits"], vm)
    same = parity.parity_stats(want, want, vm, fr, fr)
    assert same["slogits"]["max_abs_err"] == 0 and same["spans_equal_all"] == 1.0 and same["largest_margin_of_a_mismatch"] == 0.0
    got = {k: v + 4e-3 for k, v in want.items()}
    fr2 = fr.copy()
    fr2[3, 0] += 0.125                                    # one span differs
    st = parity.parity_stats(got, want, vm, fr2, fr)
    assert math.isclose(st["slogits"]["max_abs_err"], 4e-3, rel_tol=1e-3)
    assert 0 < st["slogits"]["frac_within_rtol_1e-2"] < 1 and st["slogits"]["atol_needed_with_rtol_1e-2"] <= 4e-3
    assert st["spans_equal_all"] == 1 - 1 / B
    margin = O.span_tie_margin(want["slogits"], want["elogits"], vm).numpy()
    assert math.isclose(st["largest_margin_of_a_mismatch"], margin[3] - 1, rel_tol=1e-6)
    for m, e in st["tie"].items():
        assert e["mismatch_in_kept"] == int(margin[3] > 1 + float(m))
    s = parity.summary(st, "bf16", 1e-2)
    assert s["mode"] == "bf16" and s["tie_margin"] == 1e-2 and s["untied_fraction"] == st["tie"]["0.01"]["kept"]
    assert s["spans_equal_untied"] == (st["tie"]["0.01"]["mismatch_in_kept"] == 0)
    # a logit error e can move a span-probability ratio by at most exp(4 e)
    assert math.isclose(parity.tie_margin_for_error(2.5e-3), math.expm1(1e-2))


def test_roofline_bound_follows_measured_dram_traffic():
    b = _bench()
    peaks = {"hbm": 6557.4, "tc_burst": 1639.5, "tc_sustained": 1392.3, "src": "measured"}
    work = (3 * 7.26e9, 3 * 59.5e6)         # conv block: 7.26 GFLOP and 59.5 MB of algorithmic bytes per launch
    # algorithmic bytes alone would call it hbm-bound (59.5 MB / 6.5 TB/s = 9 us > 5.2 us of tensor time) ...
    r0 = b.roofline_of("k", 3, 0.206, work, peaks, 0.3)
    assert r0["bound"] == "hbm"
    # ... but ncu sees 17.7 MB of DRAM traffic per launch (the rest lives in L2): a contraction, reported on the tensor roofline
    r1 = b.roofline_of("k", 3, 0.206, work, peaks, 0.3, traffic=17.7e6)
    assert r1["bound"] == "tensor" and r1["unit"] == "TFLOP/s"
    assert math.isclose(r1["achieved"], 7.26e9 / (0.206e-3 / 3) / 1e12, rel_tol=1e-9)
    assert math.isclose(r1["frac"], r1["tensor_frac"]) and r1["hbm_frac_dram"] < r1["hbm_frac_algorithmic"]
    # a pure copy stays on the HBM roofline
    r2 = b.roofline_of("copy", 1, 0.035, (0.0, 105e6), peaks, 0.05, traffic=105e6)
    assert r2["bound"] == "hbm" and math.isclose(r2["achieved"], 105e6 / 0.035e-3 / 1e9, rel_tol=1e-9)


def test_both_bench_arms_print_the_same_workload_label():
    b = _bench()
    from vmrframe_b200 import synth
    for name in ("charades", "anet", "tacos"):
        w = synth.WORKLOADS[name]
        s = b.workload_string(w)
        assert s.startswith(f"{name}: B={w.batch} L={w.vlen} vdim={w.vdim} Tmax={w.tmax} C={w.clen}") and "BASELINE.json configs[" in s
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"workload": workload_string(w)') == 2          # native arm and reference arm


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's reference arm: the oracle port on the host cores, no GPU): one JSON line with the
    same metric / unit / config.workload as the native arm plus `impl`, `cpu_baseline` and a zero-copy `e2e`."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "charades", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    b = _bench()
    from vmrframe_b200 import synth
    assert line["impl"] == "reference" and line["metric"] == b.METRIC and line["unit"] == b.UNIT
    assert line["config"]["workload"] == b.workload_string(synth.WORKLOADS["charades"])
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["steps"] == 1 and line["warmup"] == 0
    assert line["value"] > 0 and math.isclose(line["value"], line["cpu_baseline"]["value"]) and math.isclose(line["value"], line["e2e"]["value"])
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "charades" in line["cpu_baseline"]["sample"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["gpu_launches"] == 0


def test_bench_rejects_what_it_cannot_time_or_dump():
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"], ["--train", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-2000:])


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's outputs; with the same arguments every run sees the same inputs,
    so two runs write the same arrays."""
    import json
    import subprocess
    import sys
    from vmrframe_b200 import synth
    w = synth.WORKLOADS["charades"]
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "charades", "--steps", "3", "--warmup", "1",
                            "--no-cpu-baseline", "--no-profile", "--no-sustained", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
        dumps.append({f.stem: np.load(f) for f in d.glob("*.npy")})
    a, b = dumps
    shapes = {"slogits": (w.batch, w.vlen), "elogits": (w.batch, w.vlen), "match_score": (w.batch, w.vlen, 4), "span_fracs": (w.batch, 2)}
    assert {k: v.shape for k, v in a.items()} == shapes and all(v.dtype == np.float32 for v in a.values())
    assert np.allclose(a["match_score"].sum(-1), 1.0, atol=1e-5)
    assert np.all(a["span_fracs"][:, 0] <= a["span_fracs"][:, 1]) and np.all((a["span_fracs"] >= 0) & (a["span_fracs"] <= 1))
    for k in ("slogits", "elogits", "match_score"):
        assert np.allclose(a[k], b[k], rtol=0, atol=1e-6), k
    assert np.array_equal(a["span_fracs"], b["span_fracs"])
