import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
for p in (ROOT, GOLDEN):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def manifest_state_dict(w):
    """Zero state_dict with the reference's keys/shapes (tests/golden/state_dict_manifest.json),
    re-shaped for workload ``w`` (position tables follow vlen, GloVe table follows num_words)."""
    with open(os.path.join(GOLDEN, "state_dict_manifest.json")) as f:
        man = json.load(f)["keys"]
    sd = {}
    for k, shape in man.items():
        shape = list(shape)
        if k.endswith("position_embeddings.weight"):
            shape[0] = w.vlen
        if k.endswith("glove_vec"):
            shape[0] = w.num_words - 2
        sd[k] = torch.zeros(shape)
    return sd


def golden_case(name):
    """(workload, state_dict, batch, fixture) of one golden case, regenerated from seeds and
    checked against the checksums stored by tests/golden/make_golden.py."""
    from cases import CASES, TAPPED
    from vmrframe_b200 import synth
    w = CASES[name]
    fx = dict(np.load(os.path.join(GOLDEN, f"{name}.npz")))
    if name in TAPPED:
        fx.update(np.load(os.path.join(GOLDEN, f"{name}_taps.npz")))
    sd = synth.randomize_state_dict(manifest_state_dict(w), seed=w.config_id)
    batch = synth.make_batch(w, 0)
    chk = np.asarray([float(batch["vfeats"].double().sum()), float(batch["vfeats"].double().abs().sum())])
    assert np.allclose(chk, fx["chk_vfeats"], rtol=1e-12), "synthetic input generator drifted"
    wsum = sum(float(sd[k].double().abs().sum()) for k in sorted(sd))
    assert np.isclose(wsum, float(fx["chk_weights"][0]), rtol=1e-12), "synthetic weight generator drifted"
    return w, sd, batch, fx
