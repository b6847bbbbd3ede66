"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference on CPU.

Run in the build container only (it needs /root/reference, which does not travel to the GPU box):

    python tests/golden/make_golden.py

The reference is imported through the three shims of SURVEY.md Appendix B (no source edits):
a stub ``tkinter`` module (models/layers.py:3), a bare ``models`` package so that
``models/__init__.py`` (which needs sentence_transformers) never runs, and a no-op
``torch.cuda.synchronize`` on this CUDA-less host (models/SeqPAN.py:51,85).

Inputs and weights are NOT stored: they are regenerated bit-identically from seeds by
``vmrframe_b200/synth.py`` (CPU generators); each fixture stores float64 checksums of them so a
drifting generator is detected.  Stored: the reference's outputs and hooked intermediates.
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def import_reference():
    sys.path.insert(0, REF)
    tk = types.ModuleType("tkinter"); tk.Y = "y"; sys.modules["tkinter"] = tk
    pkg = types.ModuleType("models"); pkg.__path__ = [REF + "/models"]; sys.modules["models"] = pkg
    if not torch.cuda.is_available():
        torch.cuda.synchronize = lambda *a, **k: None
    import models.SeqPAN as S
    from models.layers import ConditionedPredictor
    from utils.engine import infer_basic
    from models.loss import append_ious, get_i345_mi
    return S, ConditionedPredictor, infer_basic, append_ious, get_i345_mi


def checksum(t):
    return float(t.double().sum()), float(t.double().abs().sum())


def main():
    from vmrframe_b200 import synth
    from cases import CASES, LATE_TAPS, TAPPED
    S, CP, infer_basic, append_ious, get_i345_mi = import_reference()
    torch.set_num_threads(8)
    manifest_written = False
    for name, w in CASES.items():
        cfg = synth.make_configs(w)
        wv = synth.make_word_vectors(w)
        torch.manual_seed(0)
        model = S.SeqPAN(cfg, wv).eval()
        if not manifest_written:
            # key/shape manifest of the reference state_dict at the ActivityNet vlen + default-init stats
            man = {k: list(v.shape) for k, v in model.state_dict().items()}
            with open(os.path.join(HERE, "state_dict_manifest.json"), "w") as f:
                json.dump({"vlen": w.vlen, "num_words": w.num_words, "keys": man}, f, indent=0)
            manifest_written = True
        sd = synth.randomize_state_dict(model.state_dict(), seed=w.config_id)
        model.load_state_dict(sd)
        batch = synth.make_batch(w, 0)
        taps = {}

        def hook(tag):
            def fn(mod, inp, out):
                taps.setdefault(tag, []).append(out.detach().clone() if torch.is_tensor(out)
                                                else [o.detach().clone() for o in out])
            return fn
        for tag, mod in [("text_emb", model.text_encoder), ("video_affine", model.video_affine),
                         ("enc", model.vfeat_encoder), ("dab1", model.dual_attention_block_1),
                         ("dab2", model.dual_attention_block_2), ("t2v", model.q2v_attn),
                         ("v2t", model.v2q_attn), ("fuse", model.cq_cat),
                         ("fep", model.predictor.feature_encoder)]:
            mod.register_forward_hook(hook(tag))
        B, L = batch["vmasks"].shape
        g = synth.gumbel_noise(B, L, seed=7)
        torch.manual_seed(7)            # pins the Gumbel draw inside forward (models/SeqPAN.py:79)
        with torch.no_grad():
            out = model(batch["words_ids"], batch["char_ids"], batch["vfeats"], batch["vmasks"], batch["tmasks"])
            fracs = infer_basic(out["slogits"], out["elogits"], out["vmask"])
            si, ei = CP.extract_index(out["slogits"], out["elogits"])
        ious = append_ious([], batch["se_fracs"].numpy(), fracs)
        metrics = get_i345_mi(ious)
        fx = {
            "slogits": out["slogits"].numpy(), "elogits": out["elogits"].numpy(),
            "match_score": out["match_score"].numpy(), "fracs": fracs.astype(np.float32),
            "extract_start": si.numpy(), "extract_end": ei.numpy(),
            "ious": np.asarray(ious, dtype=np.float64), "metrics": np.asarray(metrics, dtype=np.float64),
            "gumbel": g.numpy(),
            "chk_vfeats": np.asarray(checksum(batch["vfeats"])),
            "chk_ids": np.asarray(checksum(batch["words_ids"]) + checksum(batch["char_ids"])),
            "chk_weights": np.asarray([checksum(sd[k])[1] for k in sorted(sd)]).sum(keepdims=True),
        }
        if name in TAPPED:
            fx.update({
            "text_emb": taps["text_emb"][0].numpy(), "video_affine": taps["video_affine"][0].numpy(),
            "venc": taps["enc"][0].numpy(), "tenc": taps["enc"][1].numpy(),
            "dab1_v": taps["dab1"][0].numpy(), "dab1_t": taps["dab1"][1].numpy(),
            "dab2_v": taps["dab2"][0].numpy(), "dab2_t": taps["dab2"][1].numpy(),
            "t2v": taps["t2v"][0].numpy(), "v2t": taps["v2t"][0].numpy(), "fuse": taps["fuse"][0].numpy(),
            "fep_s": taps["fep"][0].numpy(), "fep_e": taps["fep"][1].numpy()})
            np.savez_compressed(os.path.join(HERE, f"{name}_taps.npz"), **{k: fx.pop(k) for k in LATE_TAPS})
        np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **fx)
        print(name, {k: v.shape for k, v in fx.items() if v.ndim > 1}, "metrics", metrics)

    # default-init statistics: the drop-in constructor must reproduce them under the same seed
    w = CASES["anet_small"]
    torch.manual_seed(0)
    model = S.SeqPAN(synth.make_configs(w), synth.make_word_vectors(w))
    stats = {k: [float(v.double().sum()), float(v.double().abs().sum())] for k, v in model.state_dict().items()}
    with open(os.path.join(HERE, "default_init_seed0.json"), "w") as f:
        json.dump(stats, f, indent=0)


if __name__ == "__main__":
    sys.path.insert(0, HERE)
    main()
