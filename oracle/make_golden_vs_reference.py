"""ORACLE tooling (test infrastructure): records what tests/test_oracle_vs_reference.py compares the oracle with, by
running the LIVE reference in the authoring container.

Re-creates the two synthetic models of tests/golden/{causal_ln,sym_bn}.json from their stored seeds and stores
  * the reference model's state_dict key -> shape map and its encoder-layer / decoder class names;
  * per case, the reference's decode() on its own features with settings the other fixtures do not use
    (ctc_weight 0.3, reverse_weight 0.5, beam 7, verbatimicity 0.25; `attention` mode with length_penalty 0.3;
    decoding_chunk_size 12 with one left chunk): shape and SHA-256 of the float32 encoder outputs (compared bit for
    bit) and the hypotheses;
  * the reference's ctc_align + adjust_model_time_offset on the reference's own rescoring hypotheses.
The features are the reference's and are already committed (tests/golden/<case>.npz "feats"); they are re-checked here.
Writes tests/golden/vs_reference.json.  Run from the repo root:  python oracle/make_golden_vs_reference.py
"""
import hashlib
import json
import os
import sys
import tempfile
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import refimport  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
INFOS = {"tasks": ["transcribe"], "langs": ["en"]}


def _f(x):
    return None if x is None else float(x)


def _hyp(r):
    return {"tokens": list(map(int, r.tokens)), "score": _f(r.score), "confidence": _f(r.confidence),
            "tokens_confidence": None if r.tokens_confidence is None else [float(c) for c in r.tokens_confidence],
            "times": r.times}


def _prefix(r):
    return {"nbest": [list(map(int, h)) for h in r.nbest], "nbest_scores": [float(s) for s in r.nbest_scores],
            "nbest_times": r.nbest_times}


def _encoder(t):
    a = np.ascontiguousarray(t.numpy(), dtype=np.float32)
    return {"shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}


def main():
    sys.path.insert(0, ROOT)
    from reverb_b200 import synth
    wenet = refimport.import_reference()
    from wenet.bin.ctc_align import adjust_model_time_offset, ctc_align
    out = {"torch": torch.__version__, "cases": {}}
    for name in ("causal_ln", "sym_bn"):
        meta = json.load(open(os.path.join(GOLDEN, name + ".json")))
        committed_feats = np.load(os.path.join(GOLDEN, name + ".npz"))["feats"]
        d = tempfile.mkdtemp()
        synth.write_model_dir(d, causal=meta["causal"], cnn_module_norm=meta["cnn_module_norm"],
                              seed=meta["model_seed"], blank_rate=meta["blank_rate"])
        wav = synth.write_wav(os.path.join(d, "golden.wav"), synth.synth_audio(meta["audio_seconds"], seed=meta["audio_seed"]))
        m = wenet.load_model(d)
        feats = m.compute_feats(wav, num_mel_bins=80, frame_length=25, frame_shift=10)
        assert np.array_equal(feats[0].numpy(), committed_feats), "reference features drifted from tests/golden"
        if name == "causal_ln":
            ref_sd = m.model.state_dict()
            out["state_dict_shapes"] = {k: list(v.shape) for k, v in ref_sd.items()}
            out["encoder_layer_class"] = type(m.model.encoder.encoders[0]).__name__
            out["decoder_class"] = type(m.model.decoder).__name__
            out["post_processing"] = [
                adjust_model_time_offset(ctc_align(r["tokens"], r["times"], r["tokens_confidence"], m.tokenizer, 40, 1230), 230)
                for batch in meta["batches"] for r in batch["attention_rescoring"]]
        case = {"decode": [], "attention": [], "chunked": []}
        cat = torch.tensor([0.25, 0.75])
        modes = ["ctc_greedy_search", "ctc_prefix_beam_search", "attention_rescoring"]
        with torch.no_grad():
            for bi, (fb, fl) in enumerate(m.feats_batcher(feats, 350, 2)):
                res = m.model.decode(modes, fb, fl, 7, ctc_weight=0.3, reverse_weight=0.5, cat_embs=cat, infos=INFOS)
                enc, _ = m.model._forward_encoder(fb, fl, cat_embs=cat)
                case["decode"].append({"feats_lens": fl.tolist(), "encoder_out": _encoder(enc),
                                       "ctc_greedy_search": [list(map(int, r.tokens)) for r in res["ctc_greedy_search"]],
                                       "ctc_prefix_beam_search": [_prefix(r) for r in res["ctc_prefix_beam_search"]],
                                       "attention_rescoring": [_hyp(r) for r in res["attention_rescoring"]]})
            cat = torch.tensor([0.4, 0.6])
            for bi, (fb, fl) in enumerate(m.feats_batcher(feats, 300, 2)):
                res = m.model.decode(["attention"], fb, fl, 5, length_penalty=0.3, cat_embs=cat, infos=INFOS)
                enc, _ = m.model._forward_encoder(fb, fl, decoding_chunk_size=12, num_decoding_left_chunks=1, cat_embs=cat)
                res_c = m.model.decode(["ctc_prefix_beam_search"], fb, fl, 6, decoding_chunk_size=12, num_decoding_left_chunks=1,
                                       cat_embs=cat, infos=INFOS)
                case["attention"].append({"feats_lens": fl.tolist(), "tokens": [list(map(int, r.tokens)) for r in res["attention"]]})
                case["chunked"].append({"encoder_out": _encoder(enc),
                                        "ctc_prefix_beam_search": [_prefix(r) for r in res_c["ctc_prefix_beam_search"]]})
        out["cases"][name] = case
        print(name, {k: len(v) for k, v in case.items()})
    with open(os.path.join(GOLDEN, "vs_reference.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote vs_reference.json")


if __name__ == "__main__":
    main()
