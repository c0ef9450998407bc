"""Pins the oracle and the synthetic-model generator against the live reference's outputs, recorded in
tests/golden/vs_reference.json by oracle/make_golden_vs_reference.py: the reference's state_dict layout, its decode()
with settings the other fixtures do not use, and its CTM post-processing.  Encoder outputs are recorded as the SHA-256
of their float32 bytes: equal digests are the bit-for-bit equality the oracle promises."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref_golden():
    with open(os.path.join(GOLDEN, "vs_reference.json")) as f:
        return json.load(f)


def _assert_bits_equal(want, enc):
    a = np.ascontiguousarray(enc.numpy(), dtype=np.float32)
    assert list(a.shape) == want["shape"]
    assert hashlib.sha256(a.tobytes()).hexdigest() == want["sha256"], "encoder_out differs from the reference's"


def test_synthetic_state_dict_is_strictly_loadable(ref_golden, model_dirs):
    meta = ref_golden
    d, _ = model_dirs["causal_ln"]
    ref_shapes = meta["state_dict_shapes"]
    sd = torch.load(os.path.join(d, "synth.pt"))
    assert set(ref_shapes.keys()) == set(sd.keys())
    for k in sd:
        assert list(sd[k].shape) == ref_shapes[k], k
    assert meta["encoder_layer_class"] == "LanguageSpecificConformerEncoderLayer"
    assert meta["decoder_class"] == "LanguageSpecificBiTransformerDecoder"


def _same_prefix(want, c):
    assert want["nbest"] == [list(h) for h in c.nbest]
    assert want["nbest_scores"] == c.nbest_scores and want["nbest_times"] == c.nbest_times


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_equals_live_reference(ref_golden, model_dirs, golden_cases, case):
    from oracle import pipeline_ref
    meta = ref_golden
    _, garr = golden_cases[case]
    d, wav = model_dirs[case]
    orc = pipeline_ref.OracleASR(d)
    f_ref = torch.from_numpy(garr["feats"]).unsqueeze(0)          # the reference's compute_feats on this wav
    assert (f_ref - orc.compute_feats(wav)).abs().max().item() < 5e-4
    cat = torch.tensor([0.25, 0.75])
    modes = ["ctc_greedy_search", "ctc_prefix_beam_search", "attention_rescoring"]
    batches = list(orc.feats_batcher(f_ref, 350, 2))
    assert len(batches) == len(meta["cases"][case]["decode"])
    for bi, (fb, fl) in enumerate(batches):
        want = meta["cases"][case]["decode"][bi]
        assert fl.tolist() == want["feats_lens"]
        got = orc.decode(modes, fb, fl, 7, ctc_weight=0.3, reverse_weight=0.5, cat_embs=cat, return_intermediates=True)
        _assert_bits_equal(want["encoder_out"], got["_encoder_out"])
        for b in range(fb.shape[0]):
            assert want["ctc_greedy_search"][b] == list(got["ctc_greedy_search"][b].tokens)
            _same_prefix(want["ctc_prefix_beam_search"][b], got["ctc_prefix_beam_search"][b])
            a, c = want["attention_rescoring"][b], got["attention_rescoring"][b]
            assert a["tokens"] == list(c.tokens) and a["score"] == float(c.score)
            assert a["confidence"] == c.confidence and a["tokens_confidence"] == c.tokens_confidence


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_attention_mode_and_bounded_context_equal_live_reference(ref_golden, model_dirs, golden_cases, case):
    """The later restatements — `attention` decode mode (search.py:251-360) and decoding_chunk_size > 0
    (utils/mask.py:88-197) — against the live reference with settings the other fixtures do not use."""
    from oracle import pipeline_ref
    meta = ref_golden
    _, garr = golden_cases[case]
    d, _ = model_dirs[case]
    orc = pipeline_ref.OracleASR(d)
    feats = torch.from_numpy(garr["feats"]).unsqueeze(0)
    cat = torch.tensor([0.4, 0.6])
    batches = list(orc.feats_batcher(feats, 300, 2))
    assert len(batches) == len(meta["cases"][case]["attention"])
    for bi, (fb, fl) in enumerate(batches):
        want = meta["cases"][case]["attention"][bi]
        assert fl.tolist() == want["feats_lens"]
        got = orc.decode(["attention"], fb, fl, 5, cat_embs=cat, length_penalty=0.3)
        assert [list(r.tokens) for r in got["attention"]] == want["tokens"]
        got_c = orc.decode(["ctc_prefix_beam_search"], fb, fl, 6, cat_embs=cat, return_intermediates=True,
                           decoding_chunk_size=12, num_decoding_left_chunks=1)
        want_c = meta["cases"][case]["chunked"][bi]
        _assert_bits_equal(want_c["encoder_out"], got_c["_encoder_out"])
        want_c = want_c["ctc_prefix_beam_search"]
        assert len(want_c) == len(got_c["ctc_prefix_beam_search"])
        for a, c in zip(want_c, got_c["ctc_prefix_beam_search"]):
            _same_prefix(a, c)


def test_oracle_resample_equals_torchaudio():
    import torchaudio
    from oracle import resample_ref
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 7777, generator=g) * 3000
    for rate in (8000, 32000, 44100):
        want = torchaudio.transforms.Resample(orig_freq=rate, new_freq=16000)(x)
        assert torch.equal(resample_ref.resample(x, rate, 16000), want)


def test_host_post_processing_equals_live_reference(ref_golden, golden_cases, model_dirs):
    """reverb_b200's ctc_align / CTM rendering vs the reference's, on the reference's own hypotheses."""
    from reverb_b200 import ctc_align as mine
    from reverb_b200.text import PieceTokenizer
    ref = ref_golden
    meta, _ = golden_cases["causal_ln"]
    d, _ = model_dirs["causal_ln"]
    tok = PieceTokenizer(os.path.join(d, "tk.units.txt"))
    hyps = [r for batch in meta["batches"] for r in batch["attention_rescoring"]]
    assert len(hyps) == len(ref["post_processing"])
    for r, a in zip(hyps, ref["post_processing"]):
        b = mine.adjust_model_time_offset(mine.ctc_align(r["tokens"], r["times"], r["tokens_confidence"], tok, 40, 1230), 230)
        assert a == b
