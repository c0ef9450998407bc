"""The CPU oracle (oracle/) vs the committed outputs of the live reference (tests/golden): the oracle
must reproduce the reference bit for bit on the model graph / searches (same ATen CPU ops, same float
semantics) and to fp32 round-off on fbank (numpy vs torchaudio FFT)."""
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_fbank_oracle_vs_torchaudio_golden():
    from oracle import fbank_np
    from reverb_b200 import synth
    gold = dict(np.load(os.path.join(GOLDEN, "fbank.npz")))
    assert len(gold) >= 5
    for key, ref in gold.items():
        n = int(key.split("_")[0][1:])
        seed = int(key.split("seed")[1])
        pcm = synth.synth_audio(n / 16000.0 + 1e-9, seed=seed)[:n]
        got = fbank_np.fbank(pcm.astype(np.float32))
        assert got.shape == ref.shape == (1 + (n - 400) // 160, 80)
        np.testing.assert_allclose(got, ref, rtol=0, atol=5e-4)
    assert fbank_np.fbank(np.zeros(399, np.float32)).shape == (0, 80)     # shorter than one window
    silent = fbank_np.fbank(np.zeros(800, np.float32))                    # log floor: log(eps)
    np.testing.assert_allclose(silent, np.log(np.float32(1.1920929e-07)), rtol=1e-6)


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_pipeline_vs_reference_golden(golden_cases, model_dirs, case):
    from oracle import pipeline_ref
    meta, arr = golden_cases[case]
    d, wav = model_dirs[case]
    orc = pipeline_ref.OracleASR(d)
    feats = orc.compute_feats(wav)
    np.testing.assert_allclose(feats[0].numpy(), arr["feats"], rtol=0, atol=5e-4)
    cat = torch.tensor([meta["verbatimicity"], 1.0 - meta["verbatimicity"]])
    ref_feats = torch.from_numpy(arr["feats"]).unsqueeze(0)
    modes = ["ctc_greedy_search", "ctc_prefix_beam_search", "attention_rescoring"]
    for bi, (fb, fl) in enumerate(orc.feats_batcher(ref_feats, meta["chunk_size"], meta["batch_size"])):
        assert fl.tolist() == arr[f"feats_lens_{bi}"].tolist()
        out = orc.decode(modes, fb, fl, 10, ctc_weight=meta["ctc_weight"], reverse_weight=meta["reverse_weight"],
                         cat_embs=cat, return_intermediates=True)
        assert out["_encoder_lens"].tolist() == arr[f"enc_lens_{bi}"].tolist()
        np.testing.assert_array_equal(out["_encoder_out"].numpy(), arr[f"enc_out_{bi}"])
        np.testing.assert_array_equal(out["_ctc_probs"].numpy(), arr[f"ctc_probs_{bi}"])
        g = meta["batches"][bi]
        for b in range(fb.shape[0]):
            assert out["ctc_greedy_search"][b].tokens == g["ctc_greedy_search"][b]["tokens"]
            p, gp = out["ctc_prefix_beam_search"][b], g["ctc_prefix_beam_search"][b]
            assert [list(h) for h in p.nbest] == gp["nbest"]
            assert p.nbest_scores == gp["nbest_scores"]
            assert p.nbest_times == gp["nbest_times"]
            r, gr = out["attention_rescoring"][b], g["attention_rescoring"][b]
            assert list(r.tokens) == gr["tokens"] and r.times == gr["times"]
            assert float(r.score) == gr["score"] and r.confidence == gr["confidence"]
            assert r.tokens_confidence == gr["tokens_confidence"]


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_attention_mode_vs_reference_golden(golden_cases, model_dirs, case):
    """`attention` decode mode (autoregressive beam search, search.py:251-360): the oracle's restatement returns the
    token ids the live reference returned (tests/golden/attention_mode.json, oracle/make_golden_attention.py)."""
    import json
    from oracle import pipeline_ref
    gold = json.load(open(os.path.join(GOLDEN, "attention_mode.json")))["cases"][case]
    meta, arr = golden_cases[case]
    d, _ = model_dirs[case]
    orc = pipeline_ref.OracleASR(d)
    cat = torch.tensor([meta["verbatimicity"], 1.0 - meta["verbatimicity"]])
    ref_feats = torch.from_numpy(arr["feats"]).unsqueeze(0)
    for lp in (0.0, 0.6):
        for bi, (fb, fl) in enumerate(orc.feats_batcher(ref_feats, meta["chunk_size"], meta["batch_size"])):
            out = orc.decode(["attention"], fb, fl, 10, cat_embs=cat, length_penalty=lp)
            assert [list(r.tokens) for r in out["attention"]] == gold[f"length_penalty_{lp}"][bi]


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_bounded_context_encoder_vs_reference_golden(golden_cases, model_dirs, case):
    """decoding_chunk_size > 0 (utils/mask.py:88-197): the oracle's chunk-masked encoder and the searches on top of it
    reproduce the live reference (tests/golden/chunked.*, oracle/make_golden_chunked.py) bit for bit."""
    import json
    from oracle import pipeline_ref
    gold = json.load(open(os.path.join(GOLDEN, "chunked.json")))
    arr_c = dict(np.load(os.path.join(GOLDEN, "chunked.npz")))
    meta, arr = golden_cases[case]
    orc = pipeline_ref.OracleASR(model_dirs[case][0])
    cat = torch.tensor([meta["verbatimicity"], 1.0 - meta["verbatimicity"]])
    ref_feats = torch.from_numpy(arr["feats"]).unsqueeze(0)
    for cs, left in gold["settings"]:
        for bi, (fb, fl) in enumerate(orc.feats_batcher(ref_feats, meta["chunk_size"], meta["batch_size"])):
            out = orc.decode(["ctc_greedy_search", "ctc_prefix_beam_search"], fb, fl, 10, cat_embs=cat,
                             return_intermediates=True, decoding_chunk_size=cs, num_decoding_left_chunks=left)
            np.testing.assert_array_equal(out["_encoder_out"].numpy(), arr_c[f"{case}_c{cs}_l{left}_enc_{bi}"])
            g = gold["cases"][case][f"c{cs}_l{left}"][bi]
            assert [list(r.tokens) for r in out["ctc_greedy_search"]] == g["greedy"]
            assert [list(r.tokens) for r in out["ctc_prefix_beam_search"]] == g["prefix"]


def _resample_cases():
    gold = dict(np.load(os.path.join(GOLDEN, "resample.npz")))
    for key, ref in gold.items():
        rate = int(key.split("_")[0][1:])
        n = int(key.split("_")[1][1:])
        seed = int(key.split("seed")[1])
        yield rate, n, seed, ref


def test_resample_oracle_and_host_table_vs_torchaudio_golden():
    """Resampling front-end (cli/reverb.py:125-128): the oracle's restatement reproduces torchaudio's output bit for
    bit; the product's numpy filter table (reverb_b200/resample.py, the only host math of the GPU resampler) equals
    the oracle's to float32 round-off."""
    from oracle import resample_ref
    from reverb_b200 import synth
    from reverb_b200.resample import resampled_length, sinc_resample_kernel
    for rate, n, seed, ref in _resample_cases():
        pcm = synth.synth_audio(n / 16000.0 + 1e-9, seed=seed)[:n]
        got = resample_ref.resample(torch.from_numpy(pcm.astype(np.float32)).unsqueeze(0), rate, 16000)[0].numpy()
        np.testing.assert_array_equal(got, ref)
        kern_o, orig_o, new_o, width_o = resample_ref.sinc_resample_kernel(rate, 16000)
        kern, orig, new, width = sinc_resample_kernel(rate, 16000)
        assert (orig, new, width) == (orig_o, new_o, width_o) and kern.shape == tuple(kern_o.shape[::2])
        np.testing.assert_allclose(kern, kern_o[:, 0].numpy(), rtol=0, atol=2e-7)
        assert resampled_length(n, orig, new) == ref.shape[0]


def test_log_add_and_collapse_known_answers():
    from oracle import search_ref
    inf = float("inf")
    assert search_ref.log_add([-inf, -inf]) == -inf
    assert search_ref.log_add([-inf, -1.5]) == -1.5
    assert abs(search_ref.log_add([0.0, 0.0]) - 0.6931471805599453) < 1e-15
    assert search_ref.remove_duplicates_and_blank([0, 1, 1, 0, 1, 2, 2, 0, 0, 3]) == [1, 1, 2, 3]
    assert search_ref.remove_duplicates_and_blank([]) == []


def test_reverse_hyps_docstring_example():
    """known-answer from the reference docstring (asr/wenet/transformer/asr_model.py:908-953)."""
    from oracle import model_ref
    sos = eos = 99
    hyps = torch.tensor([[sos, 1, 2, 3], [sos, 9, 8, 4], [sos, 2, eos, eos]])
    lens = torch.tensor([4, 4, 2])
    r = model_ref.reverse_hyps(hyps, lens, eos)
    assert r.tolist() == [[sos, 3, 2, 1], [sos, 4, 8, 9], [sos, 2, eos, eos]]


@pytest.mark.parametrize("case", ["causal_ln", "sym_bn"])
def test_oracle_streaming_cache_pass_vs_reference_golden(golden_cases, model_dirs, case):
    """The literal cache-based chunk-by-chunk restatement (model_ref.encoder_forward_chunk_by_chunk) reproduces the live
    reference's encoder.forward_chunk_by_chunk (tests/golden/streaming.npz); and for a CAUSAL model the single masked
    pass (chunk mask, all frames valid) is the same function — the identity the engine's simulate_streaming relies on."""
    import json
    from oracle import model_ref, pipeline_ref
    gold = json.load(open(os.path.join(GOLDEN, "streaming.json")))
    arr_s = dict(np.load(os.path.join(GOLDEN, "streaming.npz")))
    meta, arr = golden_cases[case]
    orc = pipeline_ref.OracleASR(model_dirs[case][0])
    feats = torch.from_numpy(arr["feats"][:gold["frames"]]).unsqueeze(0)
    cat = torch.tensor([meta["verbatimicity"], 1.0 - meta["verbatimicity"]])
    for cs, left in gold["settings"]:
        want = arr_s[f"{case}_c{cs}_l{left}"]
        with torch.no_grad():
            got = model_ref.encoder_forward_chunk_by_chunk(feats, orc.sd, orc.cfg, cat, cs, left)[0].numpy()
            masked = model_ref.encoder_forward(feats, torch.tensor([gold["frames"]]), orc.sd, orc.cfg, cat, cs, left)[0][0].numpy()
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)
        if meta["causal"]:
            np.testing.assert_allclose(masked, want, rtol=0, atol=2e-5)
        else:
            assert np.abs(masked - want).max() > 1e-2       # non-causal: the chunk-local convolution matters
