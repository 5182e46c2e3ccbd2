"""The oracle's restatement of the reference's orchestration equals what the UNMODIFIED reference, executed on top of
oracle.whisper_ref, returned for the same seeded inputs (tests/golden/reference_results.json, written by
oracle/make_golden_reference.py).  Token ids and timings must be equal; probabilities agree to PROB_RTOL, because the fp32
sums of the CPU model are split differently with the host's thread count and vector width, so the same arithmetic on another
host differs in the last bits."""
import json
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")
PROB_RTOL = 1e-5


@pytest.fixture(scope="module")
def ref():
    import oracle.whisper_ref as W
    with open(GOLD) as f:
        return W, json.load(f)["oracle_vs_reference"]


@pytest.mark.parametrize("name,dyn,aligner", [("tiny.en", None, "legacy"), ("tiny", None, "legacy"),
                                              ("tiny.en", True, "legacy"), ("tiny", "4,2", "legacy"),
                                              ("tiny.en", None, "new")])
def test_align_closure_identical(ref, name, dyn, aligner):
    from oracle import stable_path as SP
    W, gold = ref
    model = W.build_model(name, seed=1)
    tk = W.tokenizer.get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en",
                                   task="transcribe")
    script = SP.synth_token_script(30, tk.eot)
    wts = SP.words_from_script(script)
    words = [tk.decode(w) for w in wts]
    audio = SP.synth_audio(200000)
    r = gold["align"][f"{name}|{dyn}|{aligner}"]
    m = SP.align_audio_window(model, tk, wts, audio, words=words, dynamic_heads=dyn, aligner=aligner)
    assert len(r) == len(m)
    for a, b in zip(r, m):
        assert a["start"] == b["start"] and a["end"] == b["end"] and a["tokens"] == b["tokens"]
        assert abs(a["probability"] - b["probability"]) <= PROB_RTOL * abs(a["probability"])


def test_refine_and_decode_identical(ref):
    from oracle import stable_path as SP
    W, gold = ref
    model = W.build_model("tiny", seed=2)
    tk = W.tokenizer.get_tokenizer(True, num_languages=model.num_languages, language="en", task="transcribe")
    script = SP.synth_token_script(20, tk.eot)
    a2 = torch.stack([SP.synth_audio(160000, seed=1), SP.synth_audio(160000, seed=2)])
    probs = SP.refine_token_probs(model, tk, a2, script)
    want = gold["refine_probs"]                  # a seeded sample of the [2, N, eot] probability tensor
    assert list(probs.shape) == want["shape"]
    np.testing.assert_allclose(probs.flatten()[want["index"]].double().numpy(), want["values"], rtol=PROB_RTOL, atol=0)
    mel = W.pad_or_trim(W.log_mel_spectrogram(a2[0], 80, padding=320000), 3000)
    mask = torch.zeros(1501, dtype=torch.bool)
    mask[50:700] = True
    r = gold["decode"]
    m, _, _ = SP.decode_window(model, mel, ts_token_mask=mask, language="en", sample_len=16)
    assert r["tokens"] == m.tokens
    assert abs(r["avg_logprob"] - m.avg_logprob) <= PROB_RTOL * abs(r["avg_logprob"])
    assert abs(r["no_speech_prob"] - m.no_speech_prob) <= PROB_RTOL * r["no_speech_prob"]


@pytest.mark.parametrize("name,n_samples", [("tiny.en", 300000), ("tiny", 480000)])
def test_transcribe_window_identical(ref, name, n_samples):
    """SP.transcribe_window (decode -> slicing -> gap-padded word timestamps) == the first window of the UNMODIFIED
    transcribe_stable (original_whisper.py:492-710), captured at its add_word_timestamps_stable call."""
    from oracle import stable_path as SP
    W, gold = ref
    model = W.build_model(name, seed=3)
    tk = W.tokenizer.get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en",
                                   task="transcribe")
    audio = SP.synth_audio(n_samples, seed=21)
    mine, ex = SP.transcribe_window(model, tk, audio, language="en", sample_len=40)
    theirs = gold["transcribe_window"][name]
    assert len(mine) == len(theirs) and len(mine) > 0
    for a, b in zip(mine, theirs):
        assert a["tokens"] == [int(t) for t in b["tokens"]]
        assert a["start"] == b["start"] and a["end"] == b["end"] and a["text"] == b["text"]
        assert len(a["words"]) == len(b["words"])
        for wa, wb in zip(a["words"], b["words"]):
            assert wa["word"] == wb["word"] and wa["tokens"] == wb["tokens"]
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"]
            assert abs(wa["probability"] - wb["probability"]) <= PROB_RTOL * abs(wb["probability"])
