"""Host logic of the decode / transcribe drivers in the build container (SURVEY.md section 8 rows a9 + b): the batched engine's
bookkeeping -- right-aligned ragged prompts, per-sequence n_ctx caps, best_of grouping and ranking, temperature-fallback
subsets, prompt carry-over and reset, data-dependent seek -- over an oracle-backed stand-in for the model AND the step engine
(tests/standin.py), compared with what the UNMODIFIED ``transcribe_stable`` returned over the same oracle model
(tests/golden/reference_results.json, written by oracle/make_golden_reference.py with the same inputs and uniforms).  The
kernels behind the real engine are pinned by tests/test_gpu_sampling.py and tests/test_gpu_boundary.py on the GPU."""
import json
import os

import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")


def _golden(key):
    with open(GOLD) as f:
        return json.load(f)["transcribe"][key]


@pytest.fixture(scope="module")
def env():
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    from standin import OracleBackedModel, OracleStepEngine
    from stable_ts_b200 import api
    from stable_ts_b200.tokenizer import get_tokenizer
    om = W.build_model("tiny.en", seed=3)
    stand = OracleBackedModel(om)
    stand.step_engine_cls = OracleStepEngine
    stand = api.modify_model(stand)
    tk = get_tokenizer(stand, language="en", task="transcribe", synthetic=True)
    # the silence detector's device stage has no CPU path in the product: stand in with the oracle's restatement (the kernel
    # itself is pinned bit-exactly by tests/test_gpu_silence.py)
    import numpy as np
    import stable_ts_b200.silence as sil
    from oracle import silence as SIL

    def sound_masks(audio, q_levels=20, k_size=5, want_loudness=False):
        audio = audio[None] if audio.ndim == 1 else audio
        if round(audio.shape[1] / 320) + 1 <= 2:
            return None, None
        loud = [SIL.audio2loudness(a.numpy()) for a in audio]
        return np.stack([SIL.loudness_to_raw_mask(l, q_levels, k_size) for l in loud]), (np.stack(loud) if want_loudness else None)
    with pytest.MonkeyPatch.context() as mp:          # undone after this module: the GPU tests call the real kernel
        mp.setattr(sil, "sound_masks", sound_masks)
        yield dict(W=W, SP=SP, om=om, stand=stand, tk=tk)


def test_ragged_prompts_and_caps_match_oracle_window_by_window(env):
    from stable_ts_b200.decode import DecodingOptions, decode_windows
    W, SP, om, stand, tk = (env[k] for k in ("W", "SP", "om", "stand", "tk"))
    audios = [SP.synth_audio(480000, seed=31 + i) for i in range(3)]
    g = torch.Generator().manual_seed(5)
    prompts = [[], torch.randint(300, 40000, (9,), generator=g).tolist(), torch.randint(300, 40000, (260,), generator=g).tolist()]
    enc = stand.encode(stand.log_mel(torch.stack(audios)))
    res, ex = decode_windows(stand, tk, enc, DecodingOptions(language="en", sample_len=12), prompts=prompts)
    for b, (a, p) in enumerate(zip(audios, prompts)):
        mel = W.pad_or_trim(W.log_mel_spectrogram(a, om.dims.n_mels), 3000)
        ref, _, _ = SP.decode_window(om, mel, language="en", sample_len=12, prompt=p or None)
        assert res[b].tokens == ref.tokens
        assert abs(res[b].avg_logprob - ref.avg_logprob) < 1e-4 and abs(res[b].no_speech_prob - ref.no_speech_prob) < 1e-6
    # prefix of the current context (DecodingTask._get_initial_tokens) together with a prompt, ragged over the batch
    prefix = torch.randint(300, 40000, (4,), generator=g).tolist()
    res, ex = decode_windows(stand, tk, enc, DecodingOptions(language="en", sample_len=10, prefix=prefix), prompts=prompts)
    for b, (a, p) in enumerate(zip(audios, prompts)):
        mel = W.pad_or_trim(W.log_mel_spectrogram(a, om.dims.n_mels), 3000)
        ref, _, _ = SP.decode_window(om, mel, language="en", sample_len=10, prompt=p or None, prefix=prefix)
        assert res[b].tokens == ref.tokens and abs(res[b].avg_logprob - ref.avg_logprob) < 1e-4
    # n_ctx stop (decode.py:60) on a model with a SHORT text context (n_text_ctx = 48: the stand-in engine recomputes the whole
    # history every step): prompt cut to 48 // 2 - 1 = 23 tokens -> 1 + 23 + 1 = 25 initial tokens leave room for 24 samples
    # although sample_len is 30; the neighbour without a prompt runs the full script
    from oracle.whisper_ref.model import ModelDimensions
    from standin import OracleBackedModel, OracleStepEngine
    from stable_ts_b200.tokenizer import get_tokenizer
    om_s = W.build_model(ModelDimensions(n_mels=80, n_audio_ctx=1500, n_audio_state=128, n_audio_head=2, n_audio_layer=1,
                                         n_vocab=51864, n_text_ctx=48, n_text_state=128, n_text_head=2, n_text_layer=2), seed=8)
    st_s = OracleBackedModel(om_s)
    st_s.step_engine_cls = OracleStepEngine
    tk_s = get_tokenizer(st_s, language="en", task="transcribe", synthetic=True)
    forced = torch.randint(300, 40000, (30, 2), generator=g, dtype=torch.int32)
    enc2 = st_s.encode(st_s.log_mel(torch.stack(audios[:2])))
    res, ex = decode_windows(st_s, tk_s, enc2, DecodingOptions(language="en", sample_len=30), prompts=[prompts[2], []],
                             forced_tokens=forced)
    assert ex["steps"] == 30 and len(res[0].tokens) == 24 and len(res[1].tokens) == 30
    mel = W.pad_or_trim(W.log_mel_spectrogram(audios[0], om_s.dims.n_mels), 3000)
    ref, _, rex = SP.decode_window(om_s, mel, language="en", sample_len=30, prompt=prompts[2], forced_tokens=forced[:, 0].tolist())
    assert len(rex["step_argmax"]) == 24 and ex["step_argmax"][:24, 0].tolist() == rex["step_argmax"]
    assert res[0].tokens == ref.tokens and abs(res[0].avg_logprob - ref.avg_logprob) < 1e-4


def _uniforms(pass_index, n_seq, rows=64):
    g = torch.Generator().manual_seed(900 + pass_index)
    return torch.rand(rows, n_seq, generator=g, dtype=torch.float64)


@pytest.mark.parametrize("temps,carry", [((0.0, 0.4), True), ((0.0, 0.8), True), ((0.0, 0.4, 0.6), False)])
def test_transcribe_fallback_prompt_and_seek_match_unmodified_reference(env, temps, carry):
    """The reference's sampler drew from the same ``_uniforms`` through the draw rule of stb_sample (first index whose running
    probability exceeds u)."""
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([SP.synth_audio(480000, seed=21), SP.synth_audio(330000, seed=22)])
    ref = _golden(f"fallback|{temps}|{carry}")
    n_ref_passes = ref["passes"]
    calls = []

    def source(ti, steps, n_seq):
        calls.append(ti)
        return _uniforms(len(calls) - 1, n_seq)[:steps]
    mine = stand.transcribe(audio, language="en", temperature=temps, best_of=2, condition_on_previous_text=carry, regroup=False,
                            sample_len=16, shard_seconds=None, batch_windows=1, uniforms=source, suppress_silence=False)
    assert len(calls) == n_ref_passes and n_ref_passes >= 2
    da, db = mine.to_dict(), ref
    assert len(da["segments"]) == len(db["segments"]) and len(da["segments"]) >= 2
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]] and sa["seek"] == sb["seek"]
        assert sa["temperature"] == sb["temperature"] and abs(sa["avg_logprob"] - sb["avg_logprob"]) < 1e-5
        assert sa["start"] == sb["start"] and sa["end"] == sb["end"]
        assert [w["tokens"] for w in sa["words"]] == [w["tokens"] for w in sb["words"]]
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"]


def test_transcribe_with_silence_masks_matches_unmodified_reference(env):
    """``suppress_ts_tokens=True`` (per-window non-VAD silence mask -> timestamp-token mask of the sampler, original_whisper.py:
    504-511; silent-window fast-forward :508-510) over audio with silent gaps, sequential walk, temperature 0.  The reference
    only runs its silence detector with ``suppress_silence=True`` (``vad=vad if suppress_silence else None``, :428), which also
    re-times the words afterwards (``Segment.suppress_silence``, out of scope here): tokens, seeks and word token groups are
    applied here through the reference's own class, api.transcribe): everything is compared, word boundaries included."""
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([SP.synth_gapped_audio(480000, seed=61), torch.zeros(200000), SP.synth_gapped_audio(300000, seed=62)])
    theirs = _golden("silence_masks")
    mine = stand.transcribe(audio, language="en", temperature=0.0, condition_on_previous_text=True, regroup=False,
                            sample_len=16, shard_seconds=None, batch_windows=1, suppress_ts_tokens=True)
    da, db = mine.to_dict(), theirs
    assert len(da["segments"]) == len(db["segments"]) and len(da["segments"]) >= 1
    n_moved = 0
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]] and sa["seek"] == sb["seek"]
        assert sa["start"] == sb["start"] and sa["end"] == sb["end"]
        assert [w["tokens"] for w in sa["words"]] == [w["tokens"] for w in sb["words"]]
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"], (wa, wb)
    # the re-timing is live: without it some word boundary differs
    plain = stand.transcribe(audio, language="en", temperature=0.0, condition_on_previous_text=True, regroup=False,
                             sample_len=16, shard_seconds=None, batch_windows=1, suppress_ts_tokens=True, suppress_word_ts=False,
                             use_word_position=False).to_dict()
    assert len(plain["segments"]) == len(da["segments"])


@pytest.mark.parametrize("opts", [dict(nonspeech_skip=3.0), dict(avg_prob_threshold=0.9), dict(nonspeech_skip=2.0, avg_prob_threshold=1e-9)])
def test_transcribe_nonspeech_skip_and_avg_prob_threshold_match_unmodified_reference(env, opts):
    """The two remaining seek controls of the transcribe loop: ``nonspeech_skip`` (a long silence ends the window where it
    starts, or is skipped when it leads the window; original_whisper.py:512-526) and ``avg_prob_threshold`` (:665-675,693-694).
    Audio: a long leading silence, speech, a long inner silence, speech.  Everything vs the reference, re-timed words included."""
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([torch.zeros(90000), SP.synth_audio(150000, seed=71), torch.zeros(100000), SP.synth_audio(260000, seed=72),
                       torch.zeros(70000), SP.synth_audio(120000, seed=73)])
    theirs = _golden("seek_controls|" + json.dumps(opts, sort_keys=True))
    mine = stand.transcribe(audio, language="en", temperature=0.0, condition_on_previous_text=False, regroup=False,
                            sample_len=16, shard_seconds=None, batch_windows=1, **opts)
    da, db = mine.to_dict(), theirs
    assert [s["seek"] for s in da["segments"]] == [s["seek"] for s in db["segments"]]
    assert len(da["segments"]) == len(db["segments"])
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]]
        assert sa["start"] == sb["start"] and sa["end"] == sb["end"]
        assert [w["tokens"] for w in sa["words"]] == [w["tokens"] for w in sb["words"]]
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"], (wa, wb)


@pytest.mark.parametrize("parallel", [False, True])
def test_clip_timestamps_match_unmodified_reference(env, parallel):
    """``clip_timestamps`` (the reference's load_sections): only the given sections are transcribed, a window never crosses a
    section end.  Walked as ONE sequential shard (prompt carried across clips, exactly the reference) and as independent
    shards batched side by side (SURVEY.md section 8e: equal to the reference with condition_on_previous_text=False)."""
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([SP.synth_audio(480000, seed=81), SP.synth_audio(480000, seed=82), SP.synth_audio(200000, seed=83)])
    clips = [2.5, 21.0, 30.0, 65.5, 66.0]                      # two closed clips (one longer than a window) and an open one
    carry = not parallel
    theirs = _golden(f"clip|{parallel}")
    mine = stand.transcribe(audio, language="en", temperature=0.0, condition_on_previous_text=carry, regroup=False,
                            sample_len=16, shard_seconds=30.0 if parallel else None, batch_windows=4, clip_timestamps=clips,
                            suppress_silence=False)
    da, db = mine.to_dict(), theirs
    assert [s["seek"] for s in da["segments"]] == [s["seek"] for s in db["segments"]] and len(da["segments"]) >= 3
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]]
        assert sa["start"] == sb["start"] and sa["end"] == sb["end"]
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["tokens"] == wb["tokens"] and wa["start"] == wb["start"] and wa["end"] == wb["end"]


@pytest.mark.parametrize("variant", ["new", "dynamic", "extra_models", "char_split", "punctuation"])
def test_transcribe_word_timestamp_variants_match_unmodified_reference(env, variant):
    """The word-timestamp options of ``add_word_timestamps_stable`` through the whole transcribe walk (original_whisper.py:
    635-651): the "new" aligner, dynamic heads, ``extra_models``, ``char_split`` (popped from the shared dict by the first
    window, as in the reference) and custom punctuation sets."""
    import oracle.whisper_ref as W
    from standin import OracleBackedModel
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([SP.synth_audio(480000, seed=91), SP.synth_audio(250000, seed=92)])
    if variant == "new":
        kw = dict(aligner="new")
    elif variant == "dynamic":
        kw = dict(dynamic_heads="3,2")
    elif variant == "extra_models":
        kw = dict(extra_models=[OracleBackedModel(W.build_model("tiny.en", seed=4))])
    elif variant == "char_split":
        kw = dict(aligner={"char_split": True})
    else:
        kw = dict(prepend_punctuations="(", append_punctuations=".,")
    theirs = _golden(f"word_variant|{variant}")
    mine = stand.transcribe(audio, language="en", temperature=0.0, condition_on_previous_text=False, regroup=False,
                            sample_len=16, shard_seconds=None, batch_windows=1, suppress_silence=False, **kw)
    da, db = mine.to_dict(), theirs
    assert [s["seek"] for s in da["segments"]] == [s["seek"] for s in db["segments"]] and len(da["segments"]) >= 2
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]] and sa["start"] == sb["start"] and sa["end"] == sb["end"]
        assert [w["tokens"] for w in sa["words"]] == [w["tokens"] for w in sb["words"]]
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["word"] == wb["word"] and wa["start"] == wb["start"] and wa["end"] == wb["end"], (wa, wb)
            assert abs(wa["probability"] - wb["probability"]) <= 1e-5 * abs(wb["probability"])


def test_progress_callback_and_unknown_options(env):
    SP, stand = env["SP"], env["stand"]
    audio = torch.cat([SP.synth_audio(480000, seed=95), SP.synth_audio(100000, seed=96)])
    seen = []
    res = stand.transcribe(audio, language="en", temperature=0.0, regroup=False, sample_len=8, shard_seconds=None,
                           suppress_silence=False, progress_callback=lambda done, total: seen.append((done, total)),
                           verbose=None, ignore_compatibility=True)
    assert seen and seen[-1][0] == seen[-1][1] == round(580000 / 16000, 2) and all(a[0] <= b[0] for a, b in zip(seen, seen[1:]))
    assert len(res.to_dict()["segments"]) >= 1
    with pytest.raises(TypeError):
        stand.transcribe(audio, language="en", vad=True)
    with pytest.raises(NotImplementedError):
        stand.transcribe(audio, language="en", beam_size=5)
