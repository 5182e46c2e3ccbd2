"""GPU tests of the drop-in boundary (SURVEY.md section 8b) on the real kernels.

B2: the whisper model-object protocol of shim.py -- forward hooks on ``decoder.blocks[i].cross_attn`` see the layer's ``qk``,
    ``model(mel, tokens)`` broadcasts one token row, the ``kv_cache`` protocol decodes incrementally, ``detect_language``.
B0/B1 (when ``build()`` installed the reference package into ``oracle/_ref/``, oracle/reference_install.py): the UNMODIFIED
    ``Aligner`` / ``Refiner`` drive the B200 closures through ``model.align`` / ``align_words`` / ``refine``; the results must equal what the reference's own entry
    points produce over the CPU oracle model (words +-20 ms, probabilities 2e-3).
``locate``, ``transcribe`` and the word-timestamp variants are compared with what the unmodified reference produced over the
    CPU oracle model on the same seeded inputs (tests/golden/reference_results.json, oracle/make_golden_reference.py)."""
import copy
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "reference_results.json")


def _golden(*keys):
    import json
    with open(GOLD) as f:
        d = json.load(f)
    for k in keys:
        d = d[k]
    return d


def _gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _models(name="tiny", seed=5):
    import oracle.whisper_ref as W
    from stable_ts_b200.api import modify_model
    from stable_ts_b200.model import from_oracle
    om = W.build_model(name, seed=seed)
    gm = modify_model(from_oracle(om))
    gm.random_init = True
    return W, om, gm


def test_protocol_hooks_logits_and_kv_cache():
    _gpu()
    from oracle import stable_path as SP
    W, om, gm = _models()
    otk = W.tokenizer.get_tokenizer(True, num_languages=om.num_languages, language="en", task="transcribe")
    audio = SP.synth_audio(300000, seed=3)
    mel_ref = W.pad_or_trim(W.log_mel_spectrogram(audio, 80, padding=180000), 3000)
    script = SP.synth_token_script(12, otk.eot, seed=8)
    row = torch.tensor([SP.alignment_token_row(otk, script)])
    # --- exactly what stable_whisper/timing.py:50-61 does, on the B200 object
    qks = [None] * gm.dims.n_text_layer
    hooks = [blk.cross_attn.register_forward_hook(lambda _m, _i, outs, i=i: qks.__setitem__(i, outs[-1]))
             for i, blk in enumerate(gm.decoder.blocks)]
    xa = gm.encoder(mel_ref.cuda().unsqueeze(0))
    logits = gm.decoder(row.cuda(), xa)
    for h in hooks:
        h.remove()
    with torch.no_grad():
        xa_ref, qks_ref, logits_ref, _ = SP.window_qks(om, otk, script, mel_ref)
    rel = lambda a, b: ((a.double().cpu() - b.double()).abs().max() / b.double().abs().max()).item()
    assert rel(xa[0], xa_ref[0]) < 1e-3 and rel(logits[0], logits_ref) < 1e-3
    for l in range(gm.dims.n_text_layer):
        assert qks[l].shape == qks_ref[l].shape and rel(qks[l], qks_ref[l]) < 1e-3
    # no hooks registered -> same logits, nothing captured
    assert torch.allclose(gm.decoder(row.cuda(), xa), logits)
    # model(mel[2], tokens[1]) broadcasts the token row (alignment.py:667)
    two = gm(torch.stack([mel_ref, mel_ref.flip(-1)]).cuda(), row.cuda())
    assert two.shape[0] == 2 and rel(two[0], logits_ref) < 1e-3
    # --- kv_cache protocol: prefix in one call, then token by token == teacher-forced rows
    kv, hk = gm.install_kv_cache_hooks()
    first = gm.decoder(row[:, :4].cuda(), xa, kv_cache=kv)
    step = [gm.decoder(row[:, i:i + 1].cuda(), xa, kv_cache=kv)[:, 0] for i in range(4, row.shape[1])]
    inc = torch.cat([first[0], torch.stack(step, 1)[0]])
    assert rel(inc, logits_ref) < 1e-3 and torch.equal(inc.argmax(-1).cpu(), logits_ref.argmax(-1))
    kv.clear()
    again = gm.decoder(row[:, :4].cuda(), xa, kv_cache=kv)
    assert torch.allclose(again, first)
    # --- detect_language: same distribution as the oracle's
    from oracle.whisper_ref.decoding import detect_language
    tok_ref, probs_ref = detect_language(om, mel_ref)
    tok, probs = gm.detect_language(mel_ref.cuda())
    assert int(tok) == int(tok_ref)
    top = max(probs_ref, key=probs_ref.get)
    assert abs(probs[top] - probs_ref[top]) <= 2e-3 * probs_ref[top]


@pytest.fixture
def ref_env():
    """The reference package importable (from oracle/_ref/) for the test that drives its control plane, and no longer
    afterwards: the other tests check this package's own result classes."""
    _gpu()
    from oracle import reference_install
    root = reference_install.path()
    if root is None:
        pytest.skip("the reference package (stable-ts) is not installed in oracle/_ref/")
    import oracle.whisper_ref as W
    W.install_as_whisper()                    # the reference imports `whisper`; the CPU oracle restates it
    sys.path.insert(0, root)
    try:
        import stable_whisper  # noqa: F401
        yield _ref_inputs()
    finally:
        sys.path.remove(root)
        for name in [m for m in sys.modules if m == "stable_whisper" or m.startswith("stable_whisper.")]:
            del sys.modules[name]


def _ref_inputs():
    from oracle import stable_path as SP
    W, om, gm = _models()
    otk = W.tokenizer.get_tokenizer(True, num_languages=om.num_languages, language="en", task="transcribe")
    audio = torch.cat([SP.synth_gapped_audio(400000, seed=11), SP.synth_audio(300000, seed=12)])
    words = SP.words_from_script(SP.synth_token_script(70, otk.eot, seed=13))
    return dict(om=om, gm=gm, audio=audio, text="".join(otk.decode(w) for w in words))


def _close(a, b):
    da, db = a.to_dict(), b.to_dict()
    assert len(da["segments"]) == len(db["segments"]) and len(da["segments"]) > 0
    worst, n = 0.0, 0
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["text"] == sb["text"]
        wa_, wb_ = sa.get("words") or [], sb.get("words") or []
        assert len(wa_) == len(wb_)
        for wa, wb in zip(wa_, wb_):
            assert wa["word"] == wb["word"] and wa["tokens"] == wb["tokens"]
            worst = max(worst, abs(wa["start"] - wb["start"]), abs(wa["end"] - wb["end"]))
            assert abs(wa["probability"] - wb["probability"]) <= 2e-3 * wb["probability"] + 1e-12
            n += 1
    assert worst <= 0.0201, worst
    return n, worst


def test_unmodified_aligner_and_refiner_over_b200_kernels(ref_env):
    import stable_whisper.alignment as ref_align
    om, gm, audio, text = ref_env["om"], ref_env["gm"], ref_env["audio"], ref_env["text"]
    theirs = ref_align.align(om, audio, text, language="en", verbose=None, ignore_compatibility=True)
    mine = gm.align(audio, text, language="en", verbose=None)
    assert type(mine).__module__.startswith("stable_whisper")
    n, worst = _close(mine, theirs)
    print(f"align: {n} words through the unmodified Aligner on B200 kernels, worst |dt| {worst * 1e3:.0f} ms")
    segs = [dict(start=s.start, end=s.end, text=s.text) for s in theirs.segments]
    n, worst = _close(gm.align_words(audio, copy.deepcopy(segs), language="en", verbose=None),
                      ref_align.align_words(om, audio, copy.deepcopy(segs), language="en", verbose=None, ignore_compatibility=True))
    print(f"align_words: {n} words, worst |dt| {worst * 1e3:.0f} ms")
    r_theirs = ref_align.refine(om, audio, copy.deepcopy(theirs), verbose=None, precision=0.2)
    r_mine = gm.refine(audio, copy.deepcopy(theirs), verbose=None, precision=0.2)
    n, worst = _close(r_mine, r_theirs)
    moved = sum(a.start != b.start or a.end != b.end for a, b in zip(r_mine.all_words(), theirs.all_words()))
    print(f"refine: {n} words, {moved} boundaries moved, worst |dt| vs the reference's vanilla closure {worst * 1e3:.0f} ms")


@pytest.mark.parametrize("mode,thr", [(2, 0.5), (0, 0.0), (1, 0.0)])
def test_locate_matches_reference_over_oracle(mode, thr):
    _gpu()
    from oracle import stable_path as SP
    _, _, gm = _models()
    audio = torch.cat([SP.synth_gapped_audio(400000, seed=11), SP.synth_audio(300000, seed=12)])
    text = [700, 901, 333]
    kw = dict(count=3, mode=mode, probability_threshold=thr, exact_token=True, max_token_per_seg=8)
    theirs = _golden("boundary", "locate", f"{mode}|{thr}")
    mine = gm.locate(audio, text, "en", **kw)
    assert len(mine) == len(theirs) and len(mine) > 0
    for a, b in zip(mine, theirs):
        if mode == 2:
            assert abs(a["target_end"] - b["target_end"]) <= 0.0201
        elif mode == 1:
            assert abs(a["end"] - b["end"]) <= 0.0201
            assert [w["tokens"] for w in a["duration_window_word"]] == [w["tokens"] for w in b["duration_window_word"]]
        else:
            da, db = a.to_dict(), b
            assert [w["tokens"] for w in da["words"]] == [w["tokens"] for w in db["words"]]
            assert max(max(abs(x["start"] - y["start"]), abs(x["end"] - y["end"])) for x, y in zip(da["words"], db["words"])) <= 0.0201


def test_transcribe_method_returns_result_object():
    """model.transcribe(audio) -> WhisperResult with the reference's dict schema (built-in batched driver)."""
    _gpu()
    from oracle import stable_path as SP
    W, om, gm = _models("tiny.en", seed=3)
    audio = torch.cat([SP.synth_audio(480000, seed=21), SP.synth_audio(200000, seed=22)])
    res = gm.transcribe(audio, language="en", regroup=False, sample_len=40, temperature=0.0, suppress_silence=False)
    d = res.to_dict()
    assert set(("text", "segments", "language")) <= set(d) and d["language"] == "en"
    # first window == the oracle's transcribe_window of the same samples (free-running greedy decode)
    otk = W.tokenizer.get_tokenizer(False)
    ref, _ = SP.transcribe_window(om, otk, audio[:480000], language="en", sample_len=40, max_instant_words=0.5)
    mine = [s for s in d["segments"] if s["start"] < 30.0 and s["seek"] == 0.0]
    if ref:     # (WhisperResult.to_dict lists a segment's TEXT tokens -- its words' tokens -- without the timestamp tokens)
        assert [s["tokens"] for s in mine[: len(ref)]] == [[t for t in s["tokens"] if t < otk.eot] for s in ref]


def _extreme_uniforms(pass_index, n_seq, rows=64):
    """u = 0 (first token with probability > 0) or 1 - 2^-24 (last one), alternating over sequences and passes: the drawn
    token then depends on the logit FILTERS only, never on a near-tie of two running sums, so the CPU oracle and the GPU
    draw the same tokens although their logits differ by ~1e-5 relative.  oracle/make_golden_reference.py fed the same
    table, through the draw rule of ``stb_sample`` (first index whose running probability exceeds u), to the reference."""
    hi = 1.0 - 2.0 ** -24
    row = torch.tensor([0.0 if (s + pass_index) % 2 == 0 else hi for s in range(n_seq)], dtype=torch.float64)
    return row.repeat(rows, 1)


@pytest.mark.parametrize("temps,carry", [((0.0, 0.4), True), ((0.0, 0.8), True), ((0.0, 0.4), False)])
def test_transcribe_fallback_and_prompt_carry_match_unmodified_reference(temps, carry):
    """Whole-audio ``transcribe`` (one sequential shard) == the UNMODIFIED transcribe_stable over the CPU oracle model, its
    sampler drawing from the same ``_extreme_uniforms``: temperature fallback with best_of draws (original_whisper.py:349-393),
    prompt carry-over and its reset after a window decoded above temperature 0.5 (:533,696-698), data-dependent seek (:703-710)."""
    _gpu()
    from oracle import stable_path as SP
    _, _, gm = _models("tiny.en", seed=3)
    audio = torch.cat([SP.synth_audio(480000, seed=21), SP.synth_audio(330000, seed=22)])
    ref = _golden("transcribe", f"fallback_extreme|{temps}|{carry}")
    n_ref_passes = ref["passes"]
    # --- B200 side: same uniforms, pass by pass
    calls = []

    def source(ti, steps, n_seq):
        calls.append(ti)
        return _extreme_uniforms(len(calls) - 1, n_seq, rows=steps).float()
    mine = gm.transcribe(audio, language="en", temperature=temps, best_of=2, condition_on_previous_text=carry, regroup=False,
                         sample_len=24, shard_seconds=None, batch_windows=1, uniforms=source, suppress_silence=False)
    assert len(calls) == n_ref_passes and n_ref_passes >= 1
    da = mine.to_dict()
    assert len(da["segments"]) == len(ref["segments"])
    for sa, sb in zip(da["segments"], ref["segments"]):
        assert sa["tokens"] == [int(t) for t in sb["tokens"]] and sa["seek"] == sb["seek"]
        assert sa["temperature"] == sb["temperature"]
        assert abs(sa["avg_logprob"] - sb["avg_logprob"]) < 1e-3
        assert len(sa["words"]) == len(sb["words"])
        for wa, wb in zip(sa["words"], sb["words"]):
            assert wa["tokens"] == wb["tokens"]
            assert abs(wa["start"] - wb["start"]) <= 0.0201 and abs(wa["end"] - wb["end"]) <= 0.0201
    print(f"transcribe {temps} carry={carry}: {len(da['segments'])} segments, {n_ref_passes} sampled passes, identical to the reference")


@pytest.mark.parametrize("variant", ["char_split", "extra_models", "extra_models_dynamic"])
def test_timing_variants_match_unmodified_reference(variant):
    """``extra_models`` and the "new" aligner's ``char_split`` (timing.py:177-189,240-253,380-390,442-444) through
    ``add_word_timestamps_stable`` on the kernels vs the unmodified function over the CPU oracle models."""
    _gpu()
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    from stable_ts_b200.model import from_oracle
    from stable_ts_b200.timing import add_word_timestamps_stable
    from stable_ts_b200.tokenizer import get_tokenizer
    om, om2 = W.build_model("tiny", seed=5), W.build_model("tiny", seed=6)
    gm, gm2 = from_oracle(om), from_oracle(om2)
    otk = W.tokenizer.get_tokenizer(True, num_languages=om.num_languages, language="en", task="transcribe")
    tk = get_tokenizer(gm, language="en", task="transcribe", synthetic=True)
    audio = SP.synth_audio(400000, seed=51)
    script = SP.synth_token_script(36, otk.eot, seed=52)
    mine = [dict(seek=0.0, tokens=script[:20]), dict(seek=0.0, tokens=script[20:])]
    if variant == "char_split":
        kw, key = dict(aligner={"char_split": True}), "char_split"
    else:
        dyn = "4,2" if variant.endswith("dynamic") else None
        kw, key = dict(extra_models=[gm2], dynamic_heads=dyn), f"extra_models_{dyn}"
    theirs = _golden("timing_variants", key)
    add_word_timestamps_stable(segments=mine, model=gm, tokenizer=tk, audio=audio, num_samples=400000, **kw)
    n, worst = 0, 0.0
    for a, b in zip(mine, theirs):
        assert len(a["words"]) == len(b["words"]) and len(a["words"]) > 0
        for wa, wb in zip(a["words"], b["words"]):
            assert wa["word"] == wb["word"] and list(wa["tokens"]) == list(wb["tokens"])
            worst = max(worst, abs(wa["start"] - wb["start"]), abs(wa["end"] - wb["end"]))
            assert abs(wa["probability"] - wb["probability"]) <= 2e-3 * abs(wb["probability"])
            n += 1
    print(f"{variant}: {n} words, worst |dt| {worst * 1e3:.0f} ms vs the unmodified reference")
    assert worst <= 0.0201
