"""Fixtures written by the UNMODIFIED reference (a checkout of stable-ts) for the tests that compare against it:
tests/golden/reference_results.json, tests/golden/reference_silence.npz and tests/golden/demo_head.wav.

    python oracle/make_golden_reference.py PATH_TO_STABLE_TS_CHECKOUT

Every case regenerates its inputs from seeds (oracle.whisper_ref models, oracle.stable_path audio and token scripts), runs the
reference on them over oracle.whisper_ref (the reference imports `whisper`; the oracle restates it) and stores what the
reference returned.  The tests rebuild the same inputs and compare this package's results with the stored ones, so the
inputs here and in the tests must stay in step.
"""
import copy
import json
import os
import random
import struct
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
GOLD = os.path.join(ROOT, "tests", "golden")

# inputs shared with the tests
LOCATE_CASES = [(2, 0.5), (0, 0.0), (1, 0.0), (0, 0.5)]
LOCATE_TEXT = [700, 901, 333]
LOCATE_KW = dict(count=3, exact_token=True, max_token_per_seg=8)
SILENCE_LIVE_CASES = [(480000, 101, 0.0, 1.0), (333333, 102, 5e-4, 1.0), (480000, 103, 2e-3, 0.5), (64000, 104, 0.0, 1.0),
                      (480000, 105, 0.0, 1e-7)]
DEMO_HEAD_SECONDS = 0.1


def jsonable(x):
    """Reference outputs -> plain JSON values (numpy / torch scalars and arrays included); floats keep every bit."""
    if isinstance(x, dict):
        return {str(k): jsonable(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [jsonable(v) for v in x]
    if torch.is_tensor(x):
        return jsonable(x.tolist())
    if isinstance(x, np.ndarray):
        return jsonable(x.tolist())
    if isinstance(x, (np.bool_, bool)):
        return bool(x)
    if isinstance(x, np.integer):
        return int(x)
    if isinstance(x, np.floating):
        return float(x)
    return x


def tensor_sample(t: torch.Tensor, n: int = 4096, seed: int = 0) -> dict:
    """A fixed, seeded sample of a large tensor's entries (flat indices + values) and its shape."""
    t = t.detach().contiguous().cpu()
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return dict(shape=list(t.shape), index=idx.tolist(), values=t.flatten()[idx].double().tolist())


def result_segments(res) -> list:
    keys = ("start", "end", "text", "seek", "tokens", "temperature", "avg_logprob", "no_speech_prob")
    out = []
    for s in res.to_dict(keep_orig=False)["segments"]:
        d = {k: s.get(k) for k in keys}
        d["words"] = [{k: w.get(k) for k in ("word", "start", "end", "probability", "tokens")} for w in s.get("words") or []]
        out.append(d)
    return jsonable(out)


def timing_variants(W, SP):
    """tests/test_timing_variants_cpu.py and the timing-variant GPU test: add_word_timestamps_stable over two oracle models."""
    import stable_whisper.timing as ref_timing
    om, om2 = W.build_model("tiny", seed=5), W.build_model("tiny", seed=6)
    otk = W.tokenizer.get_tokenizer(True, num_languages=om.num_languages, language="en", task="transcribe")
    audio = SP.synth_audio(400000, seed=51)
    mel = W.pad_or_trim(W.log_mel_spectrogram(audio, om.dims.n_mels, padding=80000), 3000)
    script = SP.synth_token_script(36, otk.eot, seed=52)
    cases = {"char_split": dict(aligner={"char_split": True}), "char_split_topk10": dict(aligner={"char_split": True, "topk": 10})}
    for dyn in (None, 4, "4,2"):
        cases[f"extra_models_{dyn}"] = dict(extra_models=[om2], dynamic_heads=dyn)
    out = {}
    for name, kw in cases.items():
        segs = [dict(seek=0.0, tokens=script[:20]), dict(seek=0.0, tokens=script[20:])]
        ref_timing.add_word_timestamps_stable(segments=segs, model=om, tokenizer=otk, mel=mel, num_samples=400000,
                                              **{k: copy.deepcopy(v) if isinstance(v, dict) else v for k, v in kw.items()})
        out[name] = jsonable([dict(start=s["start"], end=s["end"],
                                   words=[{k: w[k] for k in ("word", "tokens", "start", "end", "probability")} for w in s["words"]])
                              for s in segs])
    return out


def oracle_vs_reference(W, SP):
    """tests/test_oracle_vs_reference.py: alignment closure, refinement closure, decode_stable, first transcribe window."""
    from stable_whisper.alignment import get_whisper_alignment_func, get_whisper_refinement_func
    from stable_whisper.decode import decode_stable
    from stable_whisper.non_whisper.alignment import WordToken
    import stable_whisper.whisper_word_level.original_whisper as ow
    from whisper.decoding import DecodingOptions
    out = {"align": {}, "transcribe_window": {}}
    for name, dyn, aligner in [("tiny.en", None, "legacy"), ("tiny", None, "legacy"), ("tiny.en", True, "legacy"),
                               ("tiny", "4,2", "legacy"), ("tiny.en", None, "new")]:
        model = W.build_model(name, seed=1)
        tk = W.tokenizer.get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en", task="transcribe")
        wts = SP.words_from_script(SP.synth_token_script(30, tk.eot))
        words = [tk.decode(w) for w in wts]

        class O:
            class align:
                extra_models = None
                dynamic_heads = dyn
        O.align.aligner = aligner
        r = get_whisper_alignment_func(model, tk, None, O)(SP.synth_audio(200000), [WordToken(w, t) for w, t in zip(words, wts)])
        out["align"][f"{name}|{dyn}|{aligner}"] = jsonable([{k: w[k] for k in ("start", "end", "tokens", "probability")} for w in r])
    model = W.build_model("tiny", seed=2)
    tk = W.tokenizer.get_tokenizer(True, num_languages=model.num_languages, language="en", task="transcribe")
    script = SP.synth_token_script(20, tk.eot)
    a2 = torch.stack([SP.synth_audio(160000, seed=1), SP.synth_audio(160000, seed=2)])
    out["refine_probs"] = tensor_sample(get_whisper_refinement_func(model, tk, None)(a2, script))
    mel = W.pad_or_trim(W.log_mel_spectrogram(a2[0], 80, padding=320000), 3000)
    mask = torch.zeros(1501, dtype=torch.bool)
    mask[50:700] = True
    r, _ = decode_stable(model, mel, DecodingOptions(language="en", fp16=False, sample_len=16), ts_token_mask=mask)
    out["decode"] = jsonable(dict(tokens=r.tokens, avg_logprob=r.avg_logprob, no_speech_prob=r.no_speech_prob))
    for name, n_samples in [("tiny.en", 300000), ("tiny", 480000)]:
        model = W.build_model(name, seed=3)
        audio = SP.synth_audio(n_samples, seed=21)
        first = {}
        orig = ow.add_word_timestamps_stable

        def spy(**kw):
            orig(**kw)
            if "segments" not in first:
                first["segments"] = copy.deepcopy(kw["segments"])
        ow.add_word_timestamps_stable = spy
        try:
            ow.transcribe_stable(model, audio, language="en", temperature=0.0, condition_on_previous_text=False,
                                 word_timestamps=True, vad=False, suppress_silence=False, suppress_ts_tokens=False,
                                 regroup=False, verbose=None, fp16=False, ignore_compatibility=True, sample_len=40)
        finally:
            ow.add_word_timestamps_stable = orig
        out["transcribe_window"][name] = jsonable(
            [dict(tokens=[int(t) for t in s["tokens"]], start=s["start"], end=s["end"], text=s["text"],
                  words=[{k: w[k] for k in ("word", "tokens", "start", "end", "probability")} for w in s["words"]])
             for s in first["segments"]])
    return out


def boundary(W, SP):
    """tests/test_boundary_reference_cpu.py (and the locate GPU test): reference locate() and the result dict of align()."""
    import stable_whisper.alignment as ref_align
    model = W.build_model("tiny", seed=5)
    tk = W.tokenizer.get_tokenizer(True, num_languages=model.num_languages, language="en", task="transcribe")
    audio = torch.cat([SP.synth_gapped_audio(400000, seed=11), SP.synth_audio(300000, seed=12)])
    words = SP.words_from_script(SP.synth_token_script(70, tk.eot, seed=13))
    text = "".join(tk.decode(w) for w in words)
    out = {"locate": {}}
    for mode, thr in LOCATE_CASES:
        res = ref_align.locate(model, audio, LOCATE_TEXT, "en", mode=mode, probability_threshold=thr, verbose=None, **LOCATE_KW)
        out["locate"][f"{mode}|{thr}"] = jsonable([r.to_dict() if mode == 0 else r for r in res])
    theirs = ref_align.align(model, audio, text, language="en", verbose=None, ignore_compatibility=True)
    out["align_result"] = jsonable(theirs.to_dict(keep_orig=False))
    return out


class _InvCDF:
    """Categorical stand-in inside the oracle: first index whose running probability exceeds u (as in the tests)."""
    table_for_pass = None
    pass_index = -1
    step = 0

    def __init__(self, logits):
        self.logits = logits

    def sample(self):
        c = torch.softmax(self.logits.double(), -1).cumsum(-1)
        u = _InvCDF.table_for_pass(_InvCDF.pass_index, c.shape[0])[_InvCDF.step]
        _InvCDF.step += 1
        return (c > u[:, None]).to(torch.uint8).argmax(-1)


def uniforms_cpu(pass_index, n_seq, rows=64):
    g = torch.Generator().manual_seed(900 + pass_index)
    return torch.rand(rows, n_seq, generator=g, dtype=torch.float64)


def uniforms_extreme(pass_index, n_seq, rows=64):
    hi = 1.0 - 2.0 ** -24
    row = torch.tensor([0.0 if (s + pass_index) % 2 == 0 else hi for s in range(n_seq)], dtype=torch.float64)
    return row.repeat(rows, 1)


def sampled_transcribe(om, audio, table, **kw):
    """transcribe_stable with the oracle's sampler drawing from `table`; -> (result, number of sampled passes)."""
    import oracle.whisper_ref.decoding as odec
    import stable_whisper.whisper_word_level.original_whisper as ow
    orig_cat, orig_dec = odec.Categorical, ow.decode_stable
    _InvCDF.table_for_pass, _InvCDF.pass_index = table, -1

    def counting_decode(model, seg, options, **k):
        if options.temperature > 0:
            _InvCDF.pass_index += 1
            _InvCDF.step = 0
        return orig_dec(model, seg, options, **k)
    odec.Categorical, ow.decode_stable = _InvCDF, counting_decode
    try:
        res = ow.transcribe_stable(om, audio, **kw)
    finally:
        odec.Categorical, ow.decode_stable = orig_cat, orig_dec
    return res, _InvCDF.pass_index + 1


def transcribe_cases(W, SP):
    """tests/test_decode_host_cpu.py and the transcribe GPU test: the unmodified transcribe_stable over oracle models."""
    import stable_whisper.whisper_word_level.original_whisper as ow
    om = W.build_model("tiny.en", seed=3)
    base = dict(language="en", word_timestamps=True, vad=False, regroup=False, verbose=None, fp16=False, ignore_compatibility=True)
    out = {}
    audio = torch.cat([SP.synth_audio(480000, seed=21), SP.synth_audio(330000, seed=22)])
    for temps, carry in [((0.0, 0.4), True), ((0.0, 0.8), True), ((0.0, 0.4, 0.6), False)]:
        res, n = sampled_transcribe(om, audio, uniforms_cpu, temperature=temps, best_of=2, condition_on_previous_text=carry,
                                    suppress_silence=False, suppress_ts_tokens=False, sample_len=16, **base)
        out[f"fallback|{temps}|{carry}"] = dict(passes=n, segments=result_segments(res))
    for temps, carry in [((0.0, 0.4), True), ((0.0, 0.8), True), ((0.0, 0.4), False)]:
        res, n = sampled_transcribe(om, audio, uniforms_extreme, temperature=temps, best_of=2, condition_on_previous_text=carry,
                                    suppress_silence=False, suppress_ts_tokens=False, sample_len=24, **base)
        out[f"fallback_extreme|{temps}|{carry}"] = dict(passes=n, segments=result_segments(res))
    audio = torch.cat([SP.synth_gapped_audio(480000, seed=61), torch.zeros(200000), SP.synth_gapped_audio(300000, seed=62)])
    res = ow.transcribe_stable(om, audio, temperature=0.0, condition_on_previous_text=True, suppress_silence=True,
                               suppress_ts_tokens=True, sample_len=16, **base)
    out["silence_masks"] = dict(segments=result_segments(res))
    audio = torch.cat([torch.zeros(90000), SP.synth_audio(150000, seed=71), torch.zeros(100000), SP.synth_audio(260000, seed=72),
                       torch.zeros(70000), SP.synth_audio(120000, seed=73)])
    for opts in [dict(nonspeech_skip=3.0), dict(avg_prob_threshold=0.9), dict(nonspeech_skip=2.0, avg_prob_threshold=1e-9)]:
        res = ow.transcribe_stable(om, audio, temperature=0.0, condition_on_previous_text=False, suppress_silence=True,
                                   suppress_ts_tokens=False, sample_len=16, **opts, **base)
        out["seek_controls|" + json.dumps(opts, sort_keys=True)] = dict(segments=result_segments(res))
    audio = torch.cat([SP.synth_audio(480000, seed=81), SP.synth_audio(480000, seed=82), SP.synth_audio(200000, seed=83)])
    for parallel in (False, True):
        res = ow.transcribe_stable(om, audio, temperature=0.0, condition_on_previous_text=not parallel, suppress_silence=False,
                                   suppress_ts_tokens=False, sample_len=16, clip_timestamps=[2.5, 21.0, 30.0, 65.5, 66.0], **base)
        out[f"clip|{parallel}"] = dict(segments=result_segments(res))
    audio = torch.cat([SP.synth_audio(480000, seed=91), SP.synth_audio(250000, seed=92)])
    for variant in ["new", "dynamic", "extra_models", "char_split", "punctuation"]:
        kw = {"new": dict(aligner="new"), "dynamic": dict(dynamic_heads="3,2"),
              "extra_models": dict(extra_models=[W.build_model("tiny.en", seed=4)]), "char_split": dict(aligner={"char_split": True}),
              "punctuation": dict(prepend_punctuations="(", append_punctuations=".,")}[variant]
        res = ow.transcribe_stable(om, audio, temperature=0.0, condition_on_previous_text=False, suppress_silence=False,
                                   suppress_ts_tokens=False, sample_len=16, **kw, **base)
        out[f"word_variant|{variant}"] = dict(segments=result_segments(res))
    return out


def host_mirror():
    """tests/test_host_mirror_cpu.py: token splitting, punctuation merge and gap-padding removal of stable_whisper.timing."""
    import stable_whisper.timing as ref_timing
    from whisper.timing import merge_punctuations as ref_merge
    from test_host_mirror_cpu import _random_tokens, _tok
    tk = _tok()
    out = {"split": {}, "merge": {}}
    for seed in range(6):
        toks = _random_tokens(tk, 40, seed)
        segs = [dict(tokens=_random_tokens(tk, 12, seed * 10 + i)) for i in range(3)]
        out["split"][str(seed)] = jsonable(dict(
            split_tokens=ref_timing._split_tokens(toks, tk),
            split_word_tokens={str(p): ref_timing.split_word_tokens([dict(s) for s in segs], tk, padding=" ...", pad_first_seg=p)
                               for p in (True, False)}))
        rng = random.Random(seed)
        words, groups = tk.split_to_word_tokens(_random_tokens(tk, 30, 100 + seed))
        t, b = 0.0, []
        for w, g in zip(words, groups):
            d = rng.random()
            b.append(ref_timing.WordTiming(w, list(g), t, t + d, rng.random()))
            t += d
        ref_merge(b, "\"'“¿([{-", "\"'.。,，!！?？:：”)]}、")
        out["merge"][str(seed)] = jsonable([(x.word, x.tokens) for x in b])
    W_ = ref_timing.WordTiming
    xb = [W_(None, [1], 0, 1, 0), W_("a", [2], 1, 2, 0), W_("b", [3], 2, 3, 0), W_(None, [1], 3, 4, 0),
          W_("c", [4], 4, 5, 0), W_("d", [5], 5, 6, 0), W_(None, [1], 6, 7, 0), W_("e", [6], 7, 8, 0)]
    pb = ref_timing.pop_empty_alignment(xb, [0, 0, 1, 1, 2])
    out["pop_empty"] = jsonable(dict(words=[w.word for w in xb], popped=sorted((k, v.start) for k, v in pb.items())))
    return out


def silence_live(SP):
    """tests/test_oracle_silence.py: loudness, wav2mask, mask2timing and timing2mask of stable_whisper.stabilization."""
    from stable_whisper.stabilization.nonvad import audio2loudness, wav2mask
    from stable_whisper.stabilization.utils import mask2timing, timing2mask
    out = {"cases": np.array(SILENCE_LIVE_CASES, dtype=np.float64)}
    for i, (n, seed, floor, scale) in enumerate(SILENCE_LIVE_CASES):
        audio = SP.synth_gapped_audio(n, seed=seed, floor=floor) * scale
        out[f"loud_{i}"] = audio2loudness(audio).numpy()
        ref = wav2mask(audio, sr=16000)
        out[f"has_mask_{i}"] = np.array(ref is not None)
        out[f"mask_{i}"] = ref.numpy() if ref is not None else np.zeros(0, bool)
        for j, off in enumerate((None, 3.25)):
            tm = None if ref is None else mask2timing(ref, time_offset=off)
            out[f"has_timing_{i}_{j}"] = np.array(tm is not None)
            if tm is not None:
                out[f"starts_{i}_{j}"], out[f"ends_{i}_{j}"] = np.asarray(tm[0]), np.asarray(tm[1])
                out[f"remask_{i}_{j}"] = timing2mask(tm[0], tm[1], 1501, time_offset=off).numpy()
    return out


def sharding_result():
    """tests/test_sharding_gloo.py: the reference's WhisperResult built from the gathered word-record dict."""
    import stable_whisper
    from test_sharding_gloo import gathered_result_dict
    theirs = stable_whisper.WhisperResult(gathered_result_dict()[0])
    return jsonable(dict(text=theirs.text, words=[w.to_dict() for w in theirs.all_words()]))


def demo_head(reference):
    """The first DEMO_HEAD_SECONDS of examples/demo.wav (44.1 kHz stereo s16), chunks before `data` kept, sizes rewritten."""
    raw = open(os.path.join(reference, "examples", "demo.wav"), "rb").read()
    pos, head = 12, bytearray(raw[:12])
    while True:
        cid, size = raw[pos:pos + 4], struct.unpack("<I", raw[pos + 4:pos + 8])[0]
        if cid == b"data":
            break
        head += raw[pos:pos + 8 + size + (size & 1)]
        pos += 8 + size + (size & 1)
    n = int(DEMO_HEAD_SECONDS * 44100) * 4
    body = raw[pos + 8:pos + 8 + n]
    out = bytes(head) + b"data" + struct.pack("<I", len(body)) + body
    return out[:4] + struct.pack("<I", len(out) - 8) + out[8:]


def main():
    reference = os.path.abspath(sys.argv[1])
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    W.install_as_whisper()
    sys.path.insert(0, reference)
    out = dict(timing_variants=timing_variants(W, SP), oracle_vs_reference=oracle_vs_reference(W, SP), boundary=boundary(W, SP),
               transcribe=transcribe_cases(W, SP), host_mirror=host_mirror(), sharding_result=sharding_result())
    path = os.path.join(GOLD, "reference_results.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"), sort_keys=True)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(GOLD, "reference_silence.npz")
    np.savez_compressed(path, **silence_live(SP))
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(GOLD, "demo_head.wav")
    with open(path, "wb") as f:
        f.write(demo_head(reference))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
