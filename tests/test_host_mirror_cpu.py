"""CPU tests of the host-side mirror (stable-ts_b200/timing.py, transcribe.py, tokenizer.py): the bookkeeping the
reference keeps in Python (SURVEY.md section 8 rows a7/a8) must behave exactly like the reference's own functions: their
results on the same inputs are stored in tests/golden/reference_results.json (oracle/make_golden_reference.py)."""
import json
import os
import random

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")


def _tok(multilingual=True):
    from stable_ts_b200.tokenizer import get_tokenizer
    return get_tokenizer(multilingual=multilingual, num_languages=100 if multilingual else 99, language="en",
                         task="transcribe", synthetic=True)


def _random_tokens(tk, n, seed):
    rng = random.Random(seed)
    out = []
    for _ in range(n):
        r = rng.random()
        if r < 0.08:
            out.append(rng.choice([ord(","), ord("."), ord("!"), ord("?"), ord('"'), ord("("), ord(")")]))
        elif r < 0.12:
            out.extend([32, rng.choice([ord("-"), ord('"')])])
        else:
            out.append(rng.randrange(256, tk.eot))
    return out


@pytest.fixture(scope="module")
def ref():
    with open(GOLD) as f:
        return json.load(f)["host_mirror"]


def _lists(x):
    """tuples -> lists, as the stored JSON holds them"""
    return [_lists(v) for v in x] if isinstance(x, (list, tuple)) else x


@pytest.mark.parametrize("seed", range(6))
def test_split_tokens_and_split_word_tokens_equal_reference(ref, seed):
    from stable_ts_b200 import timing as mine
    tk = _tok()
    toks = _random_tokens(tk, 40, seed)
    want = ref["split"][str(seed)]
    assert _lists(mine._split_tokens(toks, tk)) == want["split_tokens"]
    segs = [dict(tokens=_random_tokens(tk, 12, seed * 10 + i)) for i in range(3)]
    for pad_first in (True, False):
        a = _lists(mine.split_word_tokens([dict(s) for s in segs], tk, padding=" ...", pad_first_seg=pad_first))
        b = want["split_word_tokens"][str(pad_first)]
        assert a[0] == b[0] and a[1][0] == b[1][0] and a[1][1] == b[1][1] and a[2] == b[2]


@pytest.mark.parametrize("seed", range(6))
def test_merge_punctuations_and_pop_empty_equal_reference(ref, seed):
    from stable_ts_b200 import timing as mine
    tk = _tok()
    rng = random.Random(seed)
    toks = _random_tokens(tk, 30, 100 + seed)
    words, groups = tk.split_to_word_tokens(toks)

    def build(cls):
        t, out = 0.0, []
        for w, g in zip(words, groups):
            d = rng.random()
            out.append(cls(w, list(g), t, t + d, rng.random()))
            t += d
        return out
    rng = random.Random(seed)
    a = build(mine.WordTiming)
    mine.merge_punctuations(a, mine.PREPEND_PUNCT, mine.APPEND_PUNCT)
    assert [[x.word, x.tokens] for x in a] == ref["merge"][str(seed)]
    # gap-padding pseudo-words
    seg_idx = [0, 0, 1, 1, 2]
    mk = lambda cls: [cls(None, [1], 0, 1, 0), cls("a", [2], 1, 2, 0), cls("b", [3], 2, 3, 0), cls(None, [1], 3, 4, 0),
                      cls("c", [4], 4, 5, 0), cls("d", [5], 5, 6, 0), cls(None, [1], 6, 7, 0), cls("e", [6], 7, 8, 0)]
    xa = mk(mine.WordTiming)
    pa = mine.pop_empty_alignment(xa, seg_idx)
    assert [w.word for w in xa] == ref["pop_empty"]["words"]
    assert [[k, v.start] for k, v in sorted(pa.items())] == ref["pop_empty"]["popped"]


def test_word_timings_from_jumps_boundaries():
    from stable_ts_b200.timing import word_timings_from_jumps
    jumps = np.array([0, 10, 25, 25, 40, 90])          # N = 5 tokens -> N + 1 rows
    probs = [0.1, 0.2, 0.3, 0.4, 0.5]
    words, groups = ["a", "bc", "d", "<eot>"], [[1], [2, 3], [4, 5], [99]]
    out = word_timings_from_jumps(jumps, probs, words, groups)
    assert [(w.start, w.end) for w in out] == [(0.0, 0.2), (0.2, 0.5), (0.5, 1.8)]       # EOT pseudo-word dropped by zip
    assert np.allclose([w.probability for w in out], [0.1, 0.25, 0.45])


def test_slice_segments_matches_whisper_rules():
    from stable_ts_b200.transcribe import slice_segments
    tk = _tok()
    tb = tk.timestamp_begin

    class R:
        temperature = 0.0
        avg_logprob = -1.0
        compression_ratio = 1.0
        no_speech_prob = 0.0
    toks = [tb + 0, 300, 301, tb + 100, tb + 100, 302, tb + 250, tb + 250, 303]      # two closed pairs + open tail
    segs, end_pos, _ = slice_segments(toks, tk, time_offset=30.0, segment_duration=30.0, result=R)
    assert [(s["start"], s["end"]) for s in segs] == [(30.0, 32.0), (32.0, 35.0)] and end_pos == 250
    assert segs[0]["tokens"] == toks[:4] and segs[1]["tokens"] == toks[4:7]
    toks = [300, 301, tb + 75]                                                        # single timestamp ending
    segs, end_pos, _ = slice_segments(toks, tk, 0.0, 30.0, R)
    assert len(segs) == 1 and segs[0]["end"] == 1.5 and end_pos == 75
    segs, end_pos, _ = slice_segments([300, 301], tk, 0.0, 12.5, R)                      # no timestamps at all
    assert len(segs) == 1 and (segs[0]["start"], segs[0]["end"]) == (0.0, 12.5) and end_pos == 0


def test_n_frames_uses_bankers_rounding():
    from stable_ts_b200.timing import n_frames_for
    assert n_frames_for(480000) == 1500 and n_frames_for(160) == 0 and n_frames_for(480) == 2 and n_frames_for(800) == 2
    assert n_frames_for(1120) == 4                      # 3.5 -> 4 (even), 2.5 -> 2 above


def test_silence_host_bookkeeping_matches_oracle(monkeypatch):
    """stable_ts_b200.silence: everything after the kernel (run lengths, 0.1 s filter, suppression mask, predictor dict)
    equals the oracle / the fixtures written by the reference when it is fed the oracle's sound masks."""
    import numpy as np
    import torch
    from oracle import silence as SIL
    from oracle.make_golden_silence import CASES, case_audio
    from stable_ts_b200 import silence as S
    rng = np.random.default_rng(5)
    for _ in range(50):
        m = rng.random(int(rng.integers(3, 1502))) < rng.random()
        for off in (0.0, 7.5):
            a, b = S.mask2timing(m, time_offset=off), SIL.mask2timing(m, time_offset=off)
            assert (a is None) == (b is None)
            if a is not None:
                assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
                assert np.array_equal(S.timing2mask(a[0], a[1], len(m), time_offset=off), SIL.timing2mask(b[0], b[1], len(m), time_offset=off))
        x, y = S._silence_from_sound(m), SIL.raw_mask_to_silence_mask(m)
        assert (x is None) == (y is None) and (x is None or np.array_equal(x, y))
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "silence_cases.npz"))
    for i, (n, seed, floor, scale) in enumerate(CASES):
        audio = case_audio(int(n), int(seed), floor, scale)
        loud = SIL.audio2loudness(audio.numpy())

        def fake_sound_masks(a, q_levels=20, k_size=5, want_loudness=False):
            return (None, None) if loud is None else (SIL.loudness_to_raw_mask(loud, q_levels, k_size)[None], None)
        monkeypatch.setattr(S, "sound_masks", fake_sound_masks)
        pred = S.predict_nonvad_batch(audio[None], offsets=[12.5])[0]
        assert (pred["timings"] is not None) == bool(z[f"has_timings_{i}"])
        if pred["timings"] is not None:
            assert np.array_equal(pred["timings"], z[f"timings_{i}"])
        assert pred["is_silent"] == bool(z[f"silent_{i}"])
        assert (pred["mask"] is None) == (z[f"pmask_{i}"].size == 0)
        if pred["mask"] is not None:
            assert pred["mask"].dtype == torch.bool and np.array_equal(pred["mask"].numpy(), z[f"pmask_{i}"])
