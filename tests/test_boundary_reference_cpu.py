"""Boundary tests in the build container (SURVEY.md section 8b, B0 + B1): the UNMODIFIED reference control plane
(``stable_whisper.non_whisper.alignment.Aligner`` :252 / ``.refinement.Refiner`` :132, ``WhisperResult``) driven over
``stable_ts_b200``'s plugin closures and bound model methods, with an oracle-backed stand-in for the GPU model's method
surface (tests/standin.py).  Every result must be IDENTICAL to what the reference's own entry points
(``stable_whisper.alignment.align / align_words / refine``) produce with their vanilla closures over the same oracle
model.  The tests that drive ``Aligner`` / ``Refiner`` run the reference package itself, installed into oracle/_ref/ by
``build()`` (oracle/reference_install.py), and skip where it could not be installed;
``locate`` and the result schema are compared with what the reference returned (tests/golden/reference_results.json, written
by oracle/make_golden_reference.py).  tests/test_gpu_boundary.py covers the real kernels."""
import copy
import json
import os
import sys

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")


@pytest.fixture(scope="module")
def env():
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    from standin import OracleBackedModel
    model = W.build_model("tiny", seed=5)
    tk = W.tokenizer.get_tokenizer(True, num_languages=model.num_languages, language="en", task="transcribe")
    audio = torch.cat([SP.synth_gapped_audio(400000, seed=11), SP.synth_audio(300000, seed=12)])
    words = SP.words_from_script(SP.synth_token_script(70, tk.eot, seed=13))
    text = "".join(tk.decode(w) for w in words)
    with open(GOLD) as f:
        gold = json.load(f)["boundary"]
    return dict(W=W, SP=SP, model=model, tk=tk, audio=audio, text=text, stand=OracleBackedModel(model), gold=gold)


@pytest.fixture(scope="module")
def ref_env(env):
    """The reference package importable (from oracle/_ref/) for the rest of this module, and no longer afterwards: the
    other modules test this package's own result classes."""
    from oracle import reference_install
    root = reference_install.path()
    env["W"].install_as_whisper()             # the reference imports `whisper`; the oracle restates it
    if root is not None:
        sys.path.insert(0, root)
    try:
        pytest.importorskip("stable_whisper", reason="the reference package (stable-ts) is not installed in oracle/_ref/")
        yield env
    finally:
        if root is not None:
            sys.path.remove(root)
            for name in [m for m in sys.modules if m == "stable_whisper" or m.startswith("stable_whisper.")]:
                del sys.modules[name]


def _same_result(a, b, prob_tol=1e-5):
    da, db = a.to_dict(), b.to_dict()
    assert da["language"] == db["language"]
    assert len(da["segments"]) == len(db["segments"]) and len(da["segments"]) > 0
    for sa, sb in zip(da["segments"], db["segments"]):
        assert sa["text"] == sb["text"] and sa["start"] == sb["start"] and sa["end"] == sb["end"]
        assert len(sa.get("words") or []) == len(sb.get("words") or [])
        for wa, wb in zip(sa.get("words") or [], sb.get("words") or []):
            assert wa["word"] == wb["word"] and wa["tokens"] == wb["tokens"]
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"], (wa, wb)
            assert abs(wa["probability"] - wb["probability"]) <= prob_tol * max(abs(wb["probability"]), 1e-30)


def test_align_through_unmodified_aligner_is_identical(ref_env):
    env = ref_env
    import stable_whisper.alignment as ref_align
    from stable_ts_b200 import api
    theirs = ref_align.align(env["model"], env["audio"], env["text"], language="en", verbose=None, ignore_compatibility=True)
    stand = api.modify_model(env["stand"])
    mine = stand.align(env["audio"], env["text"], language="en", verbose=None)
    assert type(mine).__name__ == "WhisperResult" and type(mine).__module__.startswith("stable_whisper")
    _same_result(mine, theirs)
    assert env["stand"].calls["decode_forced"] >= 1


def test_align_words_and_refine_through_unmodified_control_plane(ref_env):
    env = ref_env
    import stable_whisper.alignment as ref_align
    from stable_ts_b200 import api
    base = ref_align.align(env["model"], env["audio"], env["text"], language="en", verbose=None, ignore_compatibility=True)
    stand = api.modify_model(env["stand"])
    segs = [dict(start=s.start, end=s.end, text=s.text) for s in base.segments]
    theirs = ref_align.align_words(env["model"], env["audio"], copy.deepcopy(segs), language="en", verbose=None,
                                   ignore_compatibility=True)
    mine = stand.align_words(env["audio"], copy.deepcopy(segs), language="en", verbose=None)
    _same_result(mine, theirs)
    # refine: the Refiner's decisions depend on probabilities AND on the token rank derived from the 3-D form
    r_theirs = ref_align.refine(env["model"], env["audio"], copy.deepcopy(base), verbose=None, precision=0.2)
    r_mine = stand.refine(env["audio"], copy.deepcopy(base), verbose=None, precision=0.2)
    _same_result(r_mine, r_theirs)
    moved = sum(wa.start != wb.start or wa.end != wb.end for wa, wb in zip(r_mine.all_words(), base.all_words()))
    print(f"refine moved {moved} word boundaries; identical to the reference's vanilla closure")


def test_refine_closure_3d_form_reaches_rank_test(ref_env):
    """The closure returns the 3-D tensor, so ``Refiner.get_prob`` computes real token positions (refinement.py:305-325)."""
    env = ref_env
    from stable_whisper.non_whisper.refinement import Refiner
    from stable_ts_b200.alignment import get_b200_refinement_func
    from stable_ts_b200.tokenizer import get_tokenizer
    tk = get_tokenizer(env["stand"], language="en", task="transcribe", synthetic=True)
    f = get_b200_refinement_func(env["stand"], tk)
    script = env["SP"].synth_token_script(12, tk.eot, seed=3)
    a2 = torch.stack([env["audio"][:160000], env["audio"][160000:320000]])
    out = f(a2, script)
    assert out.ndim == 3 and out.shape == (2, len(script), tk.eot)
    r = Refiner(inference_func=f)
    probs, pos = r.get_prob(a2, script, [[t] for t in script], [i % 2 for i in range(len(script))], False)
    ref3 = env["SP"].refine_token_probs(env["model"], env["tk"], a2, script)
    _, rank = env["SP"].prob_and_rank(ref3, script)
    assert pos == [int(rank[i % 2, i]) for i in range(len(script))] and any(p > 0 for p in pos)


def test_own_result_schema_loads_in_the_reference(ref_env):
    """result.py stand-in <-> stable_whisper.WhisperResult: same dict schema both ways (result.py:618-636, :1398-1406).  `d` is
    what the reference's align() returned, as its to_dict(keep_orig=False) wrote it."""
    import stable_whisper
    from stable_ts_b200.result import WhisperResult as Mine
    d = ref_env["gold"]["align_result"]         # with ori_dict kept, BOTH classes read `language` from it (result.py:938-939)
    theirs = stable_whisper.WhisperResult(copy.deepcopy(d))
    mine = Mine(copy.deepcopy(d))
    again = stable_whisper.WhisperResult(mine.to_dict(keep_orig=False))
    _same_result(again, theirs, prob_tol=0)
    assert mine.text == theirs.text and len(mine.all_words()) == len(theirs.all_words())
    md = mine.to_dict(keep_orig=False)
    assert set(md) == set(d)
    for sa, sb in zip(md["segments"], d["segments"]):
        assert set(sb) <= set(sa)
        for wa, wb in zip(sa.get("words") or [], sb.get("words") or []):
            assert wa == wb


@pytest.mark.parametrize("mode,thr", [(2, 0.5), (0, 0.0), (1, 0.0), (0, 0.5)])
def test_locate_matches_unmodified_reference(env, mode, thr):
    """stable_ts_b200.locate (host loop + kernel calls) over the stand-in == stable_whisper.alignment.locate over the oracle
    model (alignment.py:756-1116): target times (mode 2), confirmed segments with word timings (mode 0), window words (mode 1)."""
    from stable_ts_b200 import api
    stand = api.modify_model(env["stand"])
    text = [700, 901, 333]
    kw = dict(count=3, mode=mode, probability_threshold=thr, exact_token=True, max_token_per_seg=8)
    theirs = env["gold"]["locate"][f"{mode}|{thr}"]
    mine = stand.locate(env["audio"], text, "en", **kw)
    assert len(mine) == len(theirs)
    if mode != 0 or thr == 0.0:
        assert len(mine) > 0
    for a, b in zip(mine, theirs):
        if mode == 2:
            assert json.loads(json.dumps(a)) == b
        elif mode == 1:
            assert a["end"] == b["end"] and a["duration_window_text"] == b["duration_window_text"]
            assert [w["tokens"] for w in a["duration_window_word"]] == [w["tokens"] for w in b["duration_window_word"]]
            np.testing.assert_allclose([w["probability"] for w in a["duration_window_word"]],
                                       [w["probability"] for w in b["duration_window_word"]], rtol=1e-5)
        else:
            da, db = a.to_dict(), b
            assert da["seek"] == db["seek"] and da["start"] == db["start"] and da["end"] == db["end"]
            assert [(w["word"], w["tokens"], w["start"], w["end"]) for w in da["words"]] == \
                   [(w["word"], w["tokens"], w["start"], w["end"]) for w in db["words"]]
