"""``extra_models`` and the "new" aligner's ``char_split`` (stable_whisper/timing.py:177-189, 240-253, 380-390, 442-444): the host
logic of stable_ts_b200.timing over the oracle-backed stand-in vs what the UNMODIFIED ``add_word_timestamps_stable`` returned
over the same oracle models (tests/golden/reference_results.json, oracle/make_golden_reference.py).  The kernels behind the
stand-in's methods are pinned by the -m gpu tests."""
import copy
import json
import os

import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")


@pytest.fixture(scope="module")
def env():
    import oracle.whisper_ref as W
    from oracle import stable_path as SP
    from standin import OracleBackedModel
    from stable_ts_b200.tokenizer import get_tokenizer
    om, om2 = W.build_model("tiny", seed=5), W.build_model("tiny", seed=6)
    stand, stand2 = OracleBackedModel(om), OracleBackedModel(om2)
    otk = W.tokenizer.get_tokenizer(True, num_languages=om.num_languages, language="en", task="transcribe")
    tk = get_tokenizer(stand, language="en", task="transcribe", synthetic=True)
    audio = SP.synth_audio(400000, seed=51)
    script = SP.synth_token_script(36, otk.eot, seed=52)
    segs = [dict(seek=0.0, tokens=script[:20]), dict(seek=0.0, tokens=script[20:])]
    with open(GOLD) as f:
        gold = json.load(f)["timing_variants"]
    return dict(stand=stand, stand2=stand2, tk=tk, audio=audio, segs=segs, gold=gold)


def _run_both(env, key, **kw):
    from stable_ts_b200.timing import add_word_timestamps_stable
    theirs, mine = env["gold"][key], copy.deepcopy(env["segs"])
    if "extra_models" in kw:
        kw["extra_models"] = [env["stand2"]]
    add_word_timestamps_stable(segments=mine, model=env["stand"], tokenizer=env["tk"], audio=env["audio"], num_samples=400000, **kw)
    n = 0
    for a, b in zip(mine, theirs):
        assert a["start"] == b["start"] and a["end"] == b["end"]
        assert len(a["words"]) == len(b["words"]) and len(a["words"]) > 0
        for wa, wb in zip(a["words"], b["words"]):
            assert wa["word"] == wb["word"] and list(wa["tokens"]) == list(wb["tokens"])
            assert wa["start"] == wb["start"] and wa["end"] == wb["end"], (wa, wb)
            assert abs(wa["probability"] - wb["probability"]) <= 1e-5 * abs(wb["probability"])
            n += 1
    return n


def test_char_split_matches_reference(env):
    assert _run_both(env, "char_split", aligner={"char_split": True}) > 5
    assert _run_both(env, "char_split_topk10", aligner={"char_split": True, "topk": 10}) > 5


@pytest.mark.parametrize("dyn", [None, 4, "4,2"])
def test_extra_models_match_reference(env, dyn):
    assert _run_both(env, f"extra_models_{dyn}", extra_models=True, dynamic_heads=dyn) > 5
