"""Pins the silence-detection oracle (oracle/silence.py, SURVEY.md section 8f row 1): against PyTorch's own operators,
against fixtures written by the unmodified reference (tests/golden/silence_cases.npz, oracle/make_golden_silence.py;
tests/golden/reference_silence.npz, oracle/make_golden_reference.py)."""
import os

import numpy as np
import pytest
import torch
from torch.nn import functional as F

from oracle import silence as SIL
from oracle import stable_path as SP
from oracle.make_golden_silence import CASES, case_audio

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "silence_cases.npz")
GOLD_FUNCS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_silence.npz")


@pytest.mark.parametrize("n", [480000, 479999, 250001, 160000, 100000, 3000, 1234, 999])
def test_interpolate_linear_equals_torch(n):
    x = (torch.randn(n, generator=torch.Generator().manual_seed(n)) * 0.1).abs()
    size = round(n / 320) + 1
    ref = F.interpolate(x[None, None], size=size, mode="linear", align_corners=False)[0, 0].numpy()
    assert np.array_equal(SIL.interpolate_linear(x.numpy(), size), ref)


@pytest.mark.parametrize("n,k", [(1501, 5), (782, 5), (10, 5), (313, 3), (64, 7)])
def test_avg_pool_reflect_equals_torch(n, k):
    x = torch.rand(n, generator=torch.Generator().manual_seed(n + k))
    p = k // 2
    ref = torch.avg_pool1d(F.pad(x[None], (p, p), "reflect"), kernel_size=k, stride=1)[0].numpy()
    assert np.array_equal(SIL.avg_pool_reflect(x.numpy(), k), ref)


def test_kth_largest_equals_topk():
    x = SP.synth_gapped_audio(480000, seed=5)
    k = int(x.numel() * 0.001)
    assert SIL.kth_largest_abs(x.numpy(), k) == torch.topk(x.abs(), k)[0][-1].item()


def test_fixtures_written_by_the_reference():
    z = np.load(GOLD)
    assert np.array_equal(z["cases"], np.array(CASES, dtype=np.float64))
    for i, (n, seed, floor, scale) in enumerate(CASES):
        audio = case_audio(int(n), int(seed), floor, scale).numpy()
        loud = SIL.audio2loudness(audio)
        assert np.array_equal(loud, z[f"loud_{i}"]), f"case {i}: loudness differs"
        mask = SIL.wav2mask(audio)
        assert (mask is not None) == bool(z[f"has_mask_{i}"])
        if mask is not None:
            assert np.array_equal(mask, z[f"mask_{i}"]), f"case {i}: mask differs"
        pred = SIL.predict_with_nonvad(audio, offset=12.5)
        assert (pred["timings"] is not None) == bool(z[f"has_timings_{i}"])
        if pred["timings"] is not None:
            assert np.array_equal(pred["timings"], z[f"timings_{i}"]), f"case {i}: timings differ"
        assert pred["is_silent"] == bool(z[f"silent_{i}"])
        if pred["mask"] is not None:
            assert pred["mask"].shape == (1501,) and np.array_equal(pred["mask"], z[f"pmask_{i}"])
        else:
            assert z[f"pmask_{i}"].size == 0


@pytest.mark.parametrize("n,seed,floor,scale", [(480000, 101, 0.0, 1.0), (333333, 102, 5e-4, 1.0), (480000, 103, 2e-3, 0.5),
                                                (64000, 104, 0.0, 1.0), (480000, 105, 0.0, 1e-7)])
def test_live_reference_functions(n, seed, floor, scale):
    """audio2loudness / wav2mask / mask2timing / timing2mask of stable_whisper.stabilization, as the reference returned them."""
    z = np.load(GOLD_FUNCS)
    i = [tuple(c) for c in z["cases"]].index((n, seed, floor, scale))
    audio = SP.synth_gapped_audio(n, seed=seed, floor=floor) * scale
    assert np.array_equal(SIL.audio2loudness(audio.numpy()), z[f"loud_{i}"])
    got = SIL.wav2mask(audio.numpy())
    assert (got is not None) == bool(z[f"has_mask_{i}"])
    if got is not None:
        assert np.array_equal(got, z[f"mask_{i}"])
        for j, off in enumerate((None, 3.25)):
            a = SIL.mask2timing(got, time_offset=off)
            assert (a is not None) == bool(z[f"has_timing_{i}_{j}"])
            if a is not None:
                assert np.array_equal(a[0], z[f"starts_{i}_{j}"]) and np.array_equal(a[1], z[f"ends_{i}_{j}"])
                assert np.array_equal(SIL.timing2mask(a[0], a[1], 1501, time_offset=off), z[f"remask_{i}_{j}"])
