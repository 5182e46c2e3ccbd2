"""CPU tests of the audio-ingest oracle (oracle/audio_io.py) and of the host half of stable_ts_b200.audio_io (WAV parsing,
filter table).  The polyphase arithmetic is cross-checked against scipy.signal.upfirdn, an independent implementation."""
import numpy as np
import pytest

from oracle import audio_io as OA


def _signal(n, rate, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / rate
    x = sum(np.sin(2 * np.pi * f * t + p) for f, p in zip(rng.uniform(80, 7000, 5), rng.uniform(0, 6.28, 5))) / 6
    return x + 0.01 * rng.standard_normal(n)


@pytest.mark.parametrize("rate,channels", [(44100, 2), (48000, 1), (8000, 1), (22050, 2), (16000, 2)])
def test_polyphase_matches_scipy_upfirdn(rate, channels):
    import math
    from scipy.signal import upfirdn
    n = 5000
    x = np.stack([_signal(n, rate, 10 + c) for c in range(channels)], axis=1)
    pcm = np.round(x * 20000).astype(np.int16).reshape(-1)
    y = OA.resample_to_mono(pcm, channels, rate)
    g = math.gcd(rate, 16000)
    L, M = 16000 // g, rate // g
    tab = OA.polyphase_table(L, M).astype(np.float32).astype(np.float64)
    taps = tab.shape[1]
    half = taps // 2
    proto = np.zeros(L * (taps + 1))                       # prototype at the up-sampled rate: index p - (j - half) L + half L
    for p in range(L):
        for j in range(taps):
            proto[p - (j - half) * L + half * L] = tab[p][j]
    mono = (pcm.astype(np.float64) / 32768).reshape(-1, channels).astype(np.float32).astype(np.float64).sum(1) / channels
    full = upfirdn(proto, mono, up=L, down=1)              # sample k of the up-sampled grid sits at index k + half L
    want = full[half * L + np.arange(len(y)) * M]
    np.testing.assert_allclose(y, want.astype(np.float32), atol=2e-7, rtol=0)
    assert len(y) == -(-n * L // M)


def test_dc_gain_and_band_limits():
    # unit DC gain on every branch; a 3 kHz tone survives 44.1k -> 16k, a 12 kHz tone (above the new Nyquist) is removed
    tab = OA.polyphase_table(160, 441)
    np.testing.assert_allclose(tab.sum(axis=1), 1.0, atol=1e-12)
    rate, n = 44100, 44100
    t = np.arange(n) / rate
    keep = OA.resample_to_mono(np.sin(2 * np.pi * 3000 * t).astype(np.float32), 1, rate)
    kill = OA.resample_to_mono(np.sin(2 * np.pi * 12000 * t).astype(np.float32), 1, rate)
    mid = slice(2000, -2000)
    assert abs(np.sqrt(np.mean(keep[mid] ** 2)) - np.sqrt(0.5)) < 1e-3
    assert np.sqrt(np.mean(kill[mid] ** 2)) < 1e-4


def test_product_host_half_matches_oracle():
    from stable_ts_b200 import audio_io as A
    assert (A.ZEROS, A.ROLLOFF, A.BETA) == (OA.ZEROS, OA.ROLLOFF, OA.BETA)
    for rate in (44100, 48000, 8000, 11025):
        L, M = A.resample_ratio(rate)
        assert np.array_equal(A.polyphase_table(L, M), OA.polyphase_table(L, M).astype(np.float32))
    x = np.round(_signal(999, 44100, 3) * 9000).astype(np.int16)
    rate, ch, fmt, payload = A.parse_wav(OA.make_wav(np.repeat(x, 2), 44100, 2))
    assert (rate, ch, fmt) == (44100, 2, 0) and np.array_equal(np.frombuffer(payload, np.int16), np.repeat(x, 2))
    f = _signal(500, 8000, 4).astype(np.float32)
    rate, ch, fmt, payload = A.parse_wav(OA.make_wav(f, 8000, 1))
    assert (rate, ch, fmt) == (8000, 1, 2) and np.array_equal(np.frombuffer(payload, np.float32), f)
    with pytest.raises(ValueError):
        A.parse_wav(b"OggS" + b"\0" * 64)


def test_reference_demo_wav_header_if_present():
    """examples/demo.wav of the reference (44.1 kHz stereo s16; BASELINE config 1) parses: its first 0.1 s, header chunks
    kept as they are (tests/golden/demo_head.wav, oracle/make_golden_reference.py)."""
    import os
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo_head.wav")
    from stable_ts_b200 import audio_io as A
    rate, ch, fmt, payload = A.parse_wav(open(p, "rb").read())
    assert (rate, ch, fmt) == (44100, 2, 0)
    y = OA.resample_to_mono(np.frombuffer(payload, np.int16), ch, rate, quantize_s16=True)
    assert abs(len(y) / 16000 - len(payload) / 4 / 44100) < 1e-3 and np.abs(y).max() <= 1.0
