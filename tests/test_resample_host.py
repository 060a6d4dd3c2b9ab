"""CPU: the resampler in front of the voice-cloning encoder. The float64 band restatement (tests/resample_ref.py) that the device
resampler is tested against, checked against torchaudio.functional.resample; the 24- and 32-bit WAV reader; the new symbols."""
import math
import struct

import numpy as np
import pytest
import torch

import resample_ref as R

RATES = [8000, 11025, 16000, 22050, 32000, 44100, 48000, 88200, 96000, 192000]
BANDS = {8000: 13, 11025: 13, 16000: 13, 22050: 13, 32000: 17, 44100: 23, 48000: 25, 88200: 45, 96000: 49, 192000: 97}


def lengths(sr):
    o = R.plan(sr)["o"]
    return sorted({n for n in (1, o - 1, o, o + 1, int(1.3 * sr)) if n >= 1})


@pytest.mark.parametrize("sr", RATES)
def test_restatement_matches_torchaudio(sr):
    import torchaudio.functional as AF
    for n in lengths(sr):
        x = np.random.default_rng(n).standard_normal(n)
        want = AF.resample(torch.as_tensor(x)[None], sr, R.SR)[0].numpy()
        got = R.resample(x, sr)
        assert len(got) == len(want) == R.out_len(n, sr), (n, len(got), len(want))
        assert np.abs(got - want).max() <= 1e-12, (n, np.abs(got - want).max())


@pytest.mark.parametrize("sr", RATES + [99000])
def test_band_table_is_the_rounded_dense_kernel(sr):
    """Every f32 tap of torchaudio's float64 kernel outside the band is exactly zero, and the band holds the others. 99 kHz puts a tap
    exactly at |t| = L."""
    from torchaudio.functional.functional import _get_sinc_resample_kernel
    p = R.plan(sr)
    dense, width = _get_sinc_resample_kernel(sr, R.SR, math.gcd(sr, R.SR), dtype=torch.float64)
    assert width == p["w"]
    dense = dense[:, 0, :].numpy().astype(np.float32)
    band = R.dense_from_band(p, R.band_table(p).astype(np.float32))
    assert np.array_equal(band, dense)
    if sr in BANDS:
        assert p["W"] == BANDS[sr]


@pytest.mark.parametrize("sr", RATES + [44101, 24001, 8001])
def test_output_length(sr):
    """n24 = ceil(24000 n / sr), the restatement alone for a rate whose dense kernel would not fit in memory (44101 Hz: m = 24000)."""
    p = R.plan(sr)
    for n in (1, 2, p["o"] - 1, p["o"], p["o"] + 1, 3 * sr + 7):
        if n < 1:
            continue
        want = -(-n * 24000 // sr)
        assert R.out_len(n, sr) == want == len(R.resample(np.ones(n), sr))
    if sr == 44101:
        assert p["m"] == 24000 and p["W"] == 23
        y = R.resample(np.ones(sr), sr)                       # DC passes at the filter's gain
        assert len(y) == 24000 and abs(y[12000] - 1.0) < 1e-2


def write_pcm_int(path, x, bits, channels=1, rate=48000, extensible=False):
    """Integer PCM of `bits` (24 or 32) in a RIFF file; x int array [n * channels] in range."""
    nb = bits // 8
    data = np.asarray(x, "<i4").reshape(-1, 1).view(np.uint8)[:, :nb].tobytes()     # little-endian: the low nb bytes
    if extensible:
        guid = struct.pack("<H", 1) + bytes.fromhex("000000001000800000aa00389b71")
        fmt = struct.pack("<HHIIHHHHI", 0xFFFE, channels, rate, rate * channels * nb, channels * nb, bits, 22, bits, 0) + guid
    else:
        fmt = struct.pack("<HHIIHH", 1, channels, rate, rate * channels * nb, channels * nb, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    if len(data) % 2:
        body += b"\0"
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


@pytest.mark.parametrize("bits", [24, 32])
@pytest.mark.parametrize("channels", [1, 2])
@pytest.mark.parametrize("extensible", [False, True])
def test_wav_int_pcm(P, tmp_path, bits, channels, extensible):
    lim = 1 << (bits - 1)
    rng = np.random.default_rng(bits + channels)
    x = rng.integers(-lim, lim, (1001, channels), dtype=np.int64)
    x[0] = -lim; x[1] = lim - 1                               # full scale both ways
    path = str(tmp_path / "i.wav")
    write_pcm_int(path, x, bits, channels=channels, rate=44100, extensible=extensible)
    y, rate = P.read_wav(path)
    assert rate == 44100 and y.dtype == np.float32 and len(y) == 1001
    want = (x.astype(np.float64) / lim).mean(1).astype(np.float32)    # the reader averages in float64, rounds once
    assert np.array_equal(y, want)


def test_symbols_exported(P):
    L = P.lib()
    for s in ("b200_voice_embed_audio_rate", "b200_voice_create_from_audio_rate"):
        assert hasattr(L, s), s
