"""CPU: the voice-cloning pieces that need no GPU. The engine's WAV reader, the encoder assets, and self-checks of the float64
restatement of the encoder (tests/encoder_ref.py) that the device encoder is tested against."""
import hashlib
import os
import struct
import wave

import numpy as np
import pytest
import torch

from encoder_ref import EncoderRef, strided_conv_reshape
from make_assets import default_model_dir, read_safetensors, synth_encoder_weights

NEW_SYMBOLS = ["b200_has_encoder", "b200_voice_embed_audio", "b200_voice_create_from_audio", "ptts_c_voice_add_audio", "ptts_c_voice_export",
               "ptts_c_wav_read"]


def write_pcm16(path, x, channels=1, rate=24000):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(channels)
        w.setsampwidth(2)
        w.setframerate(rate)
        w.writeframes(np.asarray(x, np.int16).tobytes())


def write_f32(path, x, channels=1, rate=24000):
    data = np.asarray(x, np.float32).tobytes()
    fmt = struct.pack("<HHIIHH", 3, channels, rate, rate * channels * 4, channels * 4, 32)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_symbols_exported(P):
    L = P.lib()
    for s in NEW_SYMBOLS:
        assert hasattr(L, s), s


@pytest.mark.parametrize("n", [1, 1919, 1920, 4801])
def test_wav_pcm16_mono(P, tmp_path, n):
    x = np.random.default_rng(n).integers(-32768, 32767, n).astype(np.int16)
    write_pcm16(tmp_path / "a.wav", x)
    y, rate = P.read_wav(str(tmp_path / "a.wav"))
    assert rate == 24000 and y.dtype == np.float32
    np.testing.assert_array_equal(y, x.astype(np.float32) / 32768.0)


def test_wav_pcm16_stereo_mixdown(P, tmp_path):
    x = np.random.default_rng(1).integers(-32768, 32767, (333, 2)).astype(np.int16)
    write_pcm16(tmp_path / "s.wav", x.reshape(-1), channels=2)
    y, _ = P.read_wav(str(tmp_path / "s.wav"))
    np.testing.assert_allclose(y, x.astype(np.float64).mean(1) / 32768.0, rtol=0, atol=1e-7)


@pytest.mark.parametrize("channels", [1, 3])
def test_wav_float32(P, tmp_path, channels):
    x = np.random.default_rng(2).standard_normal((777, channels)).astype(np.float32)
    write_f32(tmp_path / "f.wav", x.reshape(-1), channels=channels)
    y, rate = P.read_wav(str(tmp_path / "f.wav"))
    assert rate == 24000 and len(y) == 777
    np.testing.assert_allclose(y, x.astype(np.float64).mean(1), rtol=0, atol=1e-6)


def test_wav_reports_other_rates(P, tmp_path):
    write_pcm16(tmp_path / "r.wav", np.zeros(100, np.int16), rate=16000)
    assert P.read_wav(str(tmp_path / "r.wav"))[1] == 16000


def test_wav_rejects_bad_files(P, tmp_path):
    write_pcm16(tmp_path / "ok.wav", np.arange(1000, dtype=np.int16))
    raw = open(tmp_path / "ok.wav", "rb").read()
    open(tmp_path / "trunc.wav", "wb").write(raw[:-100])
    open(tmp_path / "junk.wav", "wb").write(b"JUNK" + raw[4:])
    open(tmp_path / "short.wav", "wb").write(raw[:10])
    with wave.open(str(tmp_path / "u8.wav"), "wb") as w:   # 8-bit PCM: not a supported sample format
        w.setnchannels(1); w.setsampwidth(1); w.setframerate(24000); w.writeframes(bytes(100))
    for name in ("trunc.wav", "junk.wav", "short.wav", "u8.wav", "missing.wav"):
        with pytest.raises(ValueError):
            P.read_wav(str(tmp_path / name))


def test_encoder_assets_leave_the_decoder_untouched():
    base = read_safetensors(default_model_dir(eos_mode="never") + "tts_b6369a24.safetensors")
    enc = read_safetensors(default_model_dir(eos_mode="never", encoder=True) + "tts_b6369a24.safetensors")
    extra = set(enc) - set(base)
    assert extra == set(synth_encoder_weights(1234)) and not set(base) - set(enc)
    for k in base:
        assert base[k].tobytes() == enc[k].tobytes(), k


def test_default_directory_bytes_unchanged(tmp_path):
    """The default assets are what they were before the encoder option existed (hashes of the previous generator's files)."""
    from make_assets import make_model_dir
    d = make_model_dir(str(tmp_path / "m"), voices=["alba"])
    digest = {f: hashlib.sha256(open(os.path.join(d, f), "rb").read()).hexdigest()[:16] for f in ("tts_b6369a24.safetensors", "embeddings/alba.safetensors", "STAMP.json")}
    assert digest == DEFAULT_DIGESTS


DEFAULT_DIGESTS = {"tts_b6369a24.safetensors": "1960f24ffdeb926a", "embeddings/alba.safetensors": "209ce10cee36e86d", "STAMP.json": "13f786ff2fc926c4"}


@pytest.mark.parametrize("r,C,co", [(4, 8, 6), (5, 3, 4), (16, 2, 5)])
def test_reshape_strided_conv_matches_conv1d(r, C, co):
    rng = np.random.default_rng(r)
    L = 7 * r
    x = rng.standard_normal((L, C)); w = rng.standard_normal((co, C, 2 * r)); b = rng.standard_normal(co)
    ref = torch.nn.functional.conv1d(torch.nn.functional.pad(torch.as_tensor(x.T)[None], (r, 0)), torch.as_tensor(w), torch.as_tensor(b), stride=r)[0].T.numpy()
    np.testing.assert_allclose(strided_conv_reshape(x, w, b, r), ref, rtol=1e-12, atol=1e-12)


@pytest.fixture(scope="module")
def ref():
    return EncoderRef(synth_encoder_weights(1234))


def test_restatement_shapes_and_causality(ref):
    x = np.random.default_rng(3).standard_normal(1920 * 24 + 5).astype(np.float32) * 0.3
    full = ref.stages(x)
    T = 25
    assert full["prompt"].shape == (T, 1024) and full["enc.seanet"].shape == (16 * T, 512) and full["enc.downsample"].shape == (T, 512)
    assert np.isfinite(full["prompt"].numpy()).all()
    for k in (1, 7, 20):
        part = ref.embed(x[:1920 * k])
        np.testing.assert_allclose(part, full["prompt"].numpy()[:k], rtol=0, atol=1e-9)
