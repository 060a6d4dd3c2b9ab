"""GPU: voice cloning from recordings at any sample rate. The device resampler against the float64 restatement (tests/resample_ref.py),
the encoder taps on the resampled signal, 24 kHz through the new entry points, determinism, the device prefill, cloning beside a running
online batch, capacity and error cases, and the context / CLI round trips with a 44.1 kHz 24-bit WAV."""
import os
import re
import subprocess
import wave

import numpy as np
import pytest

import resample_ref as R
from encoder_ref import EncoderRef
from make_assets import default_model_dir, read_safetensors
from test_resample_host import write_pcm_int

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(REPO, "pocket-tts.cpp_b200", "lib", "pocket-tts-b200")
RATES = [8000, 11025, 16000, 22050, 32000, 44100, 48000, 88200, 96000, 192000]
# max-abs of enc.input against the restatement (f32-rounded coefficients, float64 sums), inputs |x| <= ~4.1: about 4x the worst value
# measured on a B200 (DESIGN.md §2)
INPUT_BOUND = 7e-6
# the bounds tests/test_gpu_voice_clone.py uses for prompts longer than two rows
BOUNDS_LONG = {"enc.seanet": 2e-3, "enc.transformer": 4e-3, "enc.downsample": 4e-3, "prompt": 8e-3}
EINVAL, ENOTFOUND, ECAPACITY = -1, -4, -5


@pytest.fixture(scope="module")
def model_dir_enc():
    return default_model_dir(eos_mode="never", encoder=True)


@pytest.fixture(scope="module")
def ctx(P, model_dir_enc):
    c = P.Context(model_dir_enc, max_slots=2, max_voices=8, kv_capacity=1024)
    yield c
    c.close()


@pytest.fixture(scope="module")
def generated_pcm(P, model_dir):
    """24 kHz PCM the engine itself generated from a stock voice (temperature 0)."""
    c = P.Context(model_dir, max_slots=1, max_voices=1, kv_capacity=1024)
    s = c.stream("cosette", temp=0.0)
    s.send("The quick brown fox jumped over the sleeping dog. Water runs down the mountain toward the sea.")
    s.flush()
    frames = []
    while (f := s.receive()) is not None:
        frames.append(f)
    c.close()
    return np.concatenate(frames)


def make_input(kind, n, sr, generated=None):
    rng = np.random.default_rng(n + sr)
    if kind == "noise":
        return (0.3 * rng.standard_normal(n)).astype(np.float32)
    if kind == "tone":                                  # just below the filter's cutoff, 0.99 min(sr, 24000) / 2
        f = 0.96 * min(sr, R.SR) / 2
        return (0.8 * np.sin(2 * np.pi * f * np.arange(n) / sr)).astype(np.float32)
    import torch
    import torchaudio.functional as AF                 # the engine's own 24 kHz speech taken to sr
    g = AF.resample(torch.as_tensor(generated)[None], R.SR, sr)[0].numpy()
    return np.resize(g, n).astype(np.float32)


def rel_l2(x, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.linalg.norm(np.asarray(x, np.float64) - ref) / max(np.linalg.norm(ref), 1e-30))


def input_cases():
    out = []
    for sr in RATES:
        o = R.plan(sr)["o"]
        n1920 = 1920 * sr // R.SR                       # the longest input with n24 = 1920
        ns = sorted({n for n in (1, o - 1, o, n1920 - 1, n1920, n1920 + 1, int(1.3 * sr), 10 * sr, 30 * sr) if n >= 1})
        out += [(sr, "noise", n) for n in ns] + [(sr, k, n) for k in ("tone", "generated") for n in (int(1.3 * sr), 10 * sr)]
    return out


@pytest.mark.parametrize("sr,kind,n", input_cases())
def test_resampled_input_matches_restatement(ctx, generated_pcm, sr, kind, n):
    x = make_input(kind, n, sr, generated_pcm)
    eng = ctx.engine
    out = eng.embed_audio(x, sample_rate=sr)
    want = R.encoder_input(x, sr)
    assert out.shape == (len(want) // 1920, 1024)
    got = eng.debug_tap("enc.input", 0)
    assert got.shape == want.shape
    n24 = R.out_len(n, sr)
    assert not got[n24:].any()                           # the encoder's zero right padding
    err = float(np.abs(got.astype(np.float64) - want).max())
    print(f"RESAMPLE sr={sr} {kind} n={n} max_abs={err:.3e} max|x|={np.abs(x).max():.2f}")
    assert err <= INPUT_BOUND, err


@pytest.fixture(scope="module")
def ref(model_dir_enc):
    import torch
    return EncoderRef(read_safetensors(model_dir_enc + "tts_b6369a24.safetensors"), device="cuda" if torch.cuda.is_available() else "cpu")


@pytest.mark.parametrize("sr", [16000, 44100, 48000])
@pytest.mark.parametrize("seconds", [1.3, 10])
def test_encoder_taps_on_resampled_signal(ctx, ref, generated_pcm, sr, seconds):
    x = make_input("generated", int(seconds * sr), sr, generated_pcm)
    eng = ctx.engine
    out = eng.embed_audio(x, sample_rate=sr)
    x24 = R.resample(x, sr, f32_table=True).astype(np.float32)
    want = {k: v.cpu().numpy() for k, v in ref.stages(x24).items()}
    errs = {tap: rel_l2(eng.debug_tap(tap, 0).reshape(want[tap].shape), want[tap]) for tap in ("enc.seanet", "enc.transformer", "enc.downsample")}
    errs["prompt"] = rel_l2(out, want["prompt"])
    print(f"TAPS sr={sr} {seconds}s " + " ".join(f"{k}={v:.3e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v <= BOUNDS_LONG[k], (k, v)


def test_24k_through_rate_entry_points_is_todays_path(P, ctx):
    L, eng = P.lib(), ctx.engine
    x = make_input("noise", 5 * R.SR + 17, R.SR)
    T = -(-len(x) // 1920)
    a, b = np.zeros((T, 1024), np.float32), np.zeros((T, 1024), np.float32)
    l0 = eng.launch_count()
    assert L.b200_voice_embed_audio(eng.h, P._fp(x), len(x), P._fp(a)) == T
    l1 = eng.launch_count()
    assert L.b200_voice_embed_audio_rate(eng.h, P._fp(x), len(x), R.SR, P._fp(b)) == T
    l2 = eng.launch_count()
    assert a.tobytes() == b.tobytes() and l1 - l0 == l2 - l1
    y = make_input("noise", 5 * 44100 + 17, 44100)
    eng.embed_audio(y, sample_rate=32000)                # another rate first, so that 44.1 kHz rebuilds its table
    l3 = eng.launch_count()
    eng.embed_audio(y, sample_rate=44100)
    l4 = eng.launch_count()
    eng.embed_audio(y, sample_rate=44100)
    l5 = eng.launch_count()
    assert l4 - l3 == (l1 - l0) + 2 and l5 - l4 == (l1 - l0) + 1      # table (only on a rate change) + resampler


def test_deterministic_44k(ctx):
    x = make_input("noise", 5 * 44100 + 17, 44100)
    a, b = ctx.engine.embed_audio(x, 44100), ctx.engine.embed_audio(x, 44100)
    assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("prefix_share", [1, 0])
def test_device_prefill_matches_host_round_trip_44k(P, model_dir_enc, prefix_share):
    c = P.Context(model_dir_enc, max_slots=1, max_voices=4, kv_capacity=512, prefix_share=prefix_share)
    eng = c.engine
    x = make_input("tone", 3 * 44100 + 5, 44100)
    v_dev = eng.voice_from_audio(x, sample_rate=44100)
    v_host = eng.voice_create(eng.embed_audio(x, sample_rate=44100))
    T = -(-R.out_len(len(x), 44100) // 1920)
    assert P.lib().b200_voice_len(eng.h, v_dev) == P.lib().b200_voice_len(eng.h, v_host) == T
    S = P.lib().b200_max_slots(eng.h)
    for layer in range(6):
        for which in (0, 1):
            assert eng.read_kv(S + v_dev, layer, which, T).tobytes() == eng.read_kv(S + v_host, layer, which, T).tobytes(), (layer, which)
    toks = c.tokenize("A small bird sings in the morning light.")
    pcm = {}
    for v in (v_dev, v_host):
        eng.begin_sentence(0, v, toks, 20, 3, 0.0)
        pcm[v] = np.stack([eng.step(0, 1)[0][0] for _ in range(20)])
    assert np.abs(pcm[v_dev]).max() > 0 and pcm[v_dev].tobytes() == pcm[v_host].tobytes()
    c.close()


def _write_wav16(path, x, rate):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(rate)
        w.writeframes((np.clip(x, -1, 1) * 32767).astype(np.int16).tobytes())


SERVE_TEXTS = ["Hello world. Read the letter again.", "Water runs down the mountain toward the sea.", "Numbers like forty two are words too."]


@pytest.mark.parametrize("overlap", [0, 1])
def test_48k_clone_while_serving(P, model_dir_enc, tmp_path, overlap):
    """A 48 kHz .wav voice added between pumps of an online batch leaves the utterances already running bitwise unchanged (the reference
    run adds the same utterance with a stock voice at the same point; private prefix copies)."""
    wav = tmp_path / "clone48.wav"
    _write_wav16(wav, make_input("tone", 2 * 48000, 48000), 48000)
    audio = {}
    for voice in ("cosette", str(wav)):
        c = P.Context(model_dir_enc, max_slots=8, max_voices=4, kv_capacity=1024, prefix_share=0, overlap=overlap)
        P.set_seed(5)
        b = P.Batch(c)
        utts = [b.add("cosette", t, temp=0.7) for t in SERVE_TEXTS]
        for _ in range(4):
            b.pump(3)
        late = b.add(voice, "The cloned voice speaks now.", temp=0.7)
        while b.pump(4) > 0:
            pass
        audio[voice] = [b.read(u) for u in utts] + [b.read(late)]
        del b
        c.close()
    base, cloned = audio["cosette"], audio[str(wav)]
    for i in range(len(SERVE_TEXTS)):
        assert len(base[i]) > 0 and base[i].tobytes() == cloned[i].tobytes(), i
    assert len(cloned[-1]) > 0


def test_capacity_and_errors(P, model_dir, model_dir_enc):
    L = P.lib()
    x = make_input("noise", 4000, 16000)
    c = P.Context(model_dir, max_slots=1, max_voices=2, kv_capacity=256)
    assert L.b200_voice_create_from_audio_rate(c.engine.h, P._fp(x), len(x), 16000) == ENOTFOUND
    assert L.b200_voice_embed_audio_rate(c.engine.h, P._fp(x), len(x), 16000, None) == ENOTFOUND
    c.close()
    c = P.Context(model_dir_enc, max_slots=1, max_voices=2, kv_capacity=64)
    h = c.engine.h
    for sr in (0, -44100, 7999, 192001):
        assert L.b200_voice_embed_audio_rate(h, P._fp(x), len(x), sr, None) == EINVAL, sr
        assert L.b200_voice_create_from_audio_rate(h, P._fp(x), len(x), sr) == EINVAL, sr
    with pytest.raises(RuntimeError):
        c.add_voice("low", x, sample_rate=7999)
    nmax = 64 * 1920 * 44100 // 24000                   # T = kv_capacity = 64 at 44.1 kHz
    big = make_input("noise", nmax + 1, 44100)
    assert L.b200_voice_embed_audio_rate(h, P._fp(big), nmax, 44100, None) == 64
    assert L.b200_voice_embed_audio_rate(h, P._fp(big), nmax + 1, 44100, None) == ECAPACITY
    assert L.b200_voice_create_from_audio_rate(h, P._fp(big), nmax + 1, 44100) == ECAPACITY
    assert c.engine.voice_from_audio(big[:nmax], sample_rate=44100) == 0
    assert L.b200_voice_len(h, 0) == 64
    c.close()


def test_context_add_and_export_44k(P, model_dir_enc, tmp_path):
    c = P.Context(model_dir_enc, max_slots=2, max_voices=4, kv_capacity=512)
    x = make_input("tone", 2 * 44100, 44100)
    v = c.add_voice("mine44", x, sample_rate=44100)
    path = str(tmp_path / "mine44.safetensors")
    c.export_voice("mine44", path)
    rows = read_safetensors(path)["audio_prompt"]
    T = -(-R.out_len(len(x), 44100) // 1920)
    assert rows.shape == (1, T, 1024)
    assert rows[0].tobytes() == c.engine.embed_audio(x, sample_rate=44100).tobytes()
    assert c.stream("mine44", temp=0.0).voice == v
    assert P.lib().b200_voice_len(c.engine.h, c.stream(path, temp=0.0).voice) == T
    c.close()


def test_cli_44k_24bit_round_trip(P, model_dir_enc, tmp_path):
    out24 = str(tmp_path / "a.wav")
    r = subprocess.run([CLI, "-m", model_dir_enc, "--bench", "-o", out24], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    x, rate = P.read_wav(out24)
    assert rate == 24000
    import torch
    import torchaudio.functional as AF
    y = AF.resample(torch.as_tensor(x, dtype=torch.float64)[None], 24000, 44100)[0].numpy()
    wav = str(tmp_path / "take_44k.wav")
    write_pcm_int(wav, np.round(np.clip(y, -1, 1 - 2 ** -23) * 2 ** 23).astype(np.int64), 24, rate=44100)
    assert P.read_wav(wav)[1] == 44100
    r = subprocess.run([CLI, "-m", model_dir_enc, "--voice", wav, "--bench"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert int(re.search(r"^frame count:\s+(\d+) frames$", r.stdout, re.M).group(1)) == 137
