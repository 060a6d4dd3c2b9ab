"""GPU: voice cloning. The device encoder against the float64 restatement (tests/encoder_ref.py) at every tap, determinism, the
device-side prefill against the host round trip, cloning beside a running online batch, the error paths and the CLI round trip."""
import os
import re
import subprocess
import wave

import numpy as np
import pytest

from encoder_ref import EncoderRef
from make_assets import default_model_dir, read_safetensors

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(REPO, "pocket-tts.cpp_b200", "lib", "pocket-tts-b200")
SR = 24000
# rel-L2 bounds per stage against the restatement (DESIGN.md §2: about 4x the worst value measured on a B200, at most 1e-2). Prompts of
# one or two rows (n <= 3840) weigh a few bf16 roundings more; from 1.3 s on the bounds are tighter.
BOUNDS_SHORT = {"enc.seanet": 2e-3, "enc.transformer": 1e-2, "enc.downsample": 1e-2, "prompt": 1e-2}
BOUNDS_LONG = {"enc.seanet": 2e-3, "enc.transformer": 4e-3, "enc.downsample": 4e-3, "prompt": 8e-3}
LENGTHS = [1, 1919, 1920, 1921, int(1.3 * SR), 10 * SR, 30 * SR]


@pytest.fixture(scope="module")
def model_dir_enc():
    return default_model_dir(eos_mode="never", encoder=True)


@pytest.fixture(scope="module")
def ctx(P, model_dir_enc):
    c = P.Context(model_dir_enc, max_slots=2, max_voices=8, kv_capacity=1024)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ref(model_dir_enc):
    import torch
    return EncoderRef(read_safetensors(model_dir_enc + "tts_b6369a24.safetensors"), device="cuda" if torch.cuda.is_available() else "cpu")


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


def make_input(kind, n, generated):
    rng = np.random.default_rng(n)
    if kind == "noise":
        return (0.3 * rng.standard_normal(n)).astype(np.float32)
    if kind == "tones":
        t = np.arange(n) / SR
        x = 0.5 * np.sin(2 * np.pi * 220 * t) + 0.25 * np.sin(2 * np.pi * 1375 * t)
        x[(t % 0.5) > 0.3] = 0.0                                # 200 ms of silence every 500 ms
        return x.astype(np.float32)
    return np.resize(generated, n).astype(np.float32)


def rel_l2(x, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.linalg.norm(np.asarray(x, np.float64) - ref) / max(np.linalg.norm(ref), 1e-30))


CASES = [("noise", n) for n in LENGTHS] + [("tones", n) for n in (1921, int(1.3 * SR), 10 * SR)] + [("generated", n) for n in (int(1.3 * SR), 10 * SR)]


@pytest.mark.parametrize("kind,n", CASES)
def test_parity_with_restatement(ctx, ref, generated_pcm, kind, n):
    x = make_input(kind, n, generated_pcm)
    eng = ctx.engine
    assert eng.has_encoder
    out = eng.embed_audio(x)
    T = -(-n // 1920)
    assert out.shape == (T, 1024)
    want = {k: v.cpu().numpy() for k, v in ref.stages(x).items()}
    errs = {}
    for tap in ("enc.seanet", "enc.transformer", "enc.downsample"):
        got = eng.debug_tap(tap, 0).reshape(want[tap].shape)
        errs[tap] = rel_l2(got, want[tap])
    errs["prompt"] = rel_l2(out, want["prompt"])
    print(f"PARITY {kind} n={n} " + " ".join(f"{k}={v:.3e}" for k, v in errs.items()))
    bounds = BOUNDS_SHORT if n <= 2 * 1920 else BOUNDS_LONG
    for k, v in errs.items():
        assert v <= bounds[k], (k, v)


def _retrieval_qkv(R, seed=0):
    """Inputs on which every key of the window matters: query i of each head is 3x one key, cycling over i (the diagonal), i - 249 (the
    oldest visible key), i - 250 (the first key outside the window) and i - 125, so its score beats the others by ~20 and a window that is
    one key too wide, too narrow or shifted moves the output by O(|v|) on a quarter of the rows."""
    from encoder_ref import bf16
    import torch
    rng = np.random.default_rng(seed)
    k = rng.standard_normal((R, 512)).astype(np.float32)
    v = rng.standard_normal((R, 512)).astype(np.float32)
    q = np.zeros((R, 512), np.float32)
    for h in range(8):
        for i in range(R):
            t = i - (0, 249, 250, 125)[(i + h) % 4]
            q[i, h * 64:(h + 1) * 64] = 3.0 * k[max(t, 0), h * 64:(h + 1) * 64]
    return [bf16(torch.as_tensor(x, dtype=torch.float64)).numpy().astype(np.float32) for x in (q, k, v)]


@pytest.mark.parametrize("R", [1, 249, 250, 251, 313, 6000])
def test_window_attention_kernel(P, ctx, ref, R):
    """attn_window_kernel alone against the float64 masked softmax with the same rounding points, on retrieval inputs."""
    import torch
    q, k, v = _retrieval_qkv(R)
    got = ctx.engine.debug_window_attention(q, k, v)
    t = lambda x: torch.as_tensor(x, dtype=torch.float64, device=ref.dev)
    want = {w: ref.attention(t(q), t(k), t(v), window=w).cpu().numpy() for w in (249, 250, 251)}
    err = rel_l2(got, want[250])
    maxerr = float(np.abs(got.astype(np.float64) - want[250]).max())
    print(f"WINDOW R={R} rel_l2={err:.3e} max_abs={maxerr:.3e}")
    assert err <= 6e-5 and maxerr <= 3e-2, (err, maxerr)            # ~4x the worst measured on a B200 (DESIGN.md §2)
    if R > 250:                                   # a window of 249 or 251 keys moves some row by far more than the bound
        for w in (249, 251):
            assert np.abs(want[w] - want[250]).max() > 10 * 3e-2, w


def test_deterministic(ctx):
    x = make_input("noise", 5 * SR + 17, None)
    a, b = ctx.engine.embed_audio(x), ctx.engine.embed_audio(x)
    assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("prefix_share,kv_f32", [(1, 0), (0, 0), (1, 1)])
def test_device_prefill_matches_host_round_trip(P, model_dir_enc, prefix_share, kv_f32):
    c = P.Context(model_dir_enc, max_slots=1, max_voices=4, kv_capacity=512, prefix_share=prefix_share, kv_f32=kv_f32)
    eng = c.engine
    x = make_input("tones", 3 * SR + 5, None)
    v_dev = eng.voice_from_audio(x)
    v_host = eng.voice_create(eng.embed_audio(x))
    T = 38
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


def _write_wav(path, x):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(SR)
        w.writeframes((np.clip(x, -1, 1) * 32767).astype(np.int16).tobytes())


SERVE_TEXTS = ["Hello world. Read the letter again.", "Water runs down the mountain toward the sea.", "Numbers like forty two are words too."]


@pytest.mark.parametrize("overlap", [0, 1])
def test_clone_while_serving(P, model_dir_enc, tmp_path, overlap):
    """A .wav voice added between pumps of an online batch leaves the utterances already running bitwise unchanged. The reference run adds
    the same utterance with a stock voice at the same point, so that both runs step the same rows (private prefix copies: the attention
    plan of a row does not depend on which voices the other rows use)."""
    wav = tmp_path / "clone.wav"
    _write_wav(wav, make_input("tones", 2 * SR, None))
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


def test_errors(P, model_dir, model_dir_enc):
    L = P.lib()
    c = P.Context(model_dir, max_slots=1, max_voices=2, kv_capacity=256)
    x = make_input("noise", 4000, None)
    assert not c.engine.has_encoder
    assert L.b200_voice_create_from_audio(c.engine.h, P._fp(x), len(x)) == -4           # B200_ENOTFOUND
    assert L.b200_voice_embed_audio(c.engine.h, P._fp(x), len(x), None) == -4
    s = c.stream("cosette", temp=0.0)
    s.send("Hello world."); s.flush()
    assert s.receive() is not None                                                      # still generates
    c.close()
    c = P.Context(model_dir_enc, max_slots=1, max_voices=2, kv_capacity=64)
    h = c.engine.h
    assert L.b200_voice_create_from_audio(h, P._fp(x), 0) == -1                          # n = 0
    assert L.b200_voice_create_from_audio(h, None, 100) == -1
    big = make_input("noise", 64 * 1920 + 1, None)                                      # T = 65 > kv_capacity
    assert L.b200_voice_create_from_audio(h, P._fp(big), len(big)) == -5
    assert L.b200_voice_embed_audio(h, P._fp(big), len(big), None) == -5
    assert c.engine.voice_from_audio(x) == 0 and c.engine.voice_from_audio(x) == 1
    assert L.b200_voice_create_from_audio(h, P._fp(x), len(x)) == -5                     # max_voices reached
    with pytest.raises(RuntimeError):
        c.add_voice("x", x, sample_rate=16000)
    c.close()


def test_context_add_and_export(P, model_dir_enc, tmp_path):
    c = P.Context(model_dir_enc, max_slots=2, max_voices=4, kv_capacity=512)
    x = make_input("generated", 2 * SR, np.sin(np.arange(5000) / 7.0).astype(np.float32))
    v = c.add_voice("mine", x)
    path = str(tmp_path / "mine.safetensors")
    c.export_voice("mine", path)
    rows = read_safetensors(path)["audio_prompt"]
    assert rows.shape == (1, 25, 1024)
    assert rows[0].tobytes() == c.engine.embed_audio(x).tobytes()
    with pytest.raises(RuntimeError):                  # a stock voice name stays the stock voice
        c.add_voice("alba", x)
    s = c.stream("mine", temp=0.0)                     # the name works wherever a voice name does
    assert s.voice == v
    s2 = c.stream(path, temp=0.0)                      # and the exported file is an ordinary voice file
    assert P.lib().b200_voice_len(c.engine.h, s2.voice) == 25
    c.close()


def test_cli_round_trip(P, model_dir_enc, tmp_path):
    wav = str(tmp_path / "a.wav")
    r = subprocess.run([CLI, "-m", model_dir_enc, "--bench", "-o", wav], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([CLI, "-m", model_dir_enc, "--voice", wav, "--bench"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert int(re.search(r"^frame count:\s+(\d+) frames$", r.stdout, re.M).group(1)) == 137
