"""GPU parity at the configuration the headline number is quoted on (BASELINE.json configs[3]) and the cases VERDICT r1 listed
as unproven: batch 256, kv_capacity 2048, 1345-row voice prefix (several prefill chunks, one sentence cut by the first chunk boundary), KV length
~1.4-1.5k, default engine options — in BOTH prefix modes (shared voice prefix = cascade attention, and the reference's private copy);
an F32 checkpoint; two voices in one batch; the second sentence of a stream; the KV-capacity edge; tap-point localisation.

Everything goes through the C ABI. The oracle follows reference src/pocket_tts.cpp:416-492 (see oracle/ptts_oracle.cpp).
Tolerances are the ones stated in tests/test_gpu_parity.py (latent max-abs 4e-2 / rel-L2 1.5e-2, waveform SNR >= 40 dB).
"""
import os

import numpy as np
import pytest

from conftest import BENCH_SENTENCE, REPO, snr_db

pytestmark = pytest.mark.gpu
LAT_MAXABS, LAT_REL, SNR_MIN = 4e-2, 1.5e-2, 40.0
B, KV_CAP, T_VOICE = 256, 2048, 1345          # bench.py defaults: t_voice = kv_len 1500 - 45 - 100 warm-up steps - steps/2


@pytest.fixture(scope="module")
def bench_dir():
    from make_assets import default_model_dir
    return default_model_dir(eos_mode="never", t_voice=T_VOICE, voices=["cosette"])


@pytest.fixture(scope="module")
def bench_oracle(oracle_mod, bench_dir):
    o = oracle_mod.Oracle(bench_dir, threads=os.cpu_count() or 1)
    base = o.stream("cosette", kv_capacity=KV_CAP)        # ONE 1345-row voice prefill on the CPU; per-slot streams are clones
    return o, base


def _check_frame(tag, lat, pcm, glat, gpcm):
    err = float(np.abs(glat - lat).max()); rel = float(np.linalg.norm(glat - lat) / np.linalg.norm(lat)); snr = snr_db(pcm, gpcm)
    assert err < LAT_MAXABS and rel < LAT_REL and snr > SNR_MIN, (tag, err, rel, snr)
    return err, rel, snr


@pytest.mark.parametrize("share", [1, 0], ids=["shared_prefix", "private_prefix"])
def test_bench_configuration_matches_oracle(share, P, bench_dir, bench_oracle, oracle_mod):
    import bench
    orc, base = bench_oracle
    ctx = P.Context(bench_dir, max_slots=B, max_voices=1, kv_capacity=KV_CAP, prefix_share=share)
    eng = ctx.engine
    st = ctx.stream("cosette", temp=0.7)
    texts = [bench.synth_paragraph(i) for i in range(B)]
    toks = [ctx.tokenize(t) for t in texts]
    cum = np.concatenate([[0], np.cumsum([len(t) for t in toks])])
    chunk = P.default_config().max_prefill_rows                           # the engine's prefill chunk size
    straddle = int(np.searchsorted(cum, chunk, side="right") - 1)         # its token rows are cut by the end of the first prefill chunk
    assert cum[straddle] < chunk < cum[straddle + 1], (chunk, straddle, cum[straddle], cum[straddle + 1])
    mg = [oracle_mod.max_gen_len_for(t) for t in texts]
    eng.begin_sentences(list(range(B)), [st.voice] * B, toks, mg, [1 << 20] * B, [0.7] * B)
    check = [0, straddle, B - 1]
    streams = {}
    for k in check:
        s = base.clone()
        assert s.sentence_init(texts[k]) == toks[k]                       # token ids bit-exact
        assert eng.slot_position(k) == s.current_end == T_VOICE + len(toks[k])
        for layer in (0, 3, 5):
            for kv in (0, 1):
                d = np.abs(eng.read_kv(k, layer, kv, s.current_end) - s.kv(layer, kv)).max()
                assert d < 6e-2, (k, layer, kv, d)                        # bf16 cache, entries of scale ~8
        streams[k] = s
    rng = np.random.default_rng(21)
    worst = [0.0, 0.0, 1e9]
    n_sync, n_pipe = 8, 6
    noise = (rng.standard_normal((n_sync + n_pipe, B, 32)) * np.sqrt(0.7)).astype(np.float32)
    refs = {k: [streams[k].step(noise[i, k]) for i in range(n_sync + n_pipe)] for k in check}
    for i in range(n_sync):                                               # synchronous b200_step
        gp, prod, glat, geos = eng.step(0, B, noise[i])
        assert prod.all()
        for k in check:
            ok, lat, pcm, e = refs[k][i]
            assert ok and abs(geos[k] - e) < 5e-2
            r = _check_frame((share, "step", i, k), lat, pcm, glat[k], gp[k])
            worst = [max(worst[0], r[0]), max(worst[1], r[1]), min(worst[2], r[2])]
    pcm = np.zeros((B, 1920), np.float32); produced = np.zeros(B, np.int32)
    got = []
    eng.submit(0, B, noise[n_sync]); eng.submit(0, B, noise[n_sync + 1])   # pipelined pair: Mimi(t) interleaved with FlowLM(t+1)
    for i in range(2, n_pipe):
        eng.submit(0, B, noise[n_sync + i]); eng.collect_into(pcm, produced); got.append(pcm.copy())
    for _ in range(2):
        eng.collect_into(pcm, produced); got.append(pcm.copy())
    for i in range(n_pipe):
        for k in check:
            ok, lat, rp, e = refs[k][n_sync + i]
            s = snr_db(rp, got[i][k])
            assert s > SNR_MIN, (share, "submit/collect", i, k, s)
            worst[2] = min(worst[2], s)
    print(f"\n[bench-config parity, prefix_share={share}] slots {check}: latent max-abs {worst[0]:.4f}, rel-L2 {worst[1]:.4f}, min SNR {worst[2]:.1f} dB "
          f"at KV length ~{streams[0].current_end}")


def test_shared_and_private_prefix_agree(P, model_dir, oracle_mod):
    """Cascade attention (prefix on tensor cores + streamed suffix) vs the reference's copy_states layout: same sentences, same noise."""
    texts = ["Hello world.", BENCH_SENTENCE, "One two three four five six seven eight nine ten eleven twelve.", "Short one.", BENCH_SENTENCE, "Hello world."]
    outs = []
    for share in (1, 0):
        c = P.Context(model_dir, max_slots=8, kv_capacity=512, prefix_share=share)
        st = c.stream("cosette", temp=0.7)
        toks = [c.tokenize(t) for t in texts]
        c.engine.begin_sentences(list(range(6)), [st.voice] * 6, toks, [oracle_mod.max_gen_len_for(t) for t in texts],
                                 [oracle_mod.frames_after_eos_guess(t) for t in texts], [0.7] * 6)
        rng = np.random.default_rng(2)
        noise = (rng.standard_normal((10, 6, 32)) * np.sqrt(0.7)).astype(np.float32)
        outs.append([c.engine.step(0, 6, noise[i]) for i in range(10)])
    for i in range(10):
        a, b = outs[0][i], outs[1][i]
        assert np.array_equal(a[1], b[1])
        for k in range(6):
            # same math, different summation order: bf16 rounding flips feed back through the latent (free running), so the bound is
            # the engine-vs-oracle one
            assert np.abs(a[2][k] - b[2][k]).max() < LAT_MAXABS, (i, k)
            assert snr_db(b[0][k], a[0][k]) > SNR_MIN, (i, k)


def test_f32_checkpoint_against_f32_weights_oracle(P, oracle_mod):
    """With an F32 checkpoint the reference computes f32 linears (src/loader.h:205-210); the engine always rounds weights and the
    activation operand to bf16. Measured cost of that choice on B200 (teacher-forced, 12 frames): latent max-abs 1.9e-2, rel-L2 5.4e-3,
    waveform SNR 46.0 dB -- i.e. inside the tolerances used against the BF16-checkpoint oracle, which are asserted here too."""
    from make_assets import default_model_dir
    d = default_model_dir(eos_mode="never", dtype="F32")
    orc = oracle_mod.Oracle(d, threads=os.cpu_count() or 1)
    assert orc.file_dtype == "F32"
    c = P.Context(d, max_slots=4, kv_capacity=512)
    st = c.stream("cosette", temp=0.7)
    toks = c.tokenize(BENCH_SENTENCE)
    c.engine.begin_sentences([0, 1, 2, 3], [st.voice] * 4, [toks] * 4, [oracle_mod.max_gen_len_for(BENCH_SENTENCE)] * 4, [3] * 4, [0.7] * 4)
    os_ = orc.stream("cosette", kv_capacity=512)
    os_.sentence_init(BENCH_SENTENCE)
    rng = np.random.default_rng(4)
    worst = [0.0, 0.0, 1e9]
    for i in range(12):
        noise = (rng.standard_normal(32) * np.sqrt(0.7)).astype(np.float32)
        ok, lat, pcm, e = os_.step(noise)
        gp, prod, glat, geos = c.engine.step(0, 4, np.stack([noise] * 4))
        err = float(np.abs(glat[3] - lat).max()); rel = float(np.linalg.norm(glat[3] - lat) / np.linalg.norm(lat)); snr = snr_db(pcm, gp[3])
        worst = [max(worst[0], err), max(worst[1], rel), min(worst[2], snr)]
        # teacher forcing keeps the comparison per frame (errors of a bf16-weight model would otherwise feed back through the latent)
        c.engine.debug_set_latent(0, 4, np.stack([lat] * 4))
    print(f"\n[F32 checkpoint vs f32-weights oracle] latent max-abs {worst[0]:.4f}, rel-L2 {worst[1]:.4f}, min SNR {worst[2]:.1f} dB")
    assert worst[0] < LAT_MAXABS and worst[1] < LAT_REL and worst[2] > SNR_MIN, worst


def test_two_voices_in_one_batch(P, model_dir, orc, oracle_mod):
    """max_voices > 1: rows are grouped per voice for the shared-prefix tiles; every slot must match the oracle stream of ITS voice."""
    c = P.Context(model_dir, max_slots=8, max_voices=2, kv_capacity=512)
    eng = c.engine
    sa, sb = c.stream("cosette", temp=0.7), c.stream("alba", temp=0.7)
    assert sa.voice != sb.voice
    texts = [BENCH_SENTENCE, "Hello world.", "Short one.", BENCH_SENTENCE, "How are you today my friend?", "Hello world."]
    voices = [sa.voice, sb.voice, sb.voice, sb.voice, sa.voice, sa.voice]
    names = {sa.voice: "cosette", sb.voice: "alba"}
    toks = [c.tokenize(t) for t in texts]
    eng.begin_sentences(list(range(6)), voices, toks, [oracle_mod.max_gen_len_for(t) for t in texts], [oracle_mod.frames_after_eos_guess(t) for t in texts], [0.7] * 6)
    streams = []
    for k in range(6):
        s = orc.stream(names[voices[k]], kv_capacity=512)
        assert s.sentence_init(texts[k]) == toks[k]
        streams.append(s)
    rng = np.random.default_rng(8)
    for i in range(8):
        noise = (rng.standard_normal((6, 32)) * np.sqrt(0.7)).astype(np.float32)
        gp, prod, glat, geos = eng.step(0, 6, noise)
        for k in range(6):
            ok, lat, pcm, e = streams[k].step(noise[k])
            assert ok and prod[k] == 1
            _check_frame(("two voices", i, k), lat, pcm, glat[k], gp[k])


def test_second_sentence_through_stream_api(P, model_dir, orc, oracle_mod):
    """ptts_stream_receive rolls to the next sentence (reference src/pocket_tts.cpp:494-519): prefix restore + Mimi reset + prefill of
    sentence 2 must give the oracle's first frames of that sentence (temp 0: deterministic, independent of sentence 1's audio)."""
    c = P.Context(model_dir, max_slots=1, kv_capacity=1024)
    P.set_seed(0)
    st = c.stream("cosette", temp=0.0)
    text = "Hello there. How are you?"
    st.send(text); st.flush()
    sp = oracle_mod.StrProcessor(); sp.ingest(text); sp.flush()
    n1 = oracle_mod.max_gen_len_for(sp.sentences[0])
    frames = []
    for _ in range(n1 + 2):
        f = st.receive()
        assert f is not None
        frames.append(f.copy())
    os_ = orc.stream("cosette", kv_capacity=1024)
    os_.sentence_init(sp.sentences[1])
    for j in range(2):                                                    # frames n1, n1+1 = first two frames of sentence 2
        ok, lat, pcm, e = os_.step(None)
        assert ok and snr_db(pcm, frames[n1 + j]) > SNR_MIN, j


def test_device_rng_moments(P, model_dir, oracle_mod):
    """Device noise (Philox-4x32-10 + Box-Muller, keyed by seed/slot/step; the reference draws N(0, sqrt(temp)) on the host,
    src/context.h:465-509): mean, variance, kurtosis and independence across slots and steps of ~200k draws."""
    Bn = 64
    c = P.Context(model_dir, max_slots=Bn, kv_capacity=512)
    eng = c.engine
    st = c.stream("cosette", temp=0.7)
    toks = c.tokenize(BENCH_SENTENCE)
    eng.set_seed(4242)
    eng.begin_sentences(list(range(Bn)), [st.voice] * Bn, [toks] * Bn, [137] * Bn, [1 << 20] * Bn, [0.7] * Bn)
    draws = []
    for i in range(100):
        eng.step_enqueue(0, Bn)
        draws.append(eng.debug_read("noise_drawn", 0, Bn * 32).reshape(Bn, 32))
    z = np.stack(draws).astype(np.float64)                                # [step][slot][32]
    n = z.size
    assert abs(z.mean()) < 4 * np.sqrt(0.7 / n)
    assert abs(z.var() / 0.7 - 1.0) < 0.02
    k = ((z - z.mean()) ** 4).mean() / z.var() ** 2
    assert abs(k - 3.0) < 0.1, k
    assert len(np.unique(z)) > 0.98 * n                                   # no repeated blocks across slots / steps
    flat = z.reshape(100, -1)
    assert abs(np.corrcoef(flat[:-1].ravel(), flat[1:].ravel())[0, 1]) < 0.01     # step t vs t+1
    assert abs(np.corrcoef(z[:, :-1].ravel(), z[:, 1:].ravel())[0, 1]) < 0.01     # slot s vs s+1
    assert abs(np.corrcoef(z[..., 0::2].ravel(), z[..., 1::2].ravel())[0, 1]) < 0.01   # the two Box-Muller outputs of a draw


@pytest.mark.parametrize("share", [0, 1], ids=["private_prefix", "shared_prefix"])
def test_kv_capacity_edge_never_overruns(share, P, model_dir, oracle_mod):
    """ADVICE r1 (high): a sentence clamped by the KV capacity ends with position == capacity; the finished slot stays in the stepped
    range and must NOT append another row (that row would be row 0 of the next slot / of the voice prefix)."""
    cap = 192
    c = P.Context(model_dir, max_slots=2, max_voices=1, kv_capacity=cap, prefix_share=share)
    eng = c.engine
    st = c.stream("cosette", temp=0.7)
    texts = [BENCH_SENTENCE, "One two three four five six seven eight nine ten eleven twelve."]
    toks = [c.tokenize(t) for t in texts]
    eng.begin_sentences([0, 1], [st.voice] * 2, toks, [oracle_mod.max_gen_len_for(t) for t in texts], [1 << 20] * 2, [0.7] * 2)
    room = [cap - (125 + len(t)) for t in toks]
    assert all(r < oracle_mod.max_gen_len_for(t) for r, t in zip(room, texts))      # both sentences are clamped by the capacity
    voice_slot = 2                                                         # max_slots + voice id
    before = {(s, l, kv): eng.read_kv(s, l, kv, 125 if s == voice_slot else 8) for s in (1, voice_slot) for l in (0, 5) for kv in (0, 1)}
    counts = np.zeros(2, int)
    rng = np.random.default_rng(0)
    for i in range(max(room) + 6):                                         # keeps stepping the finished slots (as a batch server would)
        noise = (rng.standard_normal((2, 32)) * np.sqrt(0.7)).astype(np.float32)
        gp, prod, glat, geos = eng.step(0, 2, noise)
        counts += prod
    assert list(counts) == room
    assert eng.slot_position(0) == cap and eng.slot_position(1) == cap
    for (s, l, kv), ref in before.items():
        assert np.array_equal(eng.read_kv(s, l, kv, ref.shape[0]), ref), (s, l, kv)


def test_taps_localise_an_injected_weight_error(P, model_dir, orc, oracle_mod, tmp_path):
    """Engine tap points mirror the oracle's: perturb ONE weight (layer 3 linear2) in the engine's checkpoint and walk the taps; the first
    tap that disagrees with the oracle names the layer."""
    import shutil
    from make_assets import read_safetensors, write_safetensors
    bad = tmp_path / "bad_model"
    shutil.copytree(model_dir, bad)
    W = read_safetensors(os.path.join(model_dir, "tts_b6369a24.safetensors"))
    W["flow_lm.transformer.layers.3.linear2.weight"] = W["flow_lm.transformer.layers.3.linear2.weight"] * 1.5
    write_safetensors(str(bad / "tts_b6369a24.safetensors"), W, "BF16")
    o = oracle_mod.Oracle(model_dir, threads=os.cpu_count() or 1, taps=True)
    s = o.stream("cosette", kv_capacity=512)
    toks = s.sentence_init(BENCH_SENTENCE)
    rng = np.random.default_rng(1)
    noise = (rng.standard_normal(32) * np.sqrt(0.7)).astype(np.float32)
    ok, lat, pcm, e = s.step(noise)
    names = [f"flow.layer{l}" for l in range(6)] + ["mimi.upsample", "mimi.transformer", "seanet.conv0", "seanet.convt2", "seanet.res3", "seanet.res6", "seanet.res9"]

    def first_bad(path):
        c = P.Context(str(path), max_slots=4, kv_capacity=512)
        st = c.stream("cosette", temp=0.7)
        c.engine.begin_sentences([0, 1, 2, 3], [st.voice] * 4, [toks] * 4, [137] * 4, [3] * 4, [0.7] * 4)
        c.engine.debug_taps(True)
        c.engine.step(0, 4, np.stack([noise] * 4))
        for nm in names:
            ref = s.tap(nm); got = c.engine.debug_tap(nm, 2)
            assert ref is not None and ref.shape == got.shape, nm
            rel = np.linalg.norm(got - ref) / np.linalg.norm(ref)
            if rel > 2e-2:
                return nm
        return None

    assert first_bad(model_dir) is None
    assert first_bad(bad) == "flow.layer3"


def test_lookahead_frames_survive_a_second_stream(P, model_dir):
    """ADVICE r1 (medium): stream A runs one frame ahead while it is alone; when a second stream appears A's in-flight frame must be
    handed out, not dropped."""
    text = "Hello there."
    c0 = P.Context(model_dir, max_slots=2, kv_capacity=512)
    P.set_seed(5)
    a0 = c0.stream("cosette", temp=0.7)
    a0.send(text); a0.flush()
    ref = []
    while True:
        f = a0.receive()
        if f is None:
            break
        ref.append(f.copy())
    c1 = P.Context(model_dir, max_slots=2, kv_capacity=512)
    P.set_seed(5)
    a1 = c1.stream("cosette", temp=0.7)
    a1.send(text); a1.flush()
    got = [a1.receive().copy() for _ in range(3)]                         # look-ahead: one frame in flight after each receive
    b1 = c1.stream("cosette", temp=0.7)                                   # second stream: the context turns synchronous
    b1.send("Hi."); b1.flush()
    assert b1.receive() is not None
    while True:
        f = a1.receive()
        if f is None:
            break
        got.append(f.copy())
    assert len(got) == len(ref)
    for x, y in zip(got, ref):
        assert np.array_equal(x, y)
