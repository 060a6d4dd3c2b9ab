"""GPU: online continuous batching on the engine. b200_end_sentences retires slots stream-ordered (dead rows from the next enqueued step on,
under CUDA graphs and both pipeline modes) without touching the other rows' arithmetic; a pump loop takes exactly the decisions of run();
utterances added in waves between pumps get their own audio, handed out in order by pop(); a cancelled utterance stops growing while its
slot goes to the next queued sentence and the other utterances are unaffected."""
import ctypes

import numpy as np
import pytest

from conftest import snr_db
from test_gpu_batch import TEXTS

pytestmark = pytest.mark.gpu

END_TEXTS = ["Hello world.", "Water runs down the mountain toward the sea.", "Read the letter again.", "Numbers like forty two are words too."]


def _sentences(oracle_mod, text):
    sp = oracle_mod.StrProcessor(); sp.ingest(text); sp.flush()
    return [s.decode() if isinstance(s, bytes) else s for s in sp.sentences]


def _steps(eng, n_steps, n, end_after=None, end_slots=()):
    """n_steps pipelined steps of slots [0, n) with up to two in flight; b200_end_sentences is enqueued after step `end_after` was submitted."""
    pcm = np.zeros((n_steps, n, 1920), np.float32); prod = np.zeros((n_steps, n), np.int32)
    submitted = collected = 0
    while collected < n_steps:
        while submitted < n_steps and submitted - collected < 2:
            eng.submit(0, n); submitted += 1
            if submitted == end_after:
                eng.end_sentences(end_slots)
        eng.collect_into(pcm[collected], prod[collected]); collected += 1
    return pcm, prod


@pytest.mark.parametrize("overlap", [0, 1])
def test_end_sentences(P, model_dir, oracle_mod, overlap):
    runs = {}
    for ended in (False, True):
        c = P.Context(model_dir, max_slots=4, max_voices=1, kv_capacity=512, cuda_graphs=1, overlap=overlap)
        c.engine.set_seed(77)
        v = c.stream("cosette").voice
        toks = [c.tokenize(t) for t in END_TEXTS]
        c.engine.begin_sentences([0, 1, 2, 3], [v] * 4, toks, [200] * 4, [3] * 4, [0.7] * 4, rng_streams=[1, 2, 3, 4])
        # steps 1-2 are enqueued before the end and see all four slots live; steps 3-8 see slots 1 and 3 dead
        pcm, prod = _steps(c.engine, 8, 4, end_after=2 if ended else None, end_slots=[1, 3])
        pos = [c.engine.slot_position(s) for s in range(4)]
        runs[ended] = (c, v, pcm, prod, pos, [P.lib().b200_voice_len(c.engine.h, v) + len(t) for t in toks])
    c, v, pcm, prod, pos, start = runs[True]
    assert (prod[:2] == 1).all()
    assert (prod[2:] == np.array([1, 0, 1, 0])).all()
    assert pos == [start[0] + 8, start[1] + 2, start[2] + 8, start[3] + 2]          # no KV append on the ended slots
    _, _, pcm0, prod0, pos0, _ = runs[False]
    assert (prod0 == 1).all() and pos0 == [s + 8 for s in start]
    for s in (0, 2):                                                               # dead rows do not touch the other rows' arithmetic
        assert np.array_equal(pcm[:, s], pcm0[:, s]), s
    assert np.array_equal(pcm[:2, 1], pcm0[:2, 1]) and np.array_equal(pcm[:2, 3], pcm0[:2, 3])

    # a sentence started on an ended slot sounds like the same sentence on a fresh engine
    text = "A small bird sings in the morning light while the city sleeps."
    toks = c.tokenize(text)
    cap, fae = oracle_mod.max_gen_len_for(text), oracle_mod.frames_after_eos_guess(text)
    c.engine.begin_sentences([1], [v], [toks], [cap], [fae], [0.7], rng_streams=[9])
    pcm_new, prod_new = _steps(c.engine, 4, 4)
    assert (prod_new == np.array([1, 1, 1, 0])).all()
    fresh = P.Context(model_dir, max_slots=4, max_voices=1, kv_capacity=512, cuda_graphs=1, overlap=overlap)
    fresh.engine.set_seed(77)
    fv = fresh.stream("cosette").voice
    fresh.engine.begin_sentences([0], [fv], [toks], [cap], [fae], [0.7], rng_streams=[9])
    for f in range(4):
        ref, p, _, _ = fresh.engine.step(0, 1, None)
        assert p[0] == 1 and snr_db(ref[0], pcm_new[f, 1]) > 40.0, f
    for ctx in (runs[False][0], c, fresh):
        ctx.close()


def test_end_sentences_rejects_bad_arguments(P, model_dir):
    c = P.Context(model_dir, max_slots=4, max_voices=1, kv_capacity=512)
    L, h = P.lib(), c.engine.h
    ip = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    assert L.b200_end_sentences(h, 1, ip(np.array([4], np.int32))) == -1
    assert L.b200_end_sentences(h, 1, ip(np.array([-1], np.int32))) == -1
    assert L.b200_end_sentences(h, -1, ip(np.array([0], np.int32))) == -1
    assert L.b200_end_sentences(h, 1, None) == -1
    assert L.b200_end_sentences(h, 0, None) == 0
    c.close()


def _batch(P, model_dir, n_slots=4, **cfg):
    c = P.Context(model_dir, max_slots=n_slots, max_voices=2, kv_capacity=512)
    P.set_seed(77)
    b = P.Batch(c, n_slots)
    b.configure(**cfg)
    return c, b


def test_pump_loop_matches_run(P, model_dir):
    out = {}
    for mode in ("run", "pump"):
        c, b = _batch(P, model_dir, refill_min=1, refill_every=2, range_quantum=4)
        utts = [b.add(("cosette", "alba")[i % 2], t, 0.7) for i, t in enumerate(TEXTS)]
        if mode == "run":
            b.run()
        else:
            while b.pump(1):
                pass
        st = b.stats()
        out[mode] = ([b.read(u) for u in utts], {k: st[k] for k in ("steps", "frames", "slot_steps", "sentences", "refills")})
        c.close()
    assert out["run"][1] == out["pump"][1]
    for a, p in zip(out["run"][0], out["pump"][0]):
        assert np.array_equal(a, p)


WAVES = [(0, 4), (4, 8), (8, 12)]     # utterances TEXTS[a:b] arrive after 0, 6 and 15 pumps


def _online(P, model_dir, pop):
    c, b = _batch(P, model_dir, refill_min=1, refill_every=2, range_quantum=4)
    utts, popped, pumps = [], {}, 0
    for w, (a, z) in enumerate(WAVES):
        utts += [b.add(("cosette", "alba")[i % 2], TEXTS[i], 0.7) for i in range(a, z)]
        until = (6, 15, 1 << 30)[w]
        while pumps < until and b.pump(1):
            pumps += 1
            if pop:
                for u in utts:
                    popped.setdefault(u, []).append(b.pop(u))
    return c, b, utts, popped


def test_online_arrivals(P, model_dir, oracle_mod):
    c, b, utts, popped = _online(P, model_dir, pop=True)
    sents = [_sentences(oracle_mod, t) for t in TEXTS]
    caps = [[oracle_mod.max_gen_len_for(s) for s in ss] for ss in sents]
    got = [np.concatenate(popped[u]) for u in utts]
    for u, cp, g in zip(utts, caps, got):
        assert b.frames(u) == sum(cp) and g.shape == (sum(cp), 1920) and b.status(u) == ("done", 0)
    # first frames of every sentence = a direct single-slot run with the same RNG stream id (job index + 1, in order of arrival)
    d = P.Context(model_dir, max_slots=2, max_voices=2, kv_capacity=512)
    d.engine.set_seed(77)
    voices = (d.stream("cosette").voice, d.stream("alba").voice)
    job = 0
    for i, ss in enumerate(sents):
        off = 0
        for s, cap in zip(ss, caps[i]):
            job += 1
            d.engine.begin_sentences([0], [voices[i % 2]], [d.tokenize(s)], [cap], [oracle_mod.frames_after_eos_guess(s)], [0.7], rng_streams=[job])
            for f in range(3):
                pcm, prod, _, _ = d.engine.step(0, 1, None)
                assert prod[0] == 1 and snr_db(pcm[0], got[i][off + f]) > 40.0, (i, s, f)
            off += cap
    c.close(); d.close()
    # popping as the audio arrives hands out exactly what read() returns after a run of the same arrivals without pops
    c2, b2, utts2, _ = _online(P, model_dir, pop=False)
    for u, g in zip(utts2, got):
        assert np.array_equal(b2.read(u), g)
    c2.close()


def test_cancel_on_the_engine(P, model_dir_eos):
    texts = [t for t in TEXTS if t.count(".") + t.count("?") + t.count("!") == 1]     # one sentence each: a running utterance holds one slot

    def run(cancel):
        c, b = _batch(P, model_dir_eos, refill_min=1, refill_every=1, range_quantum=4)
        utts = [b.add(("cosette", "alba")[i % 2], t, 0.7) for i, t in enumerate(texts)]
        victim, frozen = None, None
        for k in range(1 << 20):
            if not b.pump(1):
                break
            if cancel and victim is None and k >= 4:
                running = [u for u in utts if b.status(u)[0] == "running"]
                queued = [u for u in utts if b.status(u)[0] == "queued"]
                assert len(running) == 4 and queued                                   # every slot busy, work waiting
                victim = max(running, key=lambda u: b.frames(u))
                b.cancel(victim)
                frozen = b.frames(victim)
                assert frozen > 0 and b.status(victim) == ("cancelled", 0)
                assert sum(b.status(u)[0] == "running" for u in utts) == 3
                b.pump(1)
                assert sum(b.status(u)[0] == "running" for u in utts) == 4            # the freed slot went to the next queued sentence
        res = ({u: b.frames(u) for u in utts}, {u: b.read(u) for u in utts}, victim, frozen)
        c.close()
        return res

    ref_frames, ref_pcm, _, _ = run(False)
    frames, pcm, victim, frozen = run(True)
    assert frames[victim] == frozen and pcm[victim].shape == (0, 1920)
    for u in ref_frames:
        if u == victim:
            continue
        assert frames[u] == ref_frames[u], u
        for f in range(min(4, frames[u])):
            assert snr_db(ref_pcm[u][f], pcm[u][f]) > 40.0, (u, f)
