"""GPU: streamed text into a batch on the engine (ptts_c_batch_open / send / close). With every send before the first pump an utterance's
audio is bitwise that of ptts_c_batch_add of its whole text. Sentences sent between the pumps of a running batch give bitwise the audio of
the same sentences appended as token ids (append_tokens_sampling) at the same pumps with the same RNG ids, caps and frames_after_eos, so the
text path reaches the engine exactly as the token path does. Frame counts follow the reference's caps on the never-EOS checkpoint, the
bookkeeping adds up on the EOS checkpoint, and each streamed sentence starts like a single-slot run with its RNG id."""
import random

import numpy as np
import pytest

from conftest import snr_db
from test_gpu_batch import TEXTS

pytestmark = pytest.mark.gpu

VOICES = ("cosette", "alba")


def _batch(P, model_dir, n_slots=4):
    c = P.Context(model_dir, max_slots=n_slots, max_voices=2, kv_capacity=512)
    P.set_seed(77)
    b = P.Batch(c, n_slots)
    b.configure(refill_min=1, refill_every=2, range_quantum=4)
    return c, b


def _chunks(rnd, text):
    """Random cuts: runs of single characters, cuts right after terminators and longer pieces."""
    out, i = [], 0
    while i < len(text):
        n = rnd.choice([1, 1, 2, 5, 15, 40])
        out.append(text[i:i + n]); i += n
    return out


@pytest.mark.parametrize("ckpt", ["model_dir", "model_dir_eos"])
def test_streamed_utterances_equal_add(P, request, oracle_mod, ckpt):
    model_dir = request.getfixturevalue(ckpt)
    out = {}
    for mode in ("add", "stream"):
        c, b = _batch(P, model_dir)
        rnd = random.Random(3)
        utts = []
        for i, t in enumerate(TEXTS):
            if mode == "add":
                utts.append(b.add(VOICES[i % 2], t, 0.7))
            else:
                u = b.open(VOICES[i % 2], 0.7)
                for ch in _chunks(rnd, t):
                    b.send(u, ch)
                b.close(u)
                utts.append(u)
        total = b.run()
        st = b.stats()
        out[mode] = (total, [b.frames(u) for u in utts], [b.read(u) for u in utts], {k: st[k] for k in ("steps", "frames", "sentences", "refills")},
                     [b.status(u) for u in utts])
        c.close()
    assert out["add"][0] == out["stream"][0] and out["add"][1] == out["stream"][1] and out["add"][3] == out["stream"][3]
    for a, s in zip(out["add"][2], out["stream"][2]):
        assert np.array_equal(a, s)
    assert all(st == ("done", f) for st, f in zip(out["stream"][4], out["stream"][1]))
    if ckpt == "model_dir":
        caps = []
        for t in TEXTS:
            sp = oracle_mod.StrProcessor(); sp.ingest(t); sp.flush()
            caps.append(sum(oracle_mod.max_gen_len_for(s) for s in sp.sentences))
        assert out["stream"][1] == caps


# utterances whose text arrives while the batch runs (two or three sentences each), beside utterances added whole at the start
STREAMED = [TEXTS[5] + " " + TEXTS[2], TEXTS[1] + "   " + TEXTS[4] + " " + TEXTS[3].lower(), TEXTS[6] + " and then some words without an end"]
BACKGROUND = TEXTS[8:12]


def _online(P, model_dir, oracle_mod, tokens):
    """Pumps a batch while the STREAMED texts arrive a chunk per pump. tokens=False: ptts_c_batch_send / close. tokens=True: a host mirror
    of the splitter gets the same chunks and each sentence it completes is appended as token ids with the reference's cap and
    frames_after_eos and RNG id 0 (= job index + 1, the id the text path gives it). Returns the popped audio, each streamed sentence's
    (RNG id, text, cap), the final and the seen states, the batch stats and the frame count of every utterance."""
    c, b = _batch(P, model_dir)
    job, background = 0, []
    for i, t in enumerate(BACKGROUND):
        background.append(b.add(VOICES[i % 2], t, 0.7))
        sp = oracle_mod.StrProcessor(); sp.ingest(t); sp.flush()
        job += len(sp.sentences)
    utts = [b.open(VOICES[i % 2], 0.7) for i in range(len(STREAMED))]
    voice_ids = {VOICES[0]: 0, VOICES[1]: 1}                 # resolved in this order on a fresh context
    assert P.lib().b200_voice_len(c.engine.h, 1) > 0 and P.lib().b200_voice_len(c.engine.h, 2) < 0
    rnd = random.Random(9)
    chunks = [_chunks(rnd, t) for t in STREAMED]
    mirror = [oracle_mod.StrProcessor() for _ in STREAMED]
    sentences = {u: [] for u in utts}
    popped = {u: [] for u in utts}
    open_states = {u: set() for u in utts}                   # states reported while the utterance was open
    k = 0
    while True:
        if k % 3 == 0:                                       # a chunk of every open utterance every third pump
            for i, u in enumerate(utts):
                if chunks[i] is None:
                    continue
                if chunks[i]:
                    ch = chunks[i].pop(0)
                    mirror[i].ingest(ch)
                    n = 0 if tokens else b.send(u, ch)
                else:
                    chunks[i] = None
                    mirror[i].flush()
                    n = b.close(u)
                assert n == (0 if tokens else len(mirror[i].sentences))
                for s in mirror[i].sentences:
                    job += 1
                    cap, fae = oracle_mod.max_gen_len_for(s), oracle_mod.frames_after_eos_guess(s)
                    sentences[u].append((job, s.decode(), cap))
                    if tokens:
                        b.add_tokens(voice_ids[VOICES[i % 2]], c.tokenize(s.decode()), cap, fae, 0.7, rng_stream=0, utt=u)
                mirror[i].sentences.clear()
        got = b.pump(1)
        for u in utts:
            popped[u].append(b.pop(u))
            if chunks[utts.index(u)] is not None:
                open_states[u].add(b.status(u)[0])
        k += 1
        if not got and all(ch is None for ch in chunks):
            break
    st = b.stats()
    res = ({u: np.concatenate(popped[u]) for u in utts}, sentences, {u: b.status(u) for u in utts}, open_states,
           {k_: st[k_] for k_ in ("steps", "frames", "sentences", "refills")}, [b.frames(u) for u in background + utts])
    c.close()
    return res


def test_sentences_between_pumps_take_the_token_path(P, model_dir, oracle_mod):
    pcm_t, sent_t, status_t, open_t, st_t, frames_t = _online(P, model_dir, oracle_mod, tokens=False)
    pcm_k, sent_k, status_k, _, st_k, frames_k = _online(P, model_dir, oracle_mod, tokens=True)
    assert sent_t == sent_k and st_t == st_k and status_t == status_k and frames_t == frames_k
    assert all("done" not in s for s in open_t.values())                                 # an open utterance is never reported done
    for u in pcm_t:
        assert np.array_equal(pcm_t[u], pcm_k[u]), u
        assert status_t[u] == ("done", 0)
        assert len(pcm_t[u]) == sum(cap for _, _, cap in sent_t[u])          # never-EOS checkpoint: every sentence runs to its cap
    assert [len(sent_t[u]) for u in sorted(sent_t)] == [3, 3, 2]

    # each streamed sentence starts like a single-slot run of the engine with its RNG id
    d = P.Context(model_dir, max_slots=2, max_voices=2, kv_capacity=512)
    d.engine.set_seed(77)
    voices = (d.stream(VOICES[0]).voice, d.stream(VOICES[1]).voice)
    for i, u in enumerate(sorted(sent_t)):
        off = 0
        for rng, s, cap in sent_t[u]:
            d.engine.begin_sentences([0], [voices[i % 2]], [d.tokenize(s)], [cap], [oracle_mod.frames_after_eos_guess(s)], [0.7], rng_streams=[rng])
            for f in range(4):
                pcm, prod, _, _ = d.engine.step(0, 1, None)
                assert prod[0] == 1 and snr_db(pcm[0], pcm_t[u][off + f]) > 40.0, (u, s, f)
            off += cap
    d.close()


def test_sentences_between_pumps_with_eos_checkpoint(P, model_dir_eos, oracle_mod):
    pcm, sents, status, open_states, st, frames = _online(P, model_dir_eos, oracle_mod, tokens=False)
    n_bg = 0
    for t in BACKGROUND:
        sp = oracle_mod.StrProcessor(); sp.ingest(t); sp.flush()
        n_bg += len(sp.sentences)
    assert st["sentences"] == n_bg + sum(len(v) for v in sents.values())
    assert st["frames"] == sum(frames)
    n_early = 0
    for u in pcm:
        cap = sum(c for _, _, c in sents[u])
        assert status[u] == ("done", 0) and len(pcm[u]) == frames[len(BACKGROUND) + sorted(pcm).index(u)]
        assert 1 <= len(pcm[u]) <= cap and np.isfinite(pcm[u]).all()
        assert "done" not in open_states[u]
        n_early += len(pcm[u]) < cap
    assert n_early >= 1                                                  # the EOS rule ends streamed sentences before their cap
