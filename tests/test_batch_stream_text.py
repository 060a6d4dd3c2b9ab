"""CPU: streamed text into the batch (ptts_c_batch_open / send / close) over a MOCK engine, with the committed tokenizer given to the batch
through ptts_c_batch_set_text. An utterance fed in chunks makes exactly the sentence jobs of its whole text: the sentences of the reference's
splitter (oracle.StrProcessor, and the engine's own ptts_c_text_* on the same chunks), their token ids, the reference's cap and
frames_after_eos, temp, sampling controls and RNG stream ids (job index + 1). The scheduler sees the same calls as for those jobs given as
token ids (ptts_c_batch_add_tokens / append_tokens). Sends between pumps: in-order delivery, the "open" state, run() not waiting for text,
pop() resuming at a later sentence; errors and cancel."""
import ctypes
import os
import random

import numpy as np
import pytest

from conftest import REPO

TOK = os.path.join(REPO, "tests", "golden", "tokenizer.model")
FRAME = 4
B200_EINVAL = -1


class MockEngine:
    """A sentence started by begin() is live from the next submitted step and produces min(length(rng id), cap) frames; frame f of the
    sentence with RNG id r holds r * 1000 + f. begin() records every sentence's arguments."""

    def __init__(self, n_slots):
        self.n_slots = n_slots
        self.slot_job = [None] * n_slots          # [rng id, frames produced, frames to produce]
        self.queue, self.trace = [], []

    @staticmethod
    def length(rng):
        return 2 + (rng * 5) % 9

    def begin(self, user, n, slots, voices, tokens, tok_off, mg, fae, temp, rng, samp):
        call = []
        for i in range(n):
            r = int(rng[i])
            job = (int(voices[i]), tuple(tokens[tok_off[i]:tok_off[i + 1]]), int(mg[i]), int(fae[i]), float(temp[i]), r,
                   (samp[i].lsd_steps, samp[i].noise_clamp, samp[i].eos_threshold))
            self.slot_job[slots[i]] = [r, 0, min(self.length(r), int(mg[i]))]
            call.append((int(slots[i]), job))
        self.trace.append(("begin", tuple(call)))
        return 0

    def jobs(self):
        return sorted((job for c in self.trace if c[0] == "begin" for _, job in c[1]), key=lambda j: j[5])

    def submit(self, user, slot0, n):
        pcm = np.zeros((n, FRAME), np.float32); produced = np.zeros(n, np.int32)
        for s in range(n):
            j = self.slot_job[s]
            if j is not None and j[1] < j[2]:
                pcm[s] = j[0] * 1000 + j[1]; produced[s] = 1; j[1] += 1
        self.queue.append((n, pcm, produced))
        self.trace.append(("submit", n))
        return 0

    def collect(self, user, pcm_out, produced_out):
        n, pcm, produced = self.queue.pop(0)
        ctypes.memmove(pcm_out, pcm.ctypes.data, pcm.nbytes)
        ctypes.memmove(produced_out, produced.ctypes.data, produced.nbytes)
        self.trace.append(("collect",))
        return n

    def end(self, user, n, slots):
        for i in range(n):
            self.slot_job[slots[i]] = None
        self.trace.append(("end", tuple(slots[i] for i in range(n))))
        return 0


@pytest.fixture(scope="module")
def front(P):
    return P.TextFrontEnd(TOK)


def make(P, front, n_slots=8, text=True, **cfg):
    eng = MockEngine(n_slots)
    b = P.Batch(n_slots=n_slots, ops=(eng.begin, eng.submit, eng.collect, eng.end), frame_size=FRAME, begin_sampling=True)
    b.configure(**(cfg or dict(refill_min=1, refill_every=1, range_quantum=1)))
    if text:
        b.set_text(front)
    return eng, b


def expected(rng, n):
    return rng * 1000 + np.arange(n, dtype=np.float32)


# ---- random texts and chunkings ---------------------------------------------------------------------------------------------------------

WORDS = ["hello", "world", "The", "quick", "brown", "fox", "a", "I", "it's", "well-known", "42", "x", "Why", "not", "été", "café", "ok"]
PUNCT = [".", "!", "?", "...", "?!", "!?.", "?!?", ". . .", ",", ""]
SPACE = [" ", " ", " ", "  ", "\t", "\n", " \n  ", "   "]


def random_text(rnd):
    kind = rnd.random()
    if kind < 0.03:
        return rnd.choice(["", " ", "  \n\t ", "...", "?!"])
    parts = []
    for _ in range(rnd.randint(1, 6)):                        # sentences
        if rnd.random() < 0.2:
            parts.append(rnd.choice(SPACE))                   # leading whitespace run
        words = [rnd.choice(WORDS) for _ in range(rnd.randint(1, 12))]
        if rnd.random() < 0.4:
            words[0] = words[0].lower()                       # lowercase start
        parts.append(rnd.choice(SPACE).join(words) if rnd.random() < 0.3 else " ".join(words))
        parts.append(rnd.choice(PUNCT))
        parts.append(rnd.choice(SPACE) if rnd.random() < 0.8 else "")
    text = "".join(parts)
    if rnd.random() < 0.3:
        text = text.rstrip(" \t\n.!?")                        # no final terminator
    return text


def random_chunks(rnd, text):
    """Cuts at random points: single characters, cuts right after every terminator in some texts, and empty chunks in between."""
    b = text.encode()
    cuts = set()
    mode = rnd.random()
    if mode < 0.25:
        cuts = set(range(1, len(b)))                          # one byte at a time
    else:
        cuts = {i for i in range(1, len(b)) if rnd.random() < 0.15}
        if mode < 0.6:
            cuts |= {i + 1 for i, c in enumerate(b) if c in b".!?"}
    cuts = sorted(c for c in cuts if 0 < c < len(b))
    chunks, prev = [], 0
    for c in cuts + [len(b)]:
        chunks.append(b[prev:c]); prev = c
        if rnd.random() < 0.1:
            chunks.append(b"")
    return [c for c in chunks if c or rnd.random() < 0.5] if b else [b""] * rnd.randint(0, 2)


def job_of(front, sent, voice, temp, samp, rng):
    """A sentence's job by the reference's rules: its token ids, cap int((words + 2) * 12.5) and frames_after_eos."""
    import oracle
    return (voice, tuple(front.encode(sent)), oracle.max_gen_len_for(sent), oracle.frames_after_eos_guess(sent), float(np.float32(temp)), rng,
            samp)


SAMPLINGS = [(1, 0.0, -4.0), (4, 0.5, -3.0), (2, 0.0, -6.5)]


def test_streamed_text_makes_the_jobs_of_the_whole_text(P, front):
    import oracle
    rnd = random.Random(11)
    n_sentences = 0
    for t in range(200):
        text = random_text(rnd)
        chunks = random_chunks(rnd, text)
        voice, temp, samp = t % 3, (0.7, 0.5, 0.0)[t % 3], SAMPLINGS[t % 3]
        eng, b = make(P, front)
        u = b.open(voice, temp, *samp)
        ref = oracle.StrProcessor()
        front.reset()
        sentences = []
        for c in chunks:
            got = b.send(u, c)
            ref.ingest(c)
            if c:
                front.send(c)                                 # ptts_c_text_send flushes on an empty chunk; send does not
            popped = front.pop_all()
            assert got == len(ref.sentences) == len(popped), (text, chunks)   # a sentence is added once its terminator is followed
            assert popped == list(ref.sentences), (text, chunks)
            sentences += popped
            ref.sentences.clear()
        ref.flush(); front.flush()
        tail = front.pop_all()
        assert b.close(u) == len(tail) and tail == list(ref.sentences)
        sentences += tail
        whole = oracle.StrProcessor(); whole.ingest(text.encode()); whole.flush()
        assert sentences == list(whole.sentences), (text, chunks)            # any chunking splits like the whole text
        b.run()
        want = [job_of(front, s, voice, temp, samp, k + 1) for k, s in enumerate(sentences)]
        assert eng.jobs() == want, (text, chunks)
        assert b.status(u) == ("done", sum(min(MockEngine.length(j[5]), j[2]) for j in want))
        assert np.array_equal(b.read(u)[:, 0], np.concatenate([expected(j[5], min(MockEngine.length(j[5]), j[2])) for j in want] + [np.zeros(0, np.float32)]))
        n_sentences += len(sentences)
    assert n_sentences > 400


def _stream_interleaved(P, front, texts, rnd):
    """Opens an utterance per text and sends their chunks interleaved at random, closing each after its last chunk, all before the first
    pump. Returns the (utterance index, sentences) events in the order the sentences were split off."""
    import oracle
    eng, b = make(P, front, n_slots=6, refill_min=2, refill_every=3, range_quantum=4)
    events = []
    utts = [b.open(i % 3, 0.7, *SAMPLINGS[i % 3]) for i in range(len(texts))]
    pending = {i: random_chunks(rnd, t) + [None] for i, t in enumerate(texts)}    # None: close
    splitters = {i: oracle.StrProcessor() for i in range(len(texts))}
    while pending:
        i = rnd.choice(sorted(pending))
        c = pending[i].pop(0)
        if c is None:
            del pending[i]
            splitters[i].flush()
            assert b.close(utts[i]) == len(splitters[i].sentences)
        else:
            splitters[i].ingest(c)
            assert b.send(utts[i], c) == len(splitters[i].sentences)
        events.append((i, list(splitters[i].sentences))); splitters[i].sentences.clear()
    return eng, b, utts, events


def test_interleaved_streams_take_the_token_path(P, front):
    """Sentences of several utterances split off in any interleaving reach the scheduler exactly as the same sentences given as token ids
    (add_tokens for an utterance's first sentence, append_tokens for the next ones) in the same order."""
    import oracle
    rnd = random.Random(5)
    for rep in range(6):
        texts = [random_text(rnd) for _ in range(10)]
        eng, b, utts, events = _stream_interleaved(P, front, texts, rnd)
        eng2, b2 = make(P, front, n_slots=6, refill_min=2, refill_every=3, range_quantum=4)
        utts2 = {}
        for i, sents in events:
            for s in sents:
                ids = front.encode(s)
                args = (i % 3, ids, oracle.max_gen_len_for(s), oracle.frames_after_eos_guess(s), 0.7, 0)
                kw = dict(zip(("lsd_steps", "noise_clamp", "eos_threshold"), SAMPLINGS[i % 3]))
                if i in utts2:
                    b2.add_tokens(*args, utt=utts2[i], **kw)
                else:
                    utts2[i] = b2.add_tokens(*args, **kw)
        b.run(); b2.run()
        assert eng.trace == eng2.trace and len(eng.trace) > 10                 # call for call, every argument of every sentence start
        for i, u in enumerate(utts):
            if i in utts2:
                assert b.status(u) == b2.status(utts2[i]) and np.array_equal(b.read(u), b2.read(utts2[i]))
            else:
                assert b.status(u) == ("done", 0) and b.frames(u) == 0     # text without a sentence


def test_sends_between_pumps(P, front):
    eng, b = make(P, front, n_slots=2)
    import oracle
    other = b.open(1, 0.7)
    assert b.send(other, "Another utterance runs beside it") == 0
    u = b.open(0, 0.7)
    assert b.status(u) == ("open", 0)
    assert b.send(u, "Hello there my friend") == 0 and b.send(u, ".") == 0         # a terminator alone completes nothing yet ...
    assert b.send(u, " How") == 1                                                     # ... the next character does: rng 1
    assert b.send(other, ". x") == 1                                                  # rng 2
    assert b.status(u)[0] == "queued"
    states, popped = [], []
    while True:
        got = b.pump(1)
        states.append(b.status(u)[0]); popped.append(b.pop(u))
        if not got:
            break
    assert states[0] == "running" and states[-1] == "open"
    assert b.run() == 0                                                               # nothing queued or running: run() does not wait for text
    assert b.status(u) == ("open", 0) and b.pop(u).shape == (0, FRAME)
    len1 = min(MockEngine.length(1), oracle.max_gen_len_for("Hello there my friend."))
    assert np.array_equal(np.concatenate(popped)[:, 0], expected(1, len1))
    assert b.send(u, " are you? I am") == 1                                           # rng 3: "How are you?"
    assert b.status(u)[0] == "running"                                                # an earlier sentence ran: the utterance has started
    assert b.run() > 0 and b.status(u)[0] == "open"                                   # run() runs what was sent and returns
    later = b.pop(u)                                                                  # pop resumes at the new sentence
    assert np.array_equal(later[:, 0], expected(3, MockEngine.length(3)))
    assert b.send(u, " fine") == 0 and b.close(u) == 1                               # rng 4: "I am fine." (final period)
    assert b.status(u)[0] == "running"
    while b.pump(1):
        pass
    assert b.status(u) == ("done", MockEngine.length(4))
    assert np.array_equal(b.pop(u)[:, 0], expected(4, MockEngine.length(4)))
    assert b.status(u) == ("done", 0) and b.frames(u) == len1 + MockEngine.length(3) + MockEngine.length(4)
    assert b.status(other)[0] == "open"
    assert b.close(other) == 1 and b.run() > 0 and b.status(other)[0] == "done"
    starts = [job[5] for c in eng.trace if c[0] == "begin" for _, job in c[1]]
    assert sorted(starts) == [1, 2, 3, 4, 5]


def test_delivery_in_order_while_sentences_arrive(P, front):
    """Sentences of one utterance sent while earlier ones still run, on 3 slots with other utterances: popped audio is each sentence's
    frames in the order they were sent."""
    rnd = random.Random(2)
    eng, b = make(P, front, n_slots=3)
    texts = ["One two three. Four five six seven eight! Nine? Ten eleven. " * 3, "Alpha beta. Gamma delta epsilon. Zeta eta theta iota. " * 2]
    utts = [b.open(i, 0.7) for i in range(2)]
    chunks = [random_chunks(rnd, t) for t in texts]
    order = {u: [] for u in utts}
    popped = {u: [] for u in utts}
    rng_of = []                                                                      # RNG id of every sentence, in the order they were added
    while True:
        for i, u in enumerate(utts):
            if chunks[i] and rnd.random() < 0.5:
                for _ in range(b.send(u, chunks[i].pop(0))):
                    rng_of.append(u); order[u].append(len(rng_of))
                if not chunks[i]:
                    for _ in range(b.close(u)):
                        rng_of.append(u); order[u].append(len(rng_of))
            popped[u].append(b.pop(u))
        if not b.pump(1) and not any(chunks):
            break
    for u in utts:
        popped[u].append(b.pop(u))
        assert b.status(u) == ("done", 0)
        want = np.concatenate([expected(r, MockEngine.length(r)) for r in order[u]])
        assert np.array_equal(np.concatenate(popped[u])[:, 0], want)
    assert len(order[utts[0]]) == 12 and len(order[utts[1]]) == 6


def test_errors_and_cancel(P, front):
    L = P.lib()
    eng, b = make(P, front, n_slots=2)
    u = b.open(0, 0.7)
    assert b.close(u) == 0
    assert b.status(u) == ("done", 0) and b.frames(u) == 0                            # open + close without text: done, no frames
    assert L.ptts_c_batch_send(b.h, u, b"More text. ") == B200_EINVAL               # send after close
    assert L.ptts_c_batch_close(b.h, u) == B200_EINVAL                               # close twice
    for bad in (-1, u + 1, 1 << 20):                                                  # unknown ids
        assert L.ptts_c_batch_send(b.h, bad, b"x") == B200_EINVAL and L.ptts_c_batch_close(b.h, bad) == B200_EINVAL
    t = b.add_tokens(0, [1, 2], 10, 3)                                                # an utterance that was never open
    assert L.ptts_c_batch_send(b.h, t, b"x") == B200_EINVAL and L.ptts_c_batch_close(b.h, t) == B200_EINVAL
    assert L.ptts_c_batch_send(None, u, b"x") == B200_EINVAL and L.ptts_c_batch_send(b.h, u, None) == B200_EINVAL
    assert L.ptts_c_batch_open_id(b.h, -1, 0.7, None) == B200_EINVAL
    bad = P.Sampling(9, 0.0, -4.0)
    assert L.ptts_c_batch_open_id(b.h, 0, 0.7, ctypes.byref(bad)) == B200_EINVAL
    assert L.ptts_c_batch_open(b.h, b"cosette", 0.7, None) == B200_EINVAL            # voice names need a context
    _, nb = make(P, front, text=False)
    assert L.ptts_c_batch_open_id(nb.h, 0, 0.7, None) == B200_EINVAL                # no tokenizer
    assert L.ptts_c_batch_set_text(None, front.h) == B200_EINVAL
    b.run()

    # cancelling an open utterance drops its queued sentences and closes it
    c = b.open(0, 0.7)
    assert b.send(c, "First one. Second one. Third") == 2
    assert b.status(c)[0] == "queued"
    b.cancel(c)
    assert b.status(c) == ("cancelled", 0)
    assert L.ptts_c_batch_send(b.h, c, b" more. ") == B200_EINVAL and L.ptts_c_batch_close(b.h, c) == B200_EINVAL
    mark = len(eng.trace)
    assert b.run() == 0 and eng.trace[mark:] == [] and b.frames(c) == 0
    # ... and an open utterance whose sentences are done is cancelled too (not left "done")
    d = b.open(1, 0.7)
    b.send(d, "Done soon. ")
    b.run()
    assert b.status(d)[0] == "open"
    b.cancel(d)
    assert b.status(d) == ("cancelled", 0) and L.ptts_c_batch_send(b.h, d, b"x") == B200_EINVAL
    # a running open utterance: its slot is freed and ended, the other sentences are unaffected
    e = b.open(0, 0.7)
    keep = b.open(1, 0.7)
    b.send(e, "Long sentence number one goes here. ")
    b.send(keep, "Kept sentence. ")
    b.send(e, "x")
    b.pump(1)
    assert b.status(e)[0] == "running"
    b.cancel(e)
    b.close(keep)
    while b.pump(1):
        pass
    assert b.status(e)[0] == "cancelled" and b.status(keep)[0] == "done" and any(c_[0] == "end" for c_ in eng.trace)
    r = [job[5] for c_ in eng.trace if c_[0] == "begin" for _, job in c_[1] if job[1] == tuple(front.encode("Kept sentence."))][0]
    assert np.array_equal(b.read(keep)[:, 0], expected(r, MockEngine.length(r)))
