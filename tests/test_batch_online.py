"""CPU: online continuous batching (pocket-tts.cpp_b200/csrc/host/batch_scheduler.hpp: pump / pop / cancel / status) through the C ABI over
a MOCK engine. The mock follows the engine's contract like the one of test_batch_scheduler.py (a sentence started by begin() becomes live
at the NEXT submitted step, produces `length` frames or stops at its cap, a finished slot reports produced = 0) and adds end(): an ended
slot is a dead row from the next submitted step on. A sentence start may reuse a slot whose sentence was ended, or belongs to a cancelled
utterance. Every call is recorded, so two drivers of the scheduler can be compared call for call."""
import ctypes

import numpy as np
import pytest

FRAME = 4
B200_EINVAL = -1


class MockEngine:
    def __init__(self, n_slots, lengths_by_stream, cancelled_streams=()):
        self.n_slots, self.lengths = n_slots, lengths_by_stream
        self.cancelled = set(cancelled_streams)   # streams whose live slot may be refilled without an end() (cancelled by the test)
        self.slot_job = [None] * n_slots          # [stream id, frames produced, length, cap]
        self.queue = []                           # in-flight steps: (n, pcm, produced)
        self.trace = []                           # every call in order
        self.steps = self.collects = 0

    @staticmethod
    def live(j):
        return j is not None and j[1] < min(j[2], j[3])

    def begin(self, user, n, slots, voices, tokens, tok_off, mg, fae, temp, rng):
        call = []
        for i in range(n):
            s, stream = slots[i], int(rng[i])
            old = self.slot_job[s]
            assert not self.live(old) or old[0] in self.cancelled, "slot refilled while its sentence is live"
            self.slot_job[s] = [stream, 0, self.lengths[stream], int(mg[i])]
            call.append((s, stream, tok_off[i + 1] - tok_off[i]))
        self.trace.append(("begin", tuple(call)))
        return 0

    def submit(self, user, slot0, n):
        assert slot0 == 0 and 0 < n <= self.n_slots and len(self.queue) < 3
        pcm = np.zeros((n, FRAME), np.float32); produced = np.zeros(n, np.int32)
        for s in range(n):
            j = self.slot_job[s]
            if self.live(j):
                pcm[s] = j[0] * 1000 + j[1]             # value identifies (sentence, frame index)
                produced[s] = 1; j[1] += 1
        self.queue.append((n, pcm, produced)); self.steps += 1
        self.trace.append(("submit", n))
        return 0

    def collect(self, user, pcm_out, produced_out):
        n, pcm, produced = self.queue.pop(0)
        ctypes.memmove(pcm_out, pcm.ctypes.data, pcm.nbytes)
        ctypes.memmove(produced_out, produced.ctypes.data, produced.nbytes)
        self.collects += 1
        self.trace.append(("collect",))
        return n

    def end(self, user, n, slots):
        ended = tuple(slots[i] for i in range(n))
        for s in ended:
            assert 0 <= s < self.n_slots
            self.slot_job[s] = None
        self.trace.append(("end", ended))
        return 0

    def ops(self, with_end=True):
        return (self.begin, self.submit, self.collect, self.end if with_end else None)


def expected(stream, n):
    return stream * 1000 + np.arange(n, dtype=np.float32)


def make(P, n_slots, lengths, cancelled=(), with_end=True, **cfg):
    eng = MockEngine(n_slots, lengths, cancelled)
    b = P.Batch(n_slots=n_slots, ops=eng.ops(with_end), frame_size=FRAME)
    if cfg:
        b.configure(**cfg)
    return eng, b


def pump_all(b, k):
    while b.pump(k):
        pass


# ---- run() and a pump loop take the same decisions --------------------------------------------------------------------------------------

def _random_jobs(seed=0, n=200):
    rng = np.random.default_rng(seed)
    lengths = [int(x) for x in rng.integers(1, 60, n)]
    caps = [int(l + rng.integers(0, 30)) if i % 5 else max(1, l // 2) for i, l in enumerate(lengths)]   # every 5th sentence is cut by its cap
    return lengths, caps


@pytest.mark.parametrize("driver", [1, 7])
def test_pump_loop_takes_the_decisions_of_run(P, driver):
    lengths, caps = _random_jobs()
    traces = {}
    for d in ("run", driver):
        eng, b = make(P, 16, {i + 1: l for i, l in enumerate(lengths)}, refill_min=2, refill_every=4, range_quantum=8)
        utts = [b.add_tokens(0, [5, 6, 7], caps[i], 3, 0.7, rng_stream=i + 1) for i in range(len(lengths))]
        if d == "run":
            total = b.run()
        else:
            total = 0
            while True:
                got = b.pump(d)
                if not got:
                    break
                total += got
        st = b.stats()
        traces[d] = (eng.trace, total, [b.read(u).tobytes() for u in utts], [b.frames(u) for u in utts],
                     {k: st[k] for k in ("steps", "frames", "slot_steps", "sentences", "refills")})
        assert eng.queue == [] and all(b.status(u) == ("done", min(lengths[i], caps[i])) for i, u in enumerate(utts))
    assert traces["run"] == traces[driver]


def test_pump_is_a_no_op_when_idle(P):
    eng, b = make(P, 4, {1: 3})
    assert b.pump(1) == 0 and eng.trace == []
    u = b.add_tokens(0, [1], 10, 3, rng_stream=1)
    assert b.status(u) == ("queued", 0)
    pump_all(b, 1)
    n = len(eng.trace)
    assert b.pump(5) == 0 and len(eng.trace) == n and b.status(u) == ("done", 3)


def test_pump_keeps_the_pipeline_full_between_calls(P):
    eng, b = make(P, 4, {1: 50, 2: 50})
    b.add_tokens(0, [1], 100, 3, rng_stream=1); b.add_tokens(0, [1], 100, 3, rng_stream=2)
    for _ in range(10):
        assert b.pump(1) == 2
        assert len(eng.queue) == 2                                   # depth steps in flight while the caller works
    pump_all(b, 3)
    assert eng.queue == []                                           # the last job finished: drained


# ---- online admission ---------------------------------------------------------------------------------------------------------------------

def test_waves_between_pumps(P):
    rng = np.random.default_rng(3)
    n_slots, refill_every, depth = 16, 4, 2
    lengths, caps = {}, {}
    eng, b = make(P, n_slots, lengths, refill_min=4, refill_every=refill_every, range_quantum=8)
    utts, arrival, first_ready, stream = {}, {}, {}, 0
    for wave in range(12):
        free_at_arrival = n_slots - sum(b.status(u)[0] in ("queued", "running") for u in utts)
        size = int(rng.integers(1, 7))
        for _ in range(size):
            stream += 1
            lengths[stream] = int(rng.integers(1, 40)); caps[stream] = int(rng.integers(1, 50))
            u = b.add_tokens(0, [1, 2], caps[stream], 3, rng_stream=stream)
            utts[u] = stream; arrival[u] = (eng.collects, free_at_arrival >= size)
        for _ in range(int(rng.integers(1, 12))):
            if not b.pump(1):
                break
            for u in utts:
                if u not in first_ready and b.status(u)[1] > 0:
                    first_ready[u] = eng.collects
    pump_all(b, 5)
    for u, s in utts.items():
        want = min(lengths[s], caps[s])
        assert b.frames(u) == want
        assert np.array_equal(b.read(u)[:, 0], expected(s, want))    # every sentence completes with its own frames, in order
        c0, slot_free = arrival[u]
        if slot_free and u in first_ready:
            assert first_ready[u] - c0 <= refill_every + depth + 1, (u, c0, first_ready[u])
    assert sum(1 for u in utts if arrival[u][1] and u in first_ready) >= 10
    begins = [c for c in eng.trace if c[0] == "begin"]
    order = [stream for c in begins for _, stream, _ in c[1]]
    assert sorted(order) == sorted(utts.values())


def test_admission_is_fifo_across_arrivals_and_lpt_within_one(P):
    eng, b = make(P, 1, {1: 2, 2: 2, 3: 2, 4: 2}, refill_min=1, refill_every=1)
    b.add_tokens(0, [1], 10, 3, rng_stream=1)
    b.pump(1)
    b.add_tokens(0, [1], 5, 3, rng_stream=2); b.add_tokens(0, [1], 40, 3, rng_stream=3)    # second wave: longest first
    b.pump(1)
    b.add_tokens(0, [1], 90, 3, rng_stream=4)                                              # later arrival waits behind both
    pump_all(b, 1)
    order = [c[1][0][1] for c in eng.trace if c[0] == "begin"]
    assert order == [1, 3, 2, 4]


# ---- in-order delivery ----------------------------------------------------------------------------------------------------------------------

def _two_sentence_utterance(P, pop):
    # sentence 1 (stream 1) runs 30 frames, sentence 2 (stream 2) only 5: both start together, the second finishes first
    eng, b = make(P, 4, {1: 30, 2: 5, 3: 12}, refill_min=1)
    u = b.add_tokens(0, [1], 30, 3, rng_stream=1)
    b.add_tokens(0, [2], 5, 3, rng_stream=2, utt=u)
    b.add_tokens(0, [3], 12, 3, rng_stream=3)
    pops, seen_running_ready = [], False
    while b.pump(1):
        state, ready = b.status(u)
        if pop:
            got = b.pop(u)
            assert len(got) == ready
            seen_running_ready |= len(got) > 0 and state == "running"      # frames are handed out while their sentence runs
            pops.append(got)
    return eng, b, u, pops, seen_running_ready


def test_pop_delivers_sentences_in_order(P):
    eng, b, u, pops, seen_running_ready = _two_sentence_utterance(P, pop=True)
    begins = [c for c in eng.trace if c[0] == "begin"]
    assert len(begins) == 1 and {s for _, s, _ in begins[0][1]} == {1, 2, 3}               # one sentence start, both sentences side by side
    got = np.concatenate(pops)
    # sentence 2 was done long before sentence 1, yet its frames come after all of sentence 1's, nothing missing or repeated
    assert np.array_equal(got[:, 0], np.concatenate([expected(1, 30), expected(2, 5)]))
    assert seen_running_ready
    assert b.status(u) == ("done", 0) and b.pop(u).shape == (0, FRAME) and b.frames(u) == 35
    _, b2, u2, _, _ = _two_sentence_utterance(P, pop=False)
    assert np.array_equal(b2.read(u2), got)                                                # same audio as read() of a no-pop run


def test_popped_sentences_are_released(P):
    eng, b = make(P, 2, {1: 6, 2: 20})
    u = b.add_tokens(0, [1], 6, 3, rng_stream=1)
    b.add_tokens(0, [1], 20, 3, rng_stream=2, utt=u)
    popped = []
    while b.status(u)[1] < 6:
        b.pump(1)
    popped.append(b.pop(u))
    assert np.array_equal(popped[0][:6, 0], expected(1, 6))
    # sentence 1 is done and handed out: read() (the frames not popped yet) holds only sentence 2's frames from here on
    rest = b.read(u)
    assert (rest[:, 0] >= 2000).all() and b.frames(u) == len(popped[0]) + len(rest)
    pump_all(b, 1)
    popped.append(b.pop(u))
    assert b.status(u) == ("done", 0) and b.read(u).shape == (0, FRAME) and b.frames(u) == 26
    assert np.array_equal(np.concatenate(popped)[:, 0], np.concatenate([expected(1, 6), expected(2, 20)]))


def test_keep_pcm_off_counts_without_audio(P):
    eng, b = make(P, 2, {1: 7}, keep_pcm=0)
    u = b.add_tokens(0, [1], 10, 3, rng_stream=1)
    pump_all(b, 1)
    assert b.frames(u) == 7 and b.status(u) == ("done", 0) and b.pop(u).shape == (0, FRAME)


# ---- cancel ------------------------------------------------------------------------------------------------------------------------------

def _other_frames(b, utts, skip):
    return {u: (b.frames(u), b.read(u).tobytes()) for u in utts if u != skip}


def test_cancel_queued(P):
    lengths = {1: 20, 2: 9, 3: 8}
    eng, b = make(P, 1, lengths)
    utts = [b.add_tokens(0, [1], 50 - i, 3, rng_stream=i + 1) for i in range(3)]
    b.pump(1)
    assert b.status(utts[2])[0] == "queued"
    b.cancel(utts[2])
    assert b.status(utts[2]) == ("cancelled", 0)
    pump_all(b, 1)
    started = [s for c in eng.trace if c[0] == "begin" for _, s, _ in c[1]]
    assert started == [1, 2] and b.frames(utts[2]) == 0
    assert [b.frames(u) for u in utts[:2]] == [20, 9] and not any(c[0] == "end" for c in eng.trace)
    assert b.stats()["sentences"] == 2


def _reference_run(P, n_slots, lengths, caps, **cfg):
    eng, b = make(P, n_slots, lengths, **cfg)
    utts = [b.add_tokens(0, [1], caps[i], 3, rng_stream=i + 1) for i in range(len(caps))]
    b.run()
    return b, utts


def test_cancel_running_with_empty_queue(P):
    lengths, caps = {1: 40, 2: 30, 3: 25}, [60, 60, 60]
    ref, ref_utts = _reference_run(P, 4, lengths, caps)
    eng, b = make(P, 4, lengths, cancelled=(2,))
    utts = [b.add_tokens(0, [1], caps[i], 3, rng_stream=i + 1) for i in range(3)]
    for _ in range(6):
        b.pump(1)
    slot = [c for c in eng.trace if c[0] == "begin"][0][1]
    slot = [s for s, stream, _ in slot if stream == 2][0]
    assert b.status(utts[1])[0] == "running"
    n_before = b.frames(utts[1])
    mark = len(eng.trace)
    b.cancel(utts[1])
    assert b.status(utts[1]) == ("cancelled", 0) and b.read(utts[1]).shape == (0, FRAME)   # undelivered audio of a cancelled utterance is freed
    pump_all(b, 1)
    after = eng.trace[mark:]
    ends = [i for i, c in enumerate(after) if c[0] == "end"]
    first_submit = next(i for i, c in enumerate(after) if c[0] == "submit")
    assert len(ends) == 1 and after[ends[0]] == ("end", (slot,)) and ends[0] < first_submit
    assert b.frames(utts[1]) == n_before and b.status(utts[1]) == ("cancelled", 0)
    assert _other_frames(b, utts, utts[1]) == _other_frames(ref, ref_utts, ref_utts[1])
    assert b.stats()["frames"] == ref.stats()["frames"] - (30 - n_before)


def test_cancel_running_with_queued_work_refills_the_slot(P):
    lengths, caps = {1: 40, 2: 30, 3: 25, 4: 10}, [60, 59, 58, 57]
    ref, ref_utts = _reference_run(P, 2, lengths, caps, refill_min=1, refill_every=1)
    eng, b = make(P, 2, lengths, cancelled=(2,), refill_min=1, refill_every=1)
    utts = [b.add_tokens(0, [1], caps[i], 3, rng_stream=i + 1) for i in range(4)]
    for _ in range(5):
        b.pump(1)
    assert b.status(utts[1])[0] == "running" and b.status(utts[2])[0] == "queued"
    n_before = b.frames(utts[1])
    mark = len(eng.trace)
    b.cancel(utts[1])
    pump_all(b, 1)
    after = eng.trace[mark:]
    first_submit = next(i for i, c in enumerate(after) if c[0] == "submit")
    first_begin = next(i for i, c in enumerate(after) if c[0] == "begin")
    assert first_begin < first_submit and after[first_begin][1][0][1] == 3                 # the freed slot is refilled right away ...
    assert not any(c[0] == "end" for c in after)                                            # ... so it needs no end()
    assert b.frames(utts[1]) == n_before
    assert _other_frames(b, utts, utts[1]) == _other_frames(ref, ref_utts, ref_utts[1])    # in-flight frames of the cancelled sentence went nowhere


def test_cancel_without_end_op_only_drops_on_the_host(P):
    lengths = {1: 30, 2: 30}
    eng, b = make(P, 2, lengths, with_end=False)
    u1, u2 = b.add_tokens(0, [1], 40, 3, rng_stream=1), b.add_tokens(0, [1], 40, 3, rng_stream=2)
    for _ in range(4):
        b.pump(1)
    n = b.frames(u2)
    b.cancel(u2)
    pump_all(b, 1)
    assert b.frames(u2) == n and b.frames(u1) == 30 and not any(c[0] == "end" for c in eng.trace)


def test_cancel_done_utterance_is_a_no_op(P):
    eng, b = make(P, 2, {1: 3})
    u = b.add_tokens(0, [1], 10, 3, rng_stream=1)
    pump_all(b, 1)
    b.cancel(u)
    assert b.status(u) == ("done", 3) and b.read(u).shape == (3, FRAME)


# ---- lifetime and errors ------------------------------------------------------------------------------------------------------------------

def test_destroy_collects_steps_in_flight(P):
    eng, b = make(P, 2, {1: 50})
    b.add_tokens(0, [1], 60, 3, rng_stream=1)
    b.pump(1)
    assert len(eng.queue) == 2
    del b
    assert eng.queue == [] and eng.trace[-2:] == [("collect",), ("collect",)]


def test_bad_arguments(P):
    L = P.lib()
    eng, b = make(P, 2, {1: 3})
    u = b.add_tokens(0, [1], 10, 3, rng_stream=1)
    buf = np.zeros((4, FRAME), np.float32)
    fp = buf.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    ready = ctypes.c_int()
    for bad in (-1, u + 1):
        assert L.ptts_c_batch_pop(b.h, bad, fp, 4) == B200_EINVAL
        assert L.ptts_c_batch_cancel(b.h, bad) == B200_EINVAL
        assert L.ptts_c_batch_status(b.h, bad, ctypes.byref(ready)) == B200_EINVAL
        assert L.ptts_c_batch_frames(b.h, bad) == B200_EINVAL
        assert L.ptts_c_batch_read(b.h, bad, fp, 4) == B200_EINVAL
        ids = np.zeros(1, np.int32)
        assert L.ptts_c_batch_append_tokens(b.h, bad, 0, ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), 1, 5, 3, 0.7, 0) == B200_EINVAL
    assert L.ptts_c_batch_pop(b.h, u, None, 4) == B200_EINVAL
    assert L.ptts_c_batch_pop(None, u, fp, 4) == B200_EINVAL
    assert L.ptts_c_batch_cancel(None, u) == B200_EINVAL
    assert L.ptts_c_batch_status(None, u, ctypes.byref(ready)) == B200_EINVAL
    assert L.ptts_c_batch_pump(None, 1) == B200_EINVAL
    assert L.ptts_c_batch_pump(b.h, 0) == B200_EINVAL
    assert L.ptts_c_batch_status(b.h, u, None) == 0                                        # ready_frames is optional
    b.cancel(u)
    ids = np.zeros(1, np.int32)
    assert L.ptts_c_batch_append_tokens(b.h, u, 0, ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), 1, 5, 3, 0.7, 0) == B200_EINVAL
    cbs = (P.BATCH_BEGIN_FN(eng.begin), P.BATCH_SUBMIT_FN(eng.submit), P.BATCH_COLLECT_FN(eng.collect), P.BATCH_END_FN())
    assert not L.ptts_c_batch_create_with_ops_ex(None, P.BATCH_BEGIN_FN(), *cbs[1:], 2, FRAME)
    assert not L.ptts_c_batch_create_with_ops_ex(None, *cbs, 0, FRAME)
    slots = np.zeros(1, np.int32)
    assert L.b200_end_sentences(None, 1, slots.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))) == B200_EINVAL
