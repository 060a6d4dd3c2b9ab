"""CPU: the per-sentence sampling controls (DESIGN.md 4.7) up to the engine boundary. The range checks of b200_sampling_check and of the
batch / stream entry points, the scheduler handing each job's b200_sampling to the sentence-start op unchanged (across refills and
append_tokens) against a mock engine, and the CLI flags."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest


def _check(P, *s):
    sp = P.Sampling(*s)
    return P.lib().b200_sampling_check(ctypes.byref(sp))


def test_default_sampling_and_range_checks(P):
    sp = P.Sampling(7, 7.0, 7.0)
    P.lib().b200_default_sampling(ctypes.byref(sp))
    assert sp.astuple() == (1, 0.0, -4.0)
    for ok in ((1, 0.0, -4.0), (8, 0.0, 0.0), (4, 0.3, -10.0), (2, 1e-6, 3.5)):
        assert _check(P, *ok) == 0, ok
    for bad in ((0, 0.0, -4.0), (9, 0.0, -4.0), (-1, 0.0, -4.0), (1, -0.1, -4.0), (1, math.nan, -4.0), (1, math.inf, -4.0),
                (1, 0.0, math.nan), (1, 0.0, math.inf), (1, 0.0, -math.inf)):
        assert _check(P, *bad) == -1, bad
    assert P.lib().b200_sampling_check(None) == -1


class MockEngine:
    """Every sentence produces `length` frames; records the sampling struct each begin hands over, per RNG stream id."""

    def __init__(self, n_slots, length=3):
        self.n_slots, self.length = n_slots, length
        self.left = [0] * n_slots
        self.seen = {}
        self.inflight = []

    def begin(self, user, n, slots, voices, tokens, tok_off, mg, fae, temp, rng, samp):
        for i in range(n):
            self.left[slots[i]] = min(self.length, mg[i])
            self.seen.setdefault(rng[i], []).append((samp[i].lsd_steps, samp[i].noise_clamp, samp[i].eos_threshold))
        return 0

    def submit(self, user, slot0, n):
        prod = []
        for s in range(slot0, slot0 + n):
            prod.append(1 if self.left[s] > 0 else 0)
            self.left[s] = max(0, self.left[s] - 1)
        self.inflight.append(prod)
        return 0

    def collect(self, user, pcm, produced):
        prod = self.inflight.pop(0)
        for i, p in enumerate(prod):
            produced[i] = p
        return len(prod)


def test_scheduler_passes_each_jobs_sampling_unchanged(P):
    rng = np.random.default_rng(5)
    m = MockEngine(4)
    b = P.Batch(ops=(m.begin, m.submit, m.collect), n_slots=4, frame_size=8, begin_sampling=True)
    b.configure(refill_min=1, refill_every=1, range_quantum=1)
    want = {}
    for k in range(11):                                               # 11 sentences over 4 slots: several refills
        s = (int(rng.integers(1, 9)), float(np.float32(rng.uniform(0, 2))) if k % 3 else 0.0, float(np.float32(rng.uniform(-8, 2))))
        b.add_tokens(0, [1, 2, 3], 5, 1, temp=0.7, rng_stream=100 + k, lsd_steps=s[0], noise_clamp=s[1], eos_threshold=s[2])
        want[100 + k] = s
    u = b.add_tokens(0, [4, 5], 5, 1, rng_stream=200)                  # defaults
    want[200] = (1, 0.0, -4.0)
    b.add_tokens(0, [6], 5, 1, rng_stream=201, utt=u, lsd_steps=3, noise_clamp=0.25, eos_threshold=-2.5)   # append_tokens
    want[201] = (3, 0.25, -2.5)
    assert b.run() == 13 * 3
    assert m.seen == {k: [v] for k, v in want.items()}
    assert b.frames(u) == 6
    for bad in (dict(lsd_steps=0), dict(lsd_steps=9), dict(noise_clamp=-1.0), dict(eos_threshold=math.inf), dict(noise_clamp=math.nan)):
        with pytest.raises(RuntimeError):
            b.add_tokens(0, [1], 5, 1, **bad)
        with pytest.raises(RuntimeError):
            b.add_tokens(0, [1], 5, 1, utt=u, **bad)


def test_scheduler_without_sampling_op_keeps_plain_begin(P):
    calls = []
    m = MockEngine(2)

    def begin(user, n, slots, voices, tokens, tok_off, mg, fae, temp, rng):
        calls.append(n)
        for i in range(n):
            m.left[slots[i]] = min(m.length, mg[i])
        return 0

    b = P.Batch(ops=(begin, m.submit, m.collect), n_slots=2, frame_size=8)
    b.add_tokens(0, [1], 5, 1, lsd_steps=4)
    assert b.run() == 3 and calls == [1]


def test_cli_parses_sampling_flags(P):
    cli = os.path.join(os.path.dirname(P.LIB_PATH), "pocket-tts-b200")
    r = subprocess.run([cli, "--help"], capture_output=True, text=True)
    for flag in ("--lsd-decode-steps", "--noise-clamp", "--eos-threshold"):
        assert flag in r.stdout + r.stderr
    # accepted flags and no text: the usage message, not "unrecognized option"
    r = subprocess.run([cli, "--lsd-decode-steps", "4", "--noise-clamp", "0.5", "--eos-threshold", "-3"], capture_output=True, text=True)
    assert "unrecognized option" not in r.stderr and r.stderr.startswith("usage:")
    for bad in (["--lsd-decode-steps", "9"], ["--lsd-decode-steps", "0"], ["--noise-clamp", "-1"], ["--eos-threshold", "nan"]):
        r = subprocess.run([cli] + bad + ["text"], capture_output=True, text=True)
        assert r.returncode == 1 and "sampling controls out of range" in r.stderr, bad
    r = subprocess.run([cli, "--noise-clamp"], capture_output=True, text=True)
    assert r.returncode == 1 and "requires value" in r.stderr
