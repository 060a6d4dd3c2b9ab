"""Streamed text into an online batch on one GPU (ptts_c_batch_open / send / close): prints one JSON line per run.

Workload: a 256-slot batch kept busy by the ragged job (bench.py's ragged sentences, 3-45 words, 8 voices), topped up after every pump so
that `--load` of its sentences are queued or running. On top of it `--streams` utterances of `--sentences` ragged sentences each are written
by a simulated LLM at `--cps` characters per second (40 tokens/s is about 160 chars/s); utterance i starts `i * --stagger` seconds into the
run. Between two pump(1) calls every utterance gets the characters that have arrived by then.

  --mode stream: the utterance is opened at its start, each chunk is sent as it arrives, it is closed with its last character.
  --mode whole:  the utterance is given to add() whole once its last character has arrived (the caller waits for the whole reply).

Reported per run: batch frames/s over the window from the start to the last streamed utterance done; time to the first audio frame of each
utterance from its start; for --mode stream, the time from the character that completes a sentence (its arrival time at the simulated rate)
to that sentence's first popped frame (p50 / p99), and playback underruns: sentences whose first frame was ready after the previous
sentence's audio would have finished playing in real time from the utterance's first frame.

The checkpoint is the never-EOS one, so that every sentence runs to its cap int((words + 2) * 12.5) and the sentence boundaries inside an
utterance's popped audio are known. The times come from a host clock around pump calls, each of which ends in the collect of a finished step
(a device synchronise). Every line carries the GPU name, power limit and max SM clock read in the same run.

    python tools/stream_text.py --mode stream --mode whole --repeats 2
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

FRAME_RATE = 12.5      # frames per second of audio


def gpu_info(device):
    from online_batch import gpu_info as info
    return info(device)


def split_points(text: bytes):
    """Byte index of the character that completes each sentence (the reference's splitter: the first character after the terminator; the
    last character of the text for the tail emitted at close), the sentences, and how many of them a send emits (the rest: close)."""
    import oracle
    sp, at = oracle.StrProcessor(), []
    for i in range(len(text)):
        n = len(sp.sentences)
        sp.ingest(text[i:i + 1])
        at += [i] * (len(sp.sentences) - n)
    n = len(sp.sentences)
    sp.flush()
    at += [len(text) - 1] * (len(sp.sentences) - n)
    return at, list(sp.sentences), n


def run(P, ctx, args, mode, info):
    from bench import ragged_sentence
    from make_assets import VOICES
    import oracle
    L = P.lib()
    P.set_seed(4321)
    b = P.Batch(ctx, args.slots)
    b.configure(refill_min=args.refill_min, refill_every=args.refill_every, range_quantum=32, keep_pcm=1)
    buf = np.zeros((1 << 12, P.FRAME), np.float32)
    ptr = buf.ctypes.data_as(ctypes.POINTER(ctypes.c_float))

    texts = [" ".join(ragged_sentence(200000 + i * args.sentences + k)[0] for k in range(args.sentences)).encode() for i in range(args.streams)]
    plan = [split_points(t) for t in texts]
    caps = [[oracle.max_gen_len_for(s) for s in ss] for _, ss, _ in plan]
    starts = [i * args.stagger for i in range(args.streams)]
    utt = [None] * args.streams
    sent = [0] * args.streams                         # bytes sent
    closed = [False] * args.streams
    popped = [0] * args.streams                       # frames popped
    first_pop = [[None] * len(c) for c in caps]       # host time of each sentence's first popped frame
    done_at = [None] * args.streams

    bg, bg_next = [], 0                               # live background utterances, next ragged sentence

    def top_up():
        nonlocal bg_next
        keep = []
        for u in bg:
            L.ptts_c_batch_pop(b.h, u, ptr, len(buf))
            if L.ptts_c_batch_status(b.h, u, None) < 2:
                keep.append(u)
        bg[:] = keep
        while len(bg) < args.load:
            bg.append(b.add(VOICES[bg_next % 8], ragged_sentence(bg_next)[0], 0.7)); bg_next += 1

    top_up()
    st0 = b.stats()
    t0 = time.perf_counter()
    while not all(d is not None for d in done_at):
        now = time.perf_counter() - t0
        if now > args.timeout:
            raise RuntimeError(f"streamed utterances not done after {args.timeout} s: {sum(d is None for d in done_at)} left")
        for i in range(args.streams):
            if closed[i] or now < starts[i]:
                continue
            upto = min(len(texts[i]), int((now - starts[i]) * args.cps))
            if mode == "stream":
                if utt[i] is None:
                    utt[i] = b.open(VOICES[i % 8], 0.7)
                if upto > sent[i]:
                    n = b.send(utt[i], texts[i][sent[i]:upto])
                    at, _, n_send = plan[i]
                    assert n == sum(sent[i] <= a < upto for a in at[:n_send]), (i, n)
                    sent[i] = upto
                if upto == len(texts[i]):
                    assert b.close(utt[i]) == len(plan[i][1]) - plan[i][2]
                    closed[i] = True
            elif upto == len(texts[i]):
                utt[i] = b.add(VOICES[i % 8], texts[i].decode(), 0.7); closed[i] = True
        b.pump(1)
        now = time.perf_counter() - t0
        for i in range(args.streams):
            if utt[i] is None or done_at[i] is not None:
                continue
            n = L.ptts_c_batch_pop(b.h, utt[i], ptr, len(buf))
            if n > 0:
                # sentence k of the utterance starts at frame sum(caps[:k]) of its audio (never-EOS checkpoint)
                edge = 0
                for k, c in enumerate(caps[i]):
                    if first_pop[i][k] is None and popped[i] <= edge < popped[i] + n:
                        first_pop[i][k] = now
                    edge += c
                popped[i] += n
            if closed[i] and L.ptts_c_batch_status(b.h, utt[i], None) == 2 and popped[i] == sum(caps[i]):
                done_at[i] = now
        top_up()
    window = time.perf_counter() - t0
    st = b.stats()
    frames = st["frames"] - st0["frames"]
    while b.pump(8):
        pass
    del b

    ms = lambda a: np.asarray(a, np.float64) * 1e3
    pct = lambda a, q: round(float(np.percentile(a, q)), 2) if len(a) else None
    ttfa = ms([first_pop[i][0] - starts[i] for i in range(args.streams)])
    out = {"workload": f"{args.slots}-slot batch with {args.load} ragged sentences (3-45 words, never-EOS checkpoint, 8 voices) kept queued or running; "
                       f"{args.streams} utterances of {args.sentences} ragged sentences written at {args.cps} chars/s, one starting every "
                       f"{args.stagger} s; pump(1), then send what arrived and pop every ready frame",
           "mode": mode, "frames": int(frames), "seconds": round(window, 3), "frames_per_s": round(frames / window, 1), "steps": st["steps"] - st0["steps"],
           "idle_slot_fraction": round(1.0 - frames / max(st["slot_steps"] - st0["slot_steps"], 1), 4),
           "utterance_first_audio_ms": {"p50": pct(ttfa, 50), "p99": pct(ttfa, 99), "max": round(float(ttfa.max()), 2)},
           "reply_text_seconds": {"mean": round(float(np.mean([len(t) / args.cps for t in texts])), 2)}}
    if mode == "stream":
        lat, underruns, n_sent = [], 0, 0
        for i in range(args.streams):
            at = plan[i][0]
            t_first = first_pop[i][0]
            played = 0.0
            for k, c in enumerate(caps[i]):
                lat.append(first_pop[i][k] - (starts[i] + (at[k] + 1) / args.cps))
                if k > 0 and first_pop[i][k] > t_first + played:
                    underruns += 1
                played += c / FRAME_RATE
                n_sent += 1
        lat = ms(lat)
        out.update({"sentences": n_sent, "sentence_complete_to_first_frame_ms": {"p50": pct(lat, 50), "p99": pct(lat, 99), "max": round(float(lat.max()), 2)},
                    "playback_underruns": underruns})
    out.update(info)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", action="append", choices=["stream", "whole"])
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--slots", type=int, default=256)
    ap.add_argument("--load", type=int, default=192, help="background ragged sentences kept queued or running")
    ap.add_argument("--streams", type=int, default=32)
    ap.add_argument("--sentences", type=int, default=4, help="sentences per streamed utterance")
    ap.add_argument("--cps", type=float, default=160.0, help="characters per second of the simulated LLM")
    ap.add_argument("--stagger", type=float, default=0.05, help="seconds between the starts of two streamed utterances")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--refill-min", type=int, default=16)
    ap.add_argument("--refill-every", type=int, default=8)
    ap.add_argument("--timeout", type=float, default=300.0, help="seconds before a run is abandoned")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import ptts_b200 as P
    from make_assets import default_model_dir
    info = gpu_info(args.device)
    ctx = P.Context(default_model_dir(eos_mode="never"), device=args.device, max_slots=args.slots, max_voices=8, kv_capacity=1024)
    run(P, ctx, argparse.Namespace(**{**vars(args), "streams": 8, "load": args.slots}), "stream", info)   # warm-up: voices, step graphs
    for rep in range(args.repeats):
        for mode in args.mode or ["stream", "whole"]:
            line = json.dumps({"repeat": rep, **run(P, ctx, args, mode, info)})
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
