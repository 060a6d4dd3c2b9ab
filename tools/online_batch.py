"""Online continuous batching on one GPU: prints one JSON line per run.

(a) --mode ragged: the configs[4] ragged job of bench.py (2048 sentences of 3-45 words, EOS-firing checkpoint, 8 voices, 256 slots), run
    once by run() counting frames only (keep_pcm=0), once by run() keeping the whole job's audio in RAM (keep_pcm=1), and once driven by
    pump(1) with every ready frame popped after each pump into a reusable buffer (what a server streaming the audio out would do). The
    three runs take the same scheduling decisions, so their frame counts agree.
(b) --mode poisson: utterances (ragged sentences) arrive at `rate` per engine step (Poisson); after each pump(1) the new arrivals are
    added and every ready frame is popped. Reports frames/s, the idle-slot fraction, and the time to first frame per utterance (arrival
    to its first pop) in engine steps and in ms. The ms figures come from a host clock around pump calls, each of which ends in the
    collect of a finished step (a device synchronise).

Every line carries the GPU name and power limit read in the same run.

    python tools/online_batch.py --mode ragged
    python tools/online_batch.py --mode poisson --rates 0.5,1,1.5 --steps 3000
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def gpu_info(device):
    out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, sm = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": sm}


class Popper:
    """Pops every ready frame of the utterances that have started, into one reusable buffer. Utterances are polled from the moment their
    status leaves 'queued' until they are done and fully popped, so a step costs calls for the running utterances only."""

    def __init__(self, P, b, max_frames=1 << 12):
        self.L, self.b = P.lib(), b
        self.buf = np.zeros((max_frames, P.FRAME), np.float32)
        self.ptr = self.buf.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        self.waiting, self.live = [], []
        self.first_pop = {}                      # utt -> (engine steps, host seconds) of its first non-empty pop
        self.frames = 0

    def arrive(self, utts, caps):
        # the scheduler starts the utterances of one arrival longest cap first (stable), so poll them in that order
        self.waiting += [u for _, u in sorted(zip(caps, utts), key=lambda x: -x[0])]

    def poll(self, steps, now, scan=64):
        L, h = self.L, self.b.h
        keep, seen = [], 0
        for u in self.waiting:                    # admission order is FIFO across arrivals: the front of the list starts first
            if seen < scan and L.ptts_c_batch_status(h, u, None) != 0:
                self.live.append(u)
            else:
                keep.append(u); seen += 1
        self.waiting = keep
        still = []
        for u in self.live:
            n = L.ptts_c_batch_pop(h, u, self.ptr, len(self.buf))
            if n > 0:
                self.frames += n
                self.first_pop.setdefault(u, (steps, now))
            if n > 0 or L.ptts_c_batch_status(h, u, None) < 2:
                still.append(u)
        self.live = still


def make_ctx(P, args):
    from make_assets import default_model_dir
    d = default_model_dir(eos_mode="late")
    return P.Context(d, device=args.device, max_slots=args.slots, max_voices=8, kv_capacity=1024)


def new_batch(P, ctx, args, keep_pcm=1):
    b = P.Batch(ctx, args.slots)
    b.configure(refill_min=args.refill_min, refill_every=args.refill_every, range_quantum=32, keep_pcm=keep_pcm)
    return b


def ragged(P, ctx, args, info):
    from bench import ragged_sentence
    from make_assets import VOICES
    sents = [ragged_sentence(i) for i in range(args.sentences)]
    caps = [int((w + 2) * 12.5) for _, w in sents]

    def one(mode):
        P.set_seed(4321)
        b = new_batch(P, ctx, args, keep_pcm=0 if mode == "run_count_only" else 1)
        utts = [b.add(VOICES[i % 8], s, 0.7) for i, (s, _) in enumerate(sents)]
        t0 = time.perf_counter()
        if mode == "pump_pop":
            pop = Popper(P, b)
            pop.arrive(utts, caps)
            while b.pump(1):
                pop.poll(0, 0.0)
            pop.poll(0, 0.0)
            frames = pop.frames
        else:
            frames = b.run()
        ctx.engine.sync()
        dt = time.perf_counter() - t0
        st = b.stats()
        return {"mode": mode, "frames": int(frames), "seconds": round(dt, 4), "frames_per_s": round(frames / dt, 1), "steps": st["steps"],
                "idle_slot_fraction": round(st["idle_slot_fraction"], 4), "host_ms": {k: round(st[k], 1) for k in ("begin_ms", "submit_ms", "collect_ms")}}

    P.set_seed(4321)                                         # warm-up: voice prefills, graph captures for the stepped ranges
    b = new_batch(P, ctx, args, keep_pcm=0)
    for i in range(min(len(sents), 2 * args.slots)):
        b.add(VOICES[i % 8], sents[i][0], 0.7)
    b.run()
    del b
    for rep in range(args.repeats):
        for mode in ("run_count_only", "run_keep_pcm", "pump_pop"):
            r = one(mode)
            print(json.dumps({"workload": f"(a) ragged job: {args.sentences} sentences (3-45 words, EOS-firing checkpoint, 8 voices), {args.slots} slots",
                              "repeat": rep, **r, **info}), flush=True)


def poisson(P, ctx, args, info, rate):
    from bench import ragged_sentence
    from make_assets import VOICES
    rng = np.random.default_rng(args.seed)
    P.set_seed(4321)
    b = new_batch(P, ctx, args, keep_pcm=1)
    pop = Popper(P, b)
    arrived_at, k, steps, n_pumps = {}, 0, 0, 0
    t0 = time.perf_counter()
    while n_pumps < args.steps:
        now = time.perf_counter() - t0
        new, caps = [], []
        for _ in range(int(rng.poisson(rate))):
            text, words = ragged_sentence(100000 + k); k += 1
            u = b.add(VOICES[k % 8], text, 0.7)
            arrived_at[u] = (steps, now); new.append(u); caps.append(int((words + 2) * 12.5))
        pop.arrive(new, caps)
        b.pump(1); n_pumps += 1
        steps = b.stats()["steps"]
        pop.poll(steps, time.perf_counter() - t0)
    dt = time.perf_counter() - t0
    st = b.stats()
    frames = st["frames"]
    ttff_steps = np.array([pop.first_pop[u][0] - arrived_at[u][0] for u in arrived_at if u in pop.first_pop], np.float64)
    ttff_ms = np.array([(pop.first_pop[u][1] - arrived_at[u][1]) * 1e3 for u in arrived_at if u in pop.first_pop], np.float64)
    pct = lambda a, q: round(float(np.percentile(a, q)), 2) if len(a) else None
    print(json.dumps({"workload": f"(b) Poisson arrivals of ragged sentences (3-45 words, EOS-firing checkpoint, 8 voices), {args.slots} slots, "
                                  f"pump(1) then pop everything ready, {args.steps} pumps",
                      "arrivals_per_step": rate, "utterances_arrived": len(arrived_at), "utterances_with_audio": len(ttff_steps),
                      "frames": int(frames), "seconds": round(dt, 3), "frames_per_s": round(frames / dt, 1), "steps": st["steps"],
                      "idle_slot_fraction": round(st["idle_slot_fraction"], 4),
                      "ttff_steps": {"p50": pct(ttff_steps, 50), "p99": pct(ttff_steps, 99)},
                      "ttff_ms": {"p50": pct(ttff_ms, 50), "p99": pct(ttff_ms, 99)}, **info}), flush=True)
    while b.pump(8):
        pass
    del b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["ragged", "poisson", "all"], default="all")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--slots", type=int, default=256)
    ap.add_argument("--sentences", type=int, default=2048)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--refill-min", type=int, default=16)
    ap.add_argument("--refill-every", type=int, default=8)
    ap.add_argument("--rates", default="0.5,1.0,1.5", help="arrivals per engine step, comma separated")
    ap.add_argument("--steps", type=int, default=3000, help="pumps per Poisson run")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    import ptts_b200 as P
    info = gpu_info(args.device)
    ctx = make_ctx(P, args)
    if args.mode in ("ragged", "all"):
        ragged(P, ctx, args, info)
    if args.mode in ("poisson", "all"):
        for r in args.rates.split(","):
            poisson(P, ctx, args, info, float(r))
    ctx.close()


if __name__ == "__main__":
    main()
