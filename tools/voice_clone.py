"""Voice-cloning measurements on one GPU; writes one JSON document (stdout, and --out if given).

(a) latency: for 1 / 5 / 10 / 30 s prompts, the device time (CUDA events on the engine stream) of the encode alone and of encode + prefill
    (b200_voice_create_from_audio), the host wall time to a usable voice id (the call plus a synchronise), and the kernels launched;
    medians over --reps runs after a warm-up of every size.
(b) flops: the multiply-adds of each encoder stage, computed from the shapes, over the measured encode time.
(c) memory: device memory the encoder's scratch takes for a 30 s prompt (cudaMemGetInfo around the first clone of that size, after a
    1 s clone has allocated everything else the path needs).
(d) cost to a running batch: frames/s of a 256-slot ragged online batch driven by pump(1), with one 10 s clone
    (b200_voice_create_from_audio) every N pumps against none.
(e) the float64 torch restatement's CPU time (tests/encoder_ref.py) for 1 and 10 s, as context.

With --rates, recordings at other rates than 24 kHz instead (profiles/voice_clone_rates_b200.json):
(f) the device resampler alone (resample_kernel, from torch.profiler's CUDA kernel records) for 10 / 30 s at 16 / 44.1 / 48 / 96 kHz,
    medians after a warm-up, and the bytes it moves (input read + table + 24 kHz output written) over that time;
(g) encode + prefill device time and wall time to a voice id for 10 s at 24 / 44.1 / 48 kHz, as in (a);
(h) as (d): a 10 s 24 kHz and a 10 s 44.1 kHz clone every 50 pumps against none, in alternating rounds (medians).

    python tools/voice_clone.py --out profiles/voice_clone_b200.json
    python tools/voice_clone.py --rates --out profiles/voice_clone_rates_b200.json
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
for p in (REPO, os.path.join(REPO, "tools"), os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SR = 24000


def stage_gflop(seconds: float) -> dict:
    """2 x multiply-adds per stage for a prompt of `seconds` (T = 12.5 rows per second)."""
    T = int(np.ceil(seconds * 12.5))
    L0 = 1920 * T; L1, L2, L3 = L0 // 4, L0 // 20, L0 // 120
    conv = lambda L, co, ci, k: 2.0 * L * co * ci * k
    seanet = (conv(L0, 64, 1, 7) + conv(L0, 32, 64, 3) + conv(L0, 64, 32, 1) + conv(L1, 128, 64, 8) + conv(L1, 64, 128, 3) + conv(L1, 128, 64, 1)
              + conv(L2, 256, 128, 10) + conv(L2, 128, 256, 3) + conv(L2, 256, 128, 1) + conv(L3, 512, 256, 12) + conv(L3, 512, 512, 3))
    lin = 2.0 * L3 * 512 * (1536 + 512 + 2048 + 2048)
    att = 2.0 * 2 * L3 * 8 * 64 * 250                 # QK^T and PV over (at most) 250 keys
    tr = 2 * (lin + att)
    ds = conv(T, 512, 512, 32) + 2.0 * T * 1024 * 512
    return {"seanet": seanet / 1e9, "transformer": tr / 1e9, "downsample_proj": ds / 1e9, "total": (seanet + tr + ds) / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--batch-steps", type=int, default=600)
    ap.add_argument("--clone-every", default="50,150")
    ap.add_argument("--out", default=None)
    ap.add_argument("--rates", action="store_true", help="measure recordings at other sample rates (f, g, h)")
    ap.add_argument("--rounds", type=int, default=3, help="--rates: alternating rounds of the batch-cost runs")
    a = ap.parse_args()
    if a.rates:
        return emit(measure_rates(a), a.out)

    import torch
    import ptts_b200 as P
    from make_assets import default_model_dir
    from online_batch import gpu_info
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"gpu_info": gpu_info(0)}
    md = default_model_dir(eos_mode="never", encoder=True)
    L = P.lib()
    rng = np.random.default_rng(0)
    secs = [1, 5, 10, 30]
    pcm = {s: (0.3 * rng.standard_normal(s * SR)).astype(np.float32) for s in secs}

    # (c) memory first, on a fresh engine
    c = P.Context(md, max_slots=1, max_voices=4, kv_capacity=1024)
    c.engine.embed_audio(pcm[1])
    free0 = torch.cuda.mem_get_info()[0]
    c.engine.embed_audio(pcm[30])
    res["scratch_bytes_30s"] = int(free0 - torch.cuda.mem_get_info()[0])
    res["scratch_mb_per_s"] = res["scratch_bytes_30s"] / 30 / 1e6
    c.close()

    # (a) + (b) latency
    c = P.Context(md, max_slots=1, max_voices=4 + len(secs) * (a.reps + 1), kv_capacity=1024)
    eng = c.engine
    st = torch.cuda.ExternalStream(eng.stream_handle())
    fp = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    for s in secs:                                    # warm-up: scratch at its largest size, tensor maps encoded, modules loaded
        eng.embed_audio(pcm[s]); eng.voice_from_audio(pcm[s]); eng.sync()
    lat = {}
    for s in secs:
        x = pcm[s]
        enc_ms, all_ms, wall_ms, launches = [], [], [], []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            eng.sync()
            e0.record(st); l0 = eng.launch_count()
            assert L.b200_voice_embed_audio(eng.h, fp(x), len(x), None) > 0
            e1.record(st); l1 = eng.launch_count()
            e1.synchronize(); enc_ms.append(e0.elapsed_time(e1))
            eng.sync()
            t0 = time.perf_counter(); e0.record(st)
            eng.voice_from_audio(x)
            e1.record(st); eng.sync(); wall_ms.append((time.perf_counter() - t0) * 1e3)
            all_ms.append(e0.elapsed_time(e1)); launches.append((l1 - l0, eng.launch_count() - l1))
        g = stage_gflop(s)
        med = lambda v: float(np.median(v))
        lat[f"{s}s"] = {"T": int(np.ceil(s * 12.5)), "encode_device_ms": med(enc_ms), "encode_prefill_device_ms": med(all_ms),
                        "prefill_device_ms": med(all_ms) - med(enc_ms), "wall_ms_to_voice_id": med(wall_ms),
                        "launches_encode": launches[0][0], "launches_encode_prefill": launches[0][1],
                        "gflop": g, "encode_tflops": g["total"] / med(enc_ms), "encode_ms_spread": [min(enc_ms), max(enc_ms)]}
    res["latency"] = lat
    c.close()

    # (d) cost to a running 256-slot batch
    costs = {}
    for every in [0] + [int(v) for v in a.clone_every.split(",")]:
        costs["none" if not every else f"every_{every}"] = batch_fps(P, md, every, a.batch_steps, lambda e: e.voice_from_audio(pcm[10]))
    res["batch_cost"] = costs

    # (e) CPU restatement
    from encoder_ref import EncoderRef
    from make_assets import read_safetensors
    ref = EncoderRef(read_safetensors(md + "tts_b6369a24.safetensors"), device="cpu")
    cpu = {}
    for s in (1, 10):
        t0 = time.perf_counter(); ref.embed(pcm[s]); cpu[f"{s}s"] = (time.perf_counter() - t0) * 1e3
    res["cpu_restatement_ms"] = {"torch_threads": torch.get_num_threads(), **cpu}

    emit(res, a.out)


def emit(res, out):
    txt = json.dumps(res, indent=1)
    print(txt)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        open(out, "w").write(txt + "\n")


def batch_fps(P, md, every, steps, clone):
    """frames/s of a 256-slot ragged online batch driven by pump(1), calling clone() every `every` pumps (0: never)."""
    from test_gpu_batch import TEXTS
    words = " ".join(TEXTS).split()
    c = P.Context(md, max_slots=256, max_voices=2 + (steps // every if every else 0), kv_capacity=1024)
    P.set_seed(1)
    b = P.Batch(c)
    r = np.random.default_rng(2)
    for i in range(1024):
        n = int(r.integers(3, 30))
        b.add("cosette", " ".join(words[(7 * i + j) % len(words)] for j in range(n)) + ".", temp=0.7)
    for _ in range(20):
        b.pump(1)
    clones, frames, t0 = 0, 0, time.perf_counter()
    for step in range(steps):
        if every and step % every == every - 1:
            clone(c.engine); clones += 1
        frames += b.pump(1)
    dt = time.perf_counter() - t0
    del b
    c.close()
    return {"frames_per_s": frames / dt, "frames": frames, "clones": clones, "seconds": dt}


def measure_rates(a):
    import torch
    import ptts_b200 as P
    import resample_ref as R
    from make_assets import default_model_dir
    from online_batch import gpu_info
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"gpu_info": gpu_info(0)}
    md = default_model_dir(eos_mode="never", encoder=True)
    L = P.lib()
    fp = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    med = lambda v: float(np.median(v))
    rng = np.random.default_rng(0)
    noise = lambda n: (0.3 * rng.standard_normal(n)).astype(np.float32)

    # (f) the resampler alone. Each clone of a rate reuses its table (built by the warm-up), so resample_kernel is the only added kernel.
    c = P.Context(md, max_slots=1, max_voices=2, kv_capacity=1024)
    eng = c.engine
    rs = {}
    for sr in (16000, 44100, 48000, 96000):
        for s in (10, 30):
            x = noise(s * sr)
            for _ in range(3):
                assert L.b200_voice_embed_audio_rate(eng.h, fp(x), len(x), sr, None) > 0
            eng.sync()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(a.reps):
                    L.b200_voice_embed_audio_rate(eng.h, fp(x), len(x), sr, None)
                eng.sync()
            us = [e.time_range.elapsed_us() for e in prof.events() if "resample_kernel(" in e.name and "table" not in e.name]
            assert len(us) == a.reps, [e.name for e in prof.events()][:20]
            n24 = R.out_len(len(x), sr)
            p = R.plan(sr)
            nbytes = 4 * (len(x) + p["m"] * p["W"] + 1920 * -(-n24 // 1920))
            rs[f"{sr}Hz_{s}s"] = {"n": len(x), "n24": n24, "band": p["W"], "phases": p["m"], "kernel_us": med(us),
                                  "kernel_us_spread": [min(us), max(us)], "bytes": nbytes, "GB_per_s": nbytes / med(us) / 1e3}
    res["resampler"] = rs
    c.close()

    # (g) encode + prefill, 10 s
    c = P.Context(md, max_slots=1, max_voices=4 + 3 * (a.reps + 1), kv_capacity=1024)
    eng = c.engine
    st = torch.cuda.ExternalStream(eng.stream_handle())
    lat = {}
    for sr in (24000, 44100, 48000):
        x = noise(10 * sr)
        eng.embed_audio(x, sr); eng.voice_from_audio(x, sr); eng.sync()
        enc_ms, all_ms, wall_ms = [], [], []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            eng.sync()
            e0.record(st)
            assert L.b200_voice_embed_audio_rate(eng.h, fp(x), len(x), sr, None) > 0
            e1.record(st); e1.synchronize(); enc_ms.append(e0.elapsed_time(e1))
            eng.sync()
            t0 = time.perf_counter(); e0.record(st)
            eng.voice_from_audio(x, sr)
            e1.record(st); eng.sync(); wall_ms.append((time.perf_counter() - t0) * 1e3)
            all_ms.append(e0.elapsed_time(e1))
        lat[f"{sr}Hz_10s"] = {"encode_device_ms": med(enc_ms), "encode_prefill_device_ms": med(all_ms), "wall_ms_to_voice_id": med(wall_ms),
                              "encode_ms_spread": [min(enc_ms), max(enc_ms)]}
    res["latency_10s"] = lat
    c.close()

    # (h) cost to a running 256-slot batch
    # (h) cost to a running 256-slot batch: no clones, a 10 s 24 kHz clone and a 10 s 44.1 kHz clone every 50 pumps, in alternating rounds
    x24, x44 = noise(10 * 24000), noise(10 * 44100)
    runs = {"none": (0, None), "every_50_24k": (50, lambda e: e.voice_from_audio(x24, 24000)),
            "every_50_44k": (50, lambda e: e.voice_from_audio(x44, 44100))}
    fps = {k: [] for k in runs}
    for _ in range(a.rounds):
        for k, (every, fn) in runs.items():
            fps[k].append(batch_fps(P, md, every, a.batch_steps, fn)["frames_per_s"])
    res["batch_cost"] = {"batch_steps": a.batch_steps, "rounds": a.rounds,
                         **{k: {"frames_per_s_median": med(v), "frames_per_s": v} for k, v in fps.items()}}
    return res


if __name__ == "__main__":
    main()
