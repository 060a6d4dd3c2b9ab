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

    python tools/voice_clone.py --out profiles/voice_clone_b200.json
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
    a = ap.parse_args()

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
    from test_gpu_batch import TEXTS
    words = " ".join(TEXTS).split()
    costs = {}
    for every in [0] + [int(v) for v in a.clone_every.split(",")]:
        c = P.Context(md, max_slots=256, max_voices=2 + (a.batch_steps // every if every else 0), kv_capacity=1024)
        P.set_seed(1)
        b = P.Batch(c)
        r = np.random.default_rng(2)
        for i in range(1024):
            n = int(r.integers(3, 30))
            b.add("cosette", " ".join(words[(7 * i + j) % len(words)] for j in range(n)) + ".", temp=0.7)
        for _ in range(20):
            b.pump(1)
        clones, frames, t0 = 0, 0, time.perf_counter()
        for step in range(a.batch_steps):
            if every and step % every == every - 1:
                c.engine.voice_from_audio(pcm[10]); clones += 1
            frames += b.pump(1)
        dt = time.perf_counter() - t0
        costs["none" if not every else f"every_{every}"] = {"frames_per_s": frames / dt, "frames": frames, "clones": clones, "seconds": dt}
        del b
        c.close()
    res["batch_cost"] = costs

    # (e) CPU restatement
    from encoder_ref import EncoderRef
    from make_assets import read_safetensors
    ref = EncoderRef(read_safetensors(md + "tts_b6369a24.safetensors"), device="cpu")
    cpu = {}
    for s in (1, 10):
        t0 = time.perf_counter(); ref.embed(pcm[s]); cpu[f"{s}s"] = (time.perf_counter() - t0) * 1e3
    res["cpu_restatement_ms"] = {"torch_threads": torch.get_num_threads(), **cpu}

    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(txt + "\n")


if __name__ == "__main__":
    main()
