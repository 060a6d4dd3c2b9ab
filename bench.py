#!/usr/bin/env python3
"""bench.py — audio frames/s of the Pocket-TTS per-frame generation path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch 256] [--kv-len 1500] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: FlowLM step -> EOS rule -> LSD head -> Mimi -> 1920 samples, for every
utterance of the batch (BASELINE.json configs[3]: batch 256, ~40-word paragraphs, KV length ~1.5k; voice prefix padded so the
FlowLM cache holds ~kv_len positions in mid-run). One process per GPU (torchrun for N>1), weights replicated, utterances sharded,
no collective on the hot path; NCCL gathers per-rank counts/timings only. Prints ONE JSON line on rank 0.

  value        device-resident throughput of the default engine (shared voice prefix = cascade attention): K steps enqueued on the
               engine stream, CUDA events, max over ranks
  e2e          same metric through the public C-ABI pair b200_submit/b200_collect with HOST buffers (H2D noise, D2H PCM + flags inside)
  roofline     dominant kernel of that step (the per-utterance KV stream of the FlowLM attention, HBM bound) + the whole step against
               the bytes it must move (unique bytes: prefix once, private rows, weights, Mimi state)
  private_kv   the same workload with the reference's copy_states layout (prefix_share=0: every slot streams a private copy of the
               prefix; round 1's configuration) with ITS roofline (9.9 GB/step KV stream)
  kv_f32       the reference's cache precision (fp32 KV, private copies) with its roofline
  multi_voice  8 voices x 32 slots (prefix sharing per voice group)
  ragged       BASELINE configs[4] as a continuous-batching job: 2048 sentences of 3-45 words per GPU (EOS-firing checkpoint, 8 voices),
               256 slots, finished slots refilled (ptts_c_batch_*), utterances LPT-sharded over ranks; text in, PCM out on the host
  verify       3 slots of the timed context compared with the CPU oracle under injected noise, outside the timed region
  sustained    >= 2 s of back-to-back steps of the primary mode with the clock record
  cpu_baseline the oracle (CPU restatement of the reference's ggml path) on this box's host cores, bounded samples
  --impl reference : the reference arm on the host cores (oracle/_ref when it was built, else the oracle port)
  --dump-outputs DIR : after the timed steps, what their last step computed for the primary mode's utterances (the arrays b200_step
               returns to its caller) as DIR/<name>.npy, so that two builds can be compared output for output (same arguments = same inputs)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
sys.path.insert(0, os.path.join(REPO, "pocket-tts.cpp_b200"))

METRIC = "audio_frames_per_sec"
UNIT = "frames/s"
PARAGRAPH_WORDS = 40
BENCH_SENTENCE = "The quick brown fox jumped over the sleeping dog."     # reference demos/pocket-tts.cpp:231


def synth_paragraph(i: int, n_words: int = PARAGRAPH_WORDS) -> str:
    from make_assets import COMMON_WORDS
    rng = np.random.default_rng(1000 + i)
    ws = [COMMON_WORDS[int(k)] for k in rng.integers(0, len(COMMON_WORDS), n_words)]
    return (" ".join(ws)).capitalize() + "."


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device: int):
        self.device = device; self.rows = []; self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], None, set(), []
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2]); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------------------
# CPU side: the reference arm and the cpu_baseline legs (the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------------------
def _ref_runner():
    """oracle/_ref (the reference's own sources compiled against the ggml shim) when it has been built, else None."""
    try:
        import oracle.ref as R
        return R if R.available() else None
    except Exception:
        return None


def run_reference(args, rank: int, world: int):
    """Reference arm / cpu_baseline: one utterance of the bench workload on all host cores. With oracle/_ref (the reference's own sources
    over the ggml stand-in headers) the paragraph runs through the reference's ptts_stream_send / flush / receive; its FlowLM cache is a
    fixed 1000 rows with no bounds check (src/pocket_tts.cpp:367), so configs[3]'s 1.5k positions cannot be reproduced there: the voice
    prefix is the standard 125 rows (the KV read is ~5 % of the CPU frame cost). Without _ref: the oracle port at the full KV length."""
    if rank != 0:
        return None
    from make_assets import default_model_dir
    cores = os.cpu_count() or 1
    text = synth_paragraph(0)
    sample = args.ref_frames_per_step
    R = _ref_runner()
    if R is not None:
        d = default_model_dir(eos_mode="never")
        r = R.Ref(d, cores)
        s = r.stream("cosette", 0.0)
        s.send(text); s.flush()
        step = lambda: s.receive() is not None
        where = lambda: s.current_end
        kind = "reference"
        what = "reference sources (src/pocket_tts.cpp) over the ggml stand-in headers, voice prefix 125 rows (the reference's cache holds 1000 positions)"
    else:
        import oracle
        oracle.build()
        d = default_model_dir(eos_mode="never", t_voice=args.t_voice, voices=["cosette"])
        o = oracle.Oracle(d, threads=cores)
        s = o.stream("cosette", kv_capacity=args.kv_capacity)
        s.sentence_init(text)
        step = lambda: bool(s.step(None)[0])
        where = lambda: s.current_end
        kind = "port"
        what = "oracle port of the reference's ggml graph"
    for _ in range(args.warmup):
        for _ in range(sample):
            step()
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        for _ in range(sample):
            n += int(step())
    dt = time.perf_counter() - t0
    fps = n / dt
    desc = f"1 utterance (batch 1, {cores} threads; {what}), {sample} frames per step of a {PARAGRAPH_WORDS}-word paragraph at FlowLM KV length ~{where()}, temp 0"
    return {"value": fps, "ms_per_step": dt * 1e3 / args.steps, "cores": cores, "sample": desc, "frames": n, "kind": kind, "kv_len": int(where())}


def cpu_config1(frames: int = 40):
    """BASELINE configs[0] (`pocket-tts --bench`: bench sentence, temp 0, text prefill INSIDE the timed region, reference formula
    frames*1000 / sum(send+receive ms), demos/pocket-tts.cpp:456-520) at the reference's default 4 threads and at nproc, bounded to
    `frames` frames each. Uses oracle/_ref (reference sources over the ggml shim) when built, else the oracle port."""
    import oracle
    from make_assets import default_model_dir
    d = default_model_dir(eos_mode="never")
    out = {"frames_per_run": frames, "sentence": BENCH_SENTENCE}
    R = _ref_runner()
    for label, th in (("threads_4", 4), ("threads_nproc", os.cpu_count() or 1)):
        if R is not None:
            fps = R.bench_sentence_fps(d, BENCH_SENTENCE, threads=th, max_frames=frames)
            out["kind"] = "reference"
        else:
            o = oracle.Oracle(d, threads=th)
            s = o.stream("cosette", kv_capacity=1000)           # stream creation (voice prefill) is outside the reference's timed region
            t0 = time.perf_counter()
            s.sentence_init(BENCH_SENTENCE)
            n = 0
            for _ in range(frames):
                ok, *_ = s.step(None)
                n += int(ok)
            fps = n / (time.perf_counter() - t0)
            out["kind"] = "port"
        out[label] = {"threads": th, "frames_per_s": round(fps, 2)}
    return out


def cpu_baseline_quick(args):
    """~10-20 s of oracle work on rank 0 (N=1 only)."""
    a = argparse.Namespace(**vars(args)); a.steps = 10; a.warmup = 1; a.ref_frames_per_step = 4
    r = run_reference(a, 0, 1)
    out = {"value": round(r["value"], 2), "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
    try:
        out["config1_bench_sentence"] = cpu_config1()
    except Exception as ex:                                      # never lose the bench line over the extra CPU leg
        out["config1_bench_sentence"] = {"error": repr(ex)}
    return out


# ------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------
class Env:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0")); self.world = int(os.environ.get("WORLD_SIZE", "1")); self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.args = args

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def run_mode(env: Env, name: str, share: int, kv_f32: int, n_voices: int = 1, primary: bool = False, verify: bool = False):
    """One engine configuration on the configs[3] workload: device-timed steps (+ e2e, profile, sustained and verify for the primary)."""
    import ptts_b200 as P
    from make_assets import default_model_dir, VOICES
    args, torch = env.args, env.torch
    B = args.batch
    voices = VOICES[:n_voices] if n_voices > 1 else ["cosette"]
    d = default_model_dir(eos_mode="never", t_voice=args.t_voice, voices=voices if n_voices > 1 else ["cosette"])
    ctx = P.Context(d, device=env.local, max_slots=B, max_voices=n_voices, kv_capacity=args.kv_capacity, kv_f32=kv_f32, gemm_path=args.gemm_path, pdl=args.pdl,
                    cuda_graphs=args.cuda_graphs, overlap=args.overlap, prefix_share=share)
    eng = ctx.engine
    streams = [ctx.stream(v, temp=0.7) for v in voices]          # prefill of the (long) voice prefixes
    vid = [streams[(i * n_voices) // B].voice for i in range(B)]  # voice groups of B / n_voices consecutive slots
    texts = [synth_paragraph(env.rank * B + i) for i in range(B)]  # this rank's utterance slice: global utterance id = rank * B + i
    toks = [ctx.tokenize(t) for t in texts]
    eng.set_seed(1234 + env.rank)
    out = {"mode": name, "prefix_share": share, "kv_dtype": "f32" if kv_f32 else "bf16", "voices": n_voices}

    def begin():
        eng.begin_sentences(list(range(B)), vid, toks, [args.kv_capacity] * B, [1 << 20] * B, [0.7] * B)

    # ---- sentence start of the whole batch (prefix restore / sharing + ragged text prefill), device-timed ----
    ext = torch.cuda.ExternalStream(eng.stream_handle(), device=torch.device("cuda", env.local))
    begin(); eng.sync()                                           # first call: lazy allocations, function attributes
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(ext); begin(); eng.join(); b1.record(ext); eng.sync()
    out["sentence_start_ms"] = round(b0.elapsed_time(b1), 3)
    out["sentence_start_rows"] = int(sum(len(t) for t in toks))
    L0 = np.array([args.t_voice + len(t) for t in toks], np.float64)

    if verify and env.rank == 0:
        out["verify"] = verify_against_oracle(args, ctx, d, texts, toks, vid[0])
        begin(); eng.sync()                                       # the verify steps advanced the slots: start the sentences again

    sampler = None
    if primary:   # clocks are sampled from the warm-up through the timed region (the timed region alone can be shorter than one sample period)
        sampler = ClockSampler(env.local); sampler.start()
        # nvidia-smi needs 0.1-0.5 s before its first row: keep the GPU under the same load until rows arrive, then start the sentences again so
        # that the cache length of the timed region is the configured one
        t_s = time.time()
        while len(sampler.rows) < 3 and time.time() - t_s < 3.0:
            eng.steps_enqueue(0, B, 25); eng.join(); eng.sync()
        begin(); eng.sync()
    steps_done = 0
    for _ in range(args.untimed):
        eng.step_enqueue(0, B); steps_done += 1
    eng.join(); eng.sync(); env.barrier()
    l0 = eng.launch_count()
    if primary and env.rank == 0:
        print(f"[bench] launches_before_timed_region={l0}", file=sys.stderr, flush=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_range = primary and os.environ.get("PTTS_NCU_RANGE") == "1"    # `ncu --profile-from-start off`: capture only the timed steps
    if ncu_range:
        P.lib().b200_profiler_range(1)
    e0.record(ext)
    eng.steps_enqueue(0, B, args.steps)                           # K steps enqueued by one native call: no interpreter between the graph launches
    eng.join()                                                    # the Mimi stream's last frame is inside the timed region
    e1.record(ext)
    eng.sync()
    if ncu_range:
        P.lib().b200_profiler_range(0)
    env.barrier()
    ms = e0.elapsed_time(e1)
    out["gpu_launches"] = int(eng.launch_count() - l0)
    if sampler:
        out["clocks"] = sampler.stop()
    mid_step = steps_done + args.steps / 2.0
    steps_done += args.steps
    ms_max = env.max_over_ranks(ms)
    out["ms_rank"] = ms
    out["ms_per_step"] = ms_max / args.steps
    out["value"] = B * env.world * args.steps / (ms_max * 1e-3)
    Lm = L0 + mid_step
    out["kv_len"] = int(Lm.mean())
    if primary and args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, B, env.rank, env.world)

    # ---- end-to-end through the public C-ABI calls with host buffers ----
    if primary and not args.no_e2e:
        rng = np.random.default_rng(5 + env.rank)
        noise = (rng.standard_normal((B, 32)) * np.sqrt(0.7)).astype(np.float32)
        pcm = np.zeros((B, P.FRAME), np.float32); produced = np.zeros(B, np.int32)
        eng.step_into(0, B, noise, pcm, produced); steps_done += 1
        if args.overlap:                                          # warm-up of the pipelined call pair: first use runs eagerly, second captures its graphs
            for _ in range(3):
                eng.submit(0, B, noise); eng.submit(0, B, noise)
                eng.collect_into(pcm, produced); eng.collect_into(pcm, produced)
                steps_done += 2
        env.barrier()
        t0 = time.perf_counter()
        if args.overlap:
            depth = min(2, args.steps)                            # submits stay two frames ahead of collects (at most three frames in flight)
            for _ in range(depth):
                eng.submit(0, B, noise)
            for _ in range(args.steps - depth):
                eng.submit(0, B, noise)
                eng.collect_into(pcm, produced)
            for _ in range(depth):
                eng.collect_into(pcm, produced)
        else:
            for _ in range(args.steps):
                eng.step_into(0, B, noise, pcm, produced)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        steps_done += args.steps
        assert produced.all(), "bench utterances must stay active (never-EOS checkpoint)"
        dt_max = env.max_over_ranks(dt)
        out["e2e"] = {"value": round(B * env.world * args.steps / dt_max, 2), "unit": UNIT, "h2d_bytes_per_step": int(noise.nbytes),
                      "d2h_bytes_per_step": int(pcm.nbytes + produced.nbytes),
                      "api": "b200_submit/b200_collect (submits kept two frames ahead of collects)" if args.overlap else "b200_step (synchronous)"}

    # ---- per-kernel-family device timing: eager single-stream pass with event pairs (b200_profile) ----
    eng.profile(True)
    prof_step0 = steps_done
    for _ in range(args.steps):
        eng.step_enqueue(0, B)
    eng.sync()
    prof = eng.profile_read()
    steps_done += args.steps
    hbm, tflops, which = peaks()
    elt = 4 if kv_f32 else 2
    Lprof = L0 + prof_step0 + args.steps / 2.0
    own = Lprof + 1 - (args.t_voice if share else 0)              # rows of the per-utterance stream (shared mode: the prefix is not streamed per row)
    stream_ms, stream_n = prof["attn_stream"]
    # algorithmic bytes of ONE streaming-kernel launch (one layer, all utterances): its K and V rows once + q in / out rows
    stream_bytes = float((2 * own * 1024 * elt).sum() + B * 1024 * (4 + 2))
    seg = {k: round(v[0] / args.steps, 4) for k, v in prof.items()}
    if stream_n:
        ach = stream_bytes / (stream_ms / stream_n * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(REPO, "profiles", f"attn_stream_traffic_{name}.json")
        if os.path.exists(tp):   # DRAM bytes of one launch from an `ncu --set full` capture (tools/make_traffic_json.py), scaled to this run's rows
            tj = json.load(open(tp))
            traffic = int((tj["dram_bytes_read"] + tj["dram_bytes_write"]) * stream_bytes / tj["algorithmic_bytes_at_capture"])
        out["roofline"] = {"bound": "hbm", "kernel": f"attn_flow_split_kernel<{'float' if kv_f32 else '__nv_bfloat16'}> (FlowLM attention, per-utterance KV stream, one layer)",
                           "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s", "frac": round(ach / hbm, 4), "traffic": traffic, "peak_source": which,
                           "algorithmic_bytes_per_launch": int(stream_bytes), "avg_launch_ms": round(stream_ms / stream_n, 4),
                           "share_of_step": round(stream_ms / max(prof["step"][0], 1e-9), 4), "segments_ms_per_step": seg,
                           "note": "peak = driver-measured copy bandwidth (read+write); a read-only stream can exceed it slightly"}
        tile_ms, tile_n = prof["attn_prefix_tiles"]
        if tile_n:
            # shared prefix x all rows on tensor cores: 4 * rows * 16 heads * keys * 64 MACs x2 (hi + lo operands) per launch
            fl = float(4.0 * B * 16 * args.t_voice * 64 * 2 * 2)
            out["roofline"]["prefix_tiles"] = {"kernel": "attn_tile_kernel (shared voice prefix, mma.sync bf16 hi+lo)", "avg_launch_ms": round(tile_ms / tile_n, 4),
                                               "tflops": round(fl / (tile_ms / tile_n * 1e-3) / 1e12, 1), "peak_tflops": tflops,
                                               "prefix_bytes_read_once": int(2 * args.t_voice * 1024 * 2 * n_voices)}
    # whole-step bound on the bytes that MUST move (SURVEY 8d): weights once + per-utterance KV + Mimi/conv state + PCM; in shared mode the
    # prefix counts once per voice and layer, not once per utterance
    kv_unique = float((12 * (Lm + 1 - (args.t_voice if share else 0)) * 1024 * elt).sum()) + (12.0 * args.t_voice * 1024 * elt * n_voices if share else 0.0)
    step_bytes = 189.6e6 + kv_unique + B * (1.09e6 + 0.12e6 + 7.7e3)
    step_flops = B * (715e6 + 0.0246e6 * float(Lm.mean()))
    t_floor = max(step_bytes / (hbm * 1e9), step_flops / (tflops * 1e12))
    out["step_roofline"] = {"unique_bytes_per_step": int(step_bytes), "flops_per_step": int(step_flops), "floor_ms": round(t_floor * 1e3, 4),
                            "bound_frames_per_s_per_gpu": round(B / t_floor, 1), "frac": round((out["value"] / env.world) / (B / t_floor), 4),
                            "binding": "hbm" if step_bytes / (hbm * 1e9) >= step_flops / (tflops * 1e12) else "tensor"}

    # ---- sustained: >= 2 s of back-to-back steps (positions rewound every few hundred steps so the cache never fills) ----
    if primary and args.sustain_s > 0:
        s2 = ClockSampler(env.local); s2.start(); time.sleep(0.2)
        room = args.kv_capacity - int(L0.max()) - 8
        chunk = max(16, min(400, room))
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_steps = 0
        t0 = time.perf_counter()
        c0.record(ext)
        while time.perf_counter() - t0 < args.sustain_s:
            eng.debug_set_position(0, B, int(L0.max()), chunk + 4)
            for _ in range(chunk):
                eng.step_enqueue(0, B)
            n_steps += chunk
            eng.sync()
        eng.join(); c1.record(ext); eng.sync()
        sus_ms = env.max_over_ranks(c0.elapsed_time(c1))
        out["sustained"] = {"seconds": round(sus_ms * 1e-3, 3), "steps": n_steps, "value": round(B * env.world * n_steps / (sus_ms * 1e-3), 1),
                            "ms_per_step": round(sus_ms / n_steps, 4), "kv_len_range": [int(L0.max()), int(L0.max()) + chunk], "clocks": s2.stop()}
    ctx.close()
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, eng, n: int, rank: int, world: int):
    """Writes what the last timed step computed for slots [0, n) of this rank: the arrays b200_step returns to its caller (PCM frame,
    produced flag, latent, EOS logit), read back from the engine's output buffers, as float32 .npy files. Above DUMP_BYTES in all, a
    fixed seeded sample of the slots is written; slots.npy lists which. With world > 1 each rank writes <name>_rank<r>.npy."""
    import ptts_b200 as P
    import torch
    row_bytes = 4 * (P.FRAME + P.LDIM + 2)
    rows = max(1, min(n, DUMP_BYTES // (row_bytes * world)))
    slots = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    ptr = P.lib().b200_device_ptr(eng.h, b"produced")

    class _Produced:                                   # b200_debug_read_f32 reads f32 buffers only: the int32 flags go through torch
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "strides": None, "version": 3}
    out = {"pcm": eng.debug_read("pcm", 0, n * P.FRAME).reshape(n, P.FRAME),
           "produced": torch.as_tensor(_Produced(), device="cuda").cpu().numpy().astype(np.float32),
           "latents": eng.debug_read("latent", 0, n * P.LDIM).reshape(n, P.LDIM),
           "eos_logit": eng.debug_read("eos", 0, n)}
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a[slots], np.float32))
    np.save(os.path.join(out_dir, "slots" + suffix + ".npy"), slots.astype(np.float64))


def verify_against_oracle(args, ctx, model_dir, texts, toks, voice, frames: int = 4):
    """Checker leg (outside every timed region): slots 0, the one whose tokens straddle the first 2048-row prefill chunk, and B-1 of the
    TIMED context against the CPU oracle under identical injected noise (same as tests/test_gpu_bench_config.py)."""
    import oracle
    eng = ctx.engine
    B = len(texts)
    o = oracle.Oracle(model_dir, threads=os.cpu_count() or 1)
    base = o.stream("cosette", kv_capacity=args.kv_capacity)
    cum = np.concatenate([[0], np.cumsum([len(t) for t in toks])])
    straddle = int(np.searchsorted(cum, 2048, side="right") - 1) if cum[-1] > 2048 else B // 2
    check = sorted({0, min(straddle, B - 1), B - 1})
    rng = np.random.default_rng(99)
    noise = (rng.standard_normal((frames, B, 32)) * np.sqrt(0.7)).astype(np.float32)
    worst = {"latent_maxabs": 0.0, "latent_rel": 0.0, "snr_db_min": 1e9, "kv_maxabs": 0.0}
    streams = {}
    for k in check:
        s = base.clone()
        assert s.sentence_init(texts[k]) == toks[k]
        for layer in (0, 5):
            for kv in (0, 1):
                worst["kv_maxabs"] = max(worst["kv_maxabs"], float(np.abs(eng.read_kv(k, layer, kv, s.current_end) - s.kv(layer, kv)).max()))
        streams[k] = s
    for i in range(frames):
        gp, prod, glat, geos = eng.step(0, B, noise[i])
        for k in check:
            ok, lat, pcm, e = streams[k].step(noise[i, k])
            err = pcm.astype(np.float64) - gp[k].astype(np.float64)
            worst["latent_maxabs"] = max(worst["latent_maxabs"], float(np.abs(glat[k] - lat).max()))
            worst["latent_rel"] = max(worst["latent_rel"], float(np.linalg.norm(glat[k] - lat) / np.linalg.norm(lat)))
            worst["snr_db_min"] = min(worst["snr_db_min"], float(10 * np.log10((pcm.astype(np.float64) ** 2).sum() / max((err ** 2).sum(), 1e-30))))
    ok = worst["latent_maxabs"] < 4e-2 and worst["latent_rel"] < 1.5e-2 and worst["snr_db_min"] > 40.0 and worst["kv_maxabs"] < 6e-2
    return {"slots": check, "frames": frames, "kv_len": int(streams[check[0]].current_end), "pass": bool(ok),
            "tolerance": {"latent_maxabs": 4e-2, "latent_rel": 1.5e-2, "snr_db_min": 40.0, "kv_maxabs": 6e-2}, **{k: round(v, 4) for k, v in worst.items()}}


def ragged_sentence(i: int) -> tuple[str, int]:
    from make_assets import COMMON_WORDS
    rng = np.random.default_rng(50000 + i)
    n = int(rng.integers(3, 46))                                  # 3..45 words
    ws = [COMMON_WORDS[int(k)] for k in rng.integers(0, len(COMMON_WORDS), n)]
    return (" ".join(ws)).capitalize() + ".", n


def run_ragged(env: Env):
    """BASELINE configs[4]: 2048 sentences per GPU through 256 slots with continuous batching (weak scaling: the global list has
    2048 x world sentences, sharded over ranks by longest-processing-time on the frame cap)."""
    import ptts_b200 as P
    import sharding
    from make_assets import default_model_dir, VOICES
    args, torch = env.args, env.torch
    per_gpu = args.ragged_sentences
    total = per_gpu * env.world
    sents = [ragged_sentence(i) for i in range(total)]
    costs = [sharding.estimate_frames(w) for _, w in sents]
    shards = sharding.shard_utterances(costs, env.world)
    mine = shards[env.rank]
    d = default_model_dir(eos_mode="late")
    ctx = P.Context(d, device=env.local, max_slots=args.batch, max_voices=8, kv_capacity=1024, pdl=args.pdl, cuda_graphs=args.cuda_graphs, overlap=args.overlap)
    P.set_seed(4321)

    def one_run(ids, keep_pcm):
        b = P.Batch(ctx, args.batch)
        b.configure(refill_min=args.refill_min, refill_every=args.refill_every, range_quantum=32, keep_pcm=keep_pcm)
        utts = [b.add(VOICES[i % 8], sents[i][0], 0.7) for i in ids]
        env.barrier()
        t0 = time.perf_counter()
        frames = b.run()
        ctx.engine.sync()
        dt = time.perf_counter() - t0
        return b, utts, frames, dt

    one_run(mine[: min(len(mine), 2 * args.batch)], 0)            # warm-up: voice prefills, graph captures for the stepped ranges
    # (a) every frame is copied to a host buffer as it is collected (D2H + one host copy per step, like the e2e leg) but not kept;
    # (b) the whole job's audio is accumulated in RAM per utterance (2+ GB here: first-touch page faults then dominate the host loop)
    b_acc, _, frames_acc, dt_acc = one_run(mine, 1)
    acc_ms = sharding.gather_stats([float(frames_acc), dt_acc * 1e3], device="cuda")
    del b_acc
    b, utts, frames, dt = one_run(mine, 0)
    st = b.stats()
    g = sharding.gather_stats([float(frames), dt * 1e3, float(st["steps"]), float(st["slot_steps"]), float(st["refills"]), float(sum(costs[i] for i in mine))], device="cuda")
    t_max = float(g[:, 1].max()) * 1e-3
    tot_frames = float(g[:, 0].sum())
    out = {"workload": f"configs[4]: {per_gpu} sentences per GPU (3-45 words, EOS-firing checkpoint, 8 voices), {args.batch} slots per GPU, continuous batching, "
                       f"text in -> PCM frames delivered to a host buffer every step, LPT sharding of {total} sentences over {env.world} rank(s)",
           "value": round(tot_frames / t_max, 1), "unit": UNIT, "scaling": "weak", "seconds": round(t_max, 3), "frames": int(tot_frames),
           "sentences": total, "steps_max": int(g[:, 2].max()), "refills_max": int(g[:, 4].max()),
           "idle_slot_fraction": round(1.0 - float(g[:, 0].sum()) / float(g[:, 3].sum()), 4),
           "rank_time_imbalance": round(float(g[:, 1].max() / g[:, 1].mean() - 1.0), 4),
           "rank_cap_imbalance": round(float(g[:, 5].max() / g[:, 5].mean() - 1.0), 5),
           "per_rank_frames": [int(x) for x in g[:, 0]], "per_rank_ms": [round(float(x), 1) for x in g[:, 1]],
           "refill_policy": {"refill_min": args.refill_min, "refill_every": args.refill_every},
           "host_ms_rank0": {k: round(st[k], 1) for k in ("wall_ms", "begin_ms", "submit_ms", "collect_ms")},
           "audio_seconds_per_wall_second": round(tot_frames / t_max / 12.5, 1),
           "value_accumulating_all_pcm_in_ram": round(float(acc_ms[:, 0].sum()) / (float(acc_ms[:, 1].max()) * 1e-3), 1)}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="utterances per GPU")
    ap.add_argument("--kv-len", type=int, default=1500, help="FlowLM cache positions per utterance in mid-run")
    ap.add_argument("--kv-capacity", type=int, default=2048)
    ap.add_argument("--gemm-path", type=int, default=0)
    ap.add_argument("--pdl", type=int, default=1)
    ap.add_argument("--cuda-graphs", type=int, default=1)
    ap.add_argument("--overlap", type=int, default=1, help="two-stream pipeline: Mimi(t) overlaps FlowLM(t+1)")
    ap.add_argument("--prefix-share", type=int, default=1, help="primary mode: 1 = shared voice prefix (cascade attention), 0 = private copies")
    ap.add_argument("--ref-frames-per-step", type=int, default=4)
    ap.add_argument("--ragged-sentences", type=int, default=2048, help="sentences per GPU of the continuous-batching workload")
    ap.add_argument("--refill-min", type=int, default=16)
    ap.add_argument("--refill-every", type=int, default=8)
    ap.add_argument("--sustain-s", type=float, default=2.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip private_kv / kv_f32 / multi_voice / ragged / verify / sustained")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--only-ragged", action="store_true", help="development: run only the continuous-batching workload")
    ap.add_argument("--verify", action="store_true", help="run the oracle check of the timed context even with --no-extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.no_extras:
        args.sustain_s = 0.0

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    # tokens of a 40-word paragraph ~ 60-75; voice prefix sized so that voice + text + steps/2 ~ kv_len
    args.untimed = max(args.warmup, 100)             # extended warm-up: also gives the clock sampler a loaded window
    args.t_voice = max(16, args.kv_len - 45 - args.untimed - args.steps // 2)
    # the primary mode runs untimed + timed + e2e (steps + 7) + profiled (steps) steps without a rewind: the cache must hold all of them
    # behind the voice prefix and the paragraph (< 256 tokens), or utterances reach their cap and a long --steps run times finished slots
    args.kv_capacity = max(args.kv_capacity, args.t_voice + 256 + args.untimed + 3 * args.steps + 8)

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = run_reference(args, rank, world)
        line = {"impl": "reference", "metric": METRIC, "value": round(r["value"], 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"configs[3]: full FlowLM+head+Mimi, ~{PARAGRAPH_WORDS}-word paragraphs (CPU arm: batch 1, KV length ~{r['kv_len']}; see cpu_baseline.sample)",
                           "batch_per_gpu": 1, "kv_len": r["kv_len"]},
                "cpu_baseline": {"value": round(r["value"], 3), "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                "e2e": {"value": round(r["value"], 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import ptts_b200 as P
    from make_assets import default_model_dir, VOICES
    if rank == 0:                                     # load the library build() made + synthesise the model directories once, the other ranks wait
        P.lib()                                       # raises when it has not been built: the benchmark never compiles into the tree
        default_model_dir(eos_mode="never", t_voice=args.t_voice, voices=["cosette"])
        if not args.no_extras:
            default_model_dir(eos_mode="never", t_voice=args.t_voice, voices=VOICES)
            default_model_dir(eos_mode="late")
    if world > 1:
        dist.barrier()
    env = Env(args)
    B = args.batch

    if args.only_ragged:
        r = run_ragged(env)
        if rank == 0:
            print(json.dumps({"ragged": r}), flush=True)
        return 0
    prim = run_mode(env, "shared" if args.prefix_share else "private", args.prefix_share, 0, primary=True, verify=((not args.no_extras or args.verify) and not args.no_verify and world == 1))
    extras = {}
    if not args.no_extras:
        other = 0 if args.prefix_share else 1
        for key, kw in (("private_kv" if args.prefix_share else "shared_kv", dict(share=other, kv_f32=0)), ("kv_f32", dict(share=0, kv_f32=1)),
                        ("multi_voice", dict(share=1, kv_f32=0, n_voices=8))):
            try:
                r = run_mode(env, key, **kw)
                extras[key] = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items() if k not in ("ms_rank",)}
                extras[key]["value"] = round(r["value"], 1)
            except Exception as ex:
                extras[key] = {"error": repr(ex)}
        try:
            extras["ragged"] = run_ragged(env)
        except Exception as ex:
            extras["ragged"] = {"error": repr(ex)}

    value = prim["value"]
    kvdesc = "shared voice prefix (cascade attention)" if args.prefix_share else "private prefix copies"
    line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(prim["ms_per_step"], 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"configs[3]: full FlowLM+head+Mimi, batch {B}/GPU of ~{PARAGRAPH_WORDS}-word paragraphs, FlowLM KV length ~{prim['kv_len']} in mid-run, {kvdesc}",
                       "batch_per_gpu": B, "kv_len": prim["kv_len"], "kv_dtype": "bf16", "kv_capacity": args.kv_capacity, "prefix_share": args.prefix_share,
                       "t_voice": args.t_voice, "parallelism": f"utterance-sharded x{world}",
                       "l2": "inputs larger than L2 (per-utterance KV + Mimi state + weights ~%.2f GB/step, streamed evict-first)" % (prim["step_roofline"]["unique_bytes_per_step"] / 1e9),
                       "rtf_per_utterance": round(12.5 / (value / (B * world)), 4),
                       "sentence_start_ms": prim["sentence_start_ms"], "sentence_start_rows": prim["sentence_start_rows"],
                       "roofline_bound_frames_per_s_per_gpu": prim["step_roofline"]["bound_frames_per_s_per_gpu"],
                       "frac_of_step_roofline": prim["step_roofline"]["frac"]},
            "clocks": prim.get("clocks"), "gpu_launches": prim["gpu_launches"], "step_roofline": prim["step_roofline"]}
    for k in ("e2e", "roofline", "verify", "sustained"):
        if k in prim:
            line[k] = prim[k]
    line.update(extras)
    if world > 1:
        import sharding
        g = sharding.gather_stats([B * args.steps, prim["ms_rank"]], device="cuda")
        line["per_rank_ms"] = [round(float(x), 3) for x in g[:, 1]]
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_quick(args)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
