"""Step-time cost of the per-sentence sampling controls (DESIGN.md 4.7) on the bench-shaped batch: 256 slots, one 1345-row voice shared
by every slot (prefix_share = 1), KV length ~1.5 k, graphs and overlap on. Cases: all defaults; all rows at N = 2, 4, 8; 10 % of rows at
N = 4; the noise clamp on (a = sigma). Cases are measured in alternating rounds in one process so that host noise hits all of them alike;
each round re-begins the sentences at the same positions and times `steps` device-resident steps (host clock around a synchronise).
Also batch-1 ms per frame (synchronous b200_step) at N = 1 and 4. Writes one JSON (default profiles/sampling_b200.json).

    python tools/sampling_cost.py [--steps 40] [--rounds 5] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO); sys.path.insert(0, HERE)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as ex:   # the measurement itself still needs the GPU; only the label is missing
        return {"error": str(ex)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "sampling_b200.json"))
    args = ap.parse_args()
    import bench
    import ptts_b200 as P
    from make_assets import default_model_dir
    B, KV_CAP, T_VOICE = 256, 2048, 1345
    d = default_model_dir(eos_mode="never", t_voice=T_VOICE, voices=["cosette"])
    ctx = P.Context(d, max_slots=B, max_voices=1, kv_capacity=KV_CAP)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=0.7).voice
    toks = [ctx.tokenize(bench.synth_paragraph(i)) for i in range(B)]
    sigma = float(np.sqrt(np.float32(0.7)))
    cases = {
        "default": [(1, 0.0, -4.0)] * B,
        "all_N2": [(2, 0.0, -4.0)] * B,
        "all_N4": [(4, 0.0, -4.0)] * B,
        "all_N8": [(8, 0.0, -4.0)] * B,
        "10pct_N4": [(4, 0.0, -4.0) if i % 10 == 0 else (1, 0.0, -4.0) for i in range(B)],
        "clamp_sigma": [(1, sigma, -4.0)] * B,
    }
    warm = 100                                        # KV length at the timed window: ~1345 + 45 tokens + 100 warm-up steps ~ 1.5 k

    def begin(samp):
        eng.begin_sentences(list(range(B)), [voice] * B, toks, [warm + args.steps + 8] * B, [1 << 20] * B, [0.7] * B,
                            rng_streams=list(range(1, B + 1)), sampling=samp)

    times = {k: [] for k in cases}
    for r in range(args.rounds + 1):                  # round 0 = warm-up (graph capture of every case)
        for name, samp in cases.items():
            begin(samp)
            eng.steps_enqueue(0, B, warm)
            eng.sync()
            t0 = time.perf_counter()
            eng.steps_enqueue(0, B, args.steps)
            eng.sync()
            if r:
                times[name].append((time.perf_counter() - t0) * 1e3 / args.steps)
    L0 = int(np.mean([T_VOICE + len(t) for t in toks]) + warm)
    res = {"card": card(), "batch": B, "voice_rows": T_VOICE, "kv_len_at_window_start": L0, "steps_per_window": args.steps, "rounds": args.rounds,
           "step_ms": {k: {"median": round(float(np.median(v)), 4), "min": round(float(np.min(v)), 4), "max": round(float(np.max(v)), 4)} for k, v in times.items()}}
    base = res["step_ms"]["default"]["median"]
    res["extra_ms_per_substep_all_rows"] = {k: round((res["step_ms"][k]["median"] - base) / (n - 1), 4) for k, n in (("all_N2", 2), ("all_N4", 4), ("all_N8", 8))}
    ctx.close()

    c1 = P.Context(d, max_slots=1, max_voices=1, kv_capacity=KV_CAP)
    e1 = c1.engine
    v1 = c1.stream("cosette", temp=0.7).voice
    b1 = {}
    for N in (1, 4):
        b1[N] = []
    for r in range(args.rounds + 1):
        for N in (1, 4):
            e1.begin_sentences([0], [v1], [toks[0]], [200], [1 << 20], [0.7], sampling=[(N, 0.0, -4.0)])
            for _ in range(10):
                e1.step(0, 1, None)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                e1.step(0, 1, None)
            if r:
                b1[N].append((time.perf_counter() - t0) * 1e3 / args.steps)
    res["batch1_ms_per_frame"] = {f"N{N}": round(float(np.median(v)), 4) for N, v in b1.items()}
    c1.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
