"""CPU: the C-ABI library loads without a GPU and exports every symbol include/ptts_b200.h declares, plus the
reference's ten C++ API functions under their original mangled names (drop-in for demos/pocket-tts.cpp)."""
import ctypes
import os
import re
import subprocess

from conftest import REPO

REFERENCE_MANGLED = [
    "_Z13ptts_set_seedj", "_Z13ptts_get_seedv", "_Z9ptts_initP12ggml_backendS0_PKc", "_Z20ptts_get_sample_rateP14ptts_context_t",
    "_Z19ptts_get_frame_sizeP14ptts_context_t", "_Z28ptts_stream_from_safetensorsP14ptts_context_tPKcf",
    "_Z17ptts_stream_resetP13ptts_stream_t", "_Z17ptts_stream_flushP13ptts_stream_t",
    "_Z16ptts_stream_sendP13ptts_stream_tPKc", "_Z19ptts_stream_receiveP13ptts_stream_tPf",
]


def test_exports(P):
    hdr = open(os.path.join(REPO, "include", "ptts_b200.h")).read()
    names = re.findall(r"B200_API\s+[\w\s\*]+?\b(\w+)\s*\(", hdr)
    assert len(names) > 40
    L = ctypes.CDLL(P.LIB_PATH)
    for n in names + REFERENCE_MANGLED:
        assert hasattr(L, n), n


def test_loads_without_gpu_and_fails_loudly(P):
    import torch
    if torch.cuda.is_available():
        return
    cfg = P.default_config(max_slots=1)
    h = ctypes.c_void_p()
    rc = P.lib().b200_engine_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc != 0 and not h.value          # no CUDA device -> error, never a CPU fallback


def test_constants(P):
    assert P.FRAME == 1920 and P.SAMPLE_RATE == 24000


def test_product_never_touches_oracle():
    pkg = os.path.join(REPO, "pocket-tts.cpp_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                src = open(os.path.join(root, f), errors="ignore").read()
                assert "oracle" not in src.replace("no CPU fallback", ""), os.path.join(root, f)


def test_gemm_planner_invariants(P):
    """The tile/split-K cost model (host code, no GPU): valid tile widths, no empty splits, workspace bound, and the decode shapes of the
    model never fall back to more partial planes than the reduction kernels were measured with."""
    import ctypes
    L = P.lib()
    L.b200_debug_gemm_plan.restype = ctypes.c_int
    L.b200_debug_gemm_plan.argtypes = [ctypes.c_int] * 5 + [ctypes.POINTER(ctypes.c_int)] * 2
    bn, sp = ctypes.c_int(), ctypes.c_int()
    shapes = [(1024, 3072), (1024, 1024), (1024, 4096), (4096, 1024), (512, 512), (1024, 512), (512, 10240), (512, 32), (512, 1536), (2048, 512), (3584, 512)]
    for R in (3, 16, 64, 256, 512, 4096, 24576):
        for K, N in shapes:
            for ln in (0, 1):
                assert L.b200_debug_gemm_plan(R, N, K, 148, ln, ctypes.byref(bn), ctypes.byref(sp)) == 0
                assert bn.value in (32, 64, 128) and N % bn.value == 0
                assert 1 <= sp.value <= 16
                if sp.value > 1:
                    kbps = -(-(K // 64) // sp.value)
                    assert kbps >= 4 and sp.value * R * N <= 32 << 20          # >= 4 k-blocks per split, partial planes fit the workspace
                if R > 512:
                    assert sp.value == 1                                       # large-M GEMMs are never split
    assert L.b200_debug_gemm_plan(0, 64, 64, 148, 0, ctypes.byref(bn), ctypes.byref(sp)) != 0


def test_attention_work_list_invariants(P):
    """The host-side work lists of the FlowLM attention (b200_debug_attn_plan runs the builders the engine uses; no GPU).
    Decode: every live row with a prefix gets one item per prefix split, whose key ranges tile [0, P) exactly once (a voice shorter than
    the longest one gets empty ranges), <= 64 rows of one prefix per item, the split count the merges read equals the items' splits.
    Prefill: every row lies in exactly one item of its own chunk; an item is a run of consecutive positions of one slot with the keys
    [0, P) of the prefix slot and [P, last position] of its own slot; a run only ends at a chunk edge, a new slot or after 64 rows."""
    import numpy as np
    AF_MAX_SPLITS, AF_PFX_SPLITS, AT_ROWS = 16, 8, 64
    rng = np.random.default_rng(0)
    for case in range(300):
        n = int(rng.choice([1, 3, 4, 63, 64, 65, 128, 200, 256]))
        nv = int(rng.integers(1, 9))
        lens = [int(rng.choice([1, 7, 63, 64, 65, 125, 1345, int(rng.integers(1, 3000))])) for _ in range(nv)]
        voice = rng.integers(-1, nv, n)                                          # -1: private cache
        pfx_slot = np.array([1000 + v if v >= 0 else 0 for v in voice], np.int32)
        pfx_len = np.array([lens[v] if v >= 0 else 0 for v in voice], np.int32)
        sms = int(rng.choice([1, 16, 132, 148]))
        splits, items, rows = P.attn_plan(False, pfx_slot, pfx_len, num_sms=sms, max_voices=8)
        assert splits >= 0, (case, splits)
        if (pfx_len == 0).all():
            assert splits == 0 and len(items) == 0
            continue
        assert 1 <= splits <= AF_PFX_SPLITS
        assert len(items) <= ((n + AT_ROWS - 1) // AT_ROWS + 8 + 1) * AF_PFX_SPLITS + 8          # the engine's work-list capacity
        per_row = {}
        for row0, nr, a_slot, a0, a1, b_slot, b0, b1, osp in items:
            assert 1 <= nr <= AT_ROWS and b1 == b0 and AF_MAX_SPLITS <= osp < AF_MAX_SPLITS + splits
            for r in rows[row0:row0 + nr]:
                assert pfx_slot[r] == a_slot and 0 <= a0 <= a1 <= pfx_len[r]
                per_row.setdefault(int(r), []).append((osp, a0, a1))
        assert sorted(per_row) == [r for r in range(n) if pfx_len[r] > 0]
        for r, its in per_row.items():
            its.sort()
            assert [o for o, _, _ in its] == list(range(AF_MAX_SPLITS, AF_MAX_SPLITS + splits)), (case, r)
            edge = 0
            for _, a0, a1 in its:
                assert a0 == min(edge, pfx_len[r]) and a1 >= a0
                edge = max(edge, a1)
            assert edge == pfx_len[r]
    for case in range(300):
        n_slots = int(rng.integers(1, 6))
        pfx_slot = np.zeros(n_slots, np.int32); pfx_len = np.zeros(n_slots, np.int32)
        slots, pos = [], []
        for s in range(n_slots):
            P_ = int(rng.choice([0, 0, 1, 64, 125, 1345]))
            pfx_slot[s] = 50 + s if P_ else 0; pfx_len[s] = P_
            start = P_ + int(rng.choice([0, 0, 125, int(rng.integers(0, 100))]))
            ln = int(rng.choice([1, 63, 64, 65, 130, int(rng.integers(1, 300))]))
            p = list(range(start, start + ln))
            if ln > 10 and rng.random() < 0.3:                                 # a gap: two runs of one slot
                p = p[:ln // 2] + [x + 5 for x in p[ln // 2:]]
            slots += [s] * ln; pos += p
        total = len(slots)
        chunk = int(rng.choice([1, 7, 64, 100, 4096]))
        nch, items, first = P.attn_plan(True, pfx_slot, pfx_len, row_slot=slots, row_pos=pos, chunk_rows=chunk)
        assert nch == -(-total // chunk) and len(first) == nch + 1 and first[0] == 0 and first[-1] == len(items)
        for c in range(nch):
            r0, R = c * chunk, min(chunk, total - c * chunk)
            covered = []
            prev = None
            for row0, nr, a_slot, a0, a1, b_slot, b0, b1, osp in items[first[c]:first[c + 1]]:
                assert 1 <= nr <= AT_ROWS and osp == -1
                rr = list(range(r0 + row0, r0 + row0 + nr))
                assert all(slots[r] == b_slot for r in rr) and all(pos[r + 1] == pos[r] + 1 for r in rr[:-1])
                P_ = pfx_len[b_slot]
                assert (a_slot, a0, a1) == (pfx_slot[b_slot], 0, P_) and (b0, b1) == (P_, pos[rr[-1]] + 1)
                if prev is not None and slots[prev[-1]] == b_slot and pos[rr[0]] == pos[prev[-1]] + 1:
                    assert len(prev) == AT_ROWS                                # a run of one slot is only cut after 64 rows
                covered += rr; prev = rr
            assert covered == list(range(r0, r0 + R)), (case, c)
