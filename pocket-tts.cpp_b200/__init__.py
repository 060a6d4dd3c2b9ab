"""ctypes binding of libptts_b200.so — the B200-native Pocket-TTS generation engine.

Mirrors the reference's `pocket_tts` streaming API (include/pocket_tts/pocket_tts.h of Codes4Fun/pocket-tts.cpp:
init / stream_from_safetensors / send / flush / receive) plus the batched device layer (include/ptts_b200.h).
There is NO CPU fallback: if the shared library is missing or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libptts_b200.so")

FRAME = 1920
SAMPLE_RATE = 24000
LDIM = 32


class B200Config(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int), ("max_slots", ctypes.c_int), ("max_voices", ctypes.c_int), ("kv_capacity", ctypes.c_int),
                ("kv_f32", ctypes.c_int), ("mimi_mask_mode", ctypes.c_int), ("convt_split", ctypes.c_int), ("gemm_path", ctypes.c_int),
                ("max_prefill_rows", ctypes.c_int), ("cuda_graphs", ctypes.c_int), ("pdl", ctypes.c_int), ("overlap", ctypes.c_int),
                ("prefix_share", ctypes.c_int)]


class AttnOpts(ctypes.Structure):
    """b200_attn_opts: per-call overrides of the attention switches (negative = keep the engine's value)."""
    _fields_ = [(k, ctypes.c_int) for k in ("stream_splits", "tile_prec", "prefill_prec", "fork_tiles", "counted_merge", "tile_min_rows")]

    def __init__(self, **kw):
        super().__init__(*([-1] * len(self._fields_)))
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError(k)
            setattr(self, k, int(v))


class BatchStats(ctypes.Structure):
    _fields_ = [("steps", ctypes.c_longlong), ("frames", ctypes.c_longlong), ("slot_steps", ctypes.c_longlong), ("sentences", ctypes.c_longlong),
                ("refills", ctypes.c_longlong), ("wall_ms", ctypes.c_double), ("begin_ms", ctypes.c_double), ("submit_ms", ctypes.c_double), ("collect_ms", ctypes.c_double)]


_I32P, _F32P, _U32P = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint32)
BATCH_BEGIN_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, _I32P, _I32P, _I32P, _I32P, _I32P, _I32P, _F32P, _U32P)
BATCH_SUBMIT_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int)
BATCH_COLLECT_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, _F32P, _I32P)
BATCH_END_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, _I32P)

_lib = None


def build(force: bool = False) -> str:
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ptts_b200_build", os.path.join(_HERE, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build(force=force)


def lib():
    """Loads the CUDA library. Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python pocket-tts.cpp_b200/build.py` (no CPU fallback exists)")
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    fp, ip, cp = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p
    sig = {
        "b200_default_config": (None, [ctypes.POINTER(B200Config)]),
        "b200_engine_create": (ci, [ctypes.POINTER(B200Config), ctypes.POINTER(vp)]),
        "b200_engine_destroy": (None, [vp]),
        "b200_upload_tensor": (ci, [vp, cp, vp, ci, ctypes.POINTER(ctypes.c_int64), ci]),
        "b200_finalize_weights": (ci, [vp]),
        "b200_voice_create": (ci, [vp, fp, ci]),
        "b200_begin_sentence": (ci, [vp, ci, ci, ip, ci, ci, ci, cf]),
        "b200_begin_sentences": (ci, [vp, ci, ip, ip, ip, ip, ip, ip, fp]),
        "b200_step": (ci, [vp, ci, ci, fp, fp, ip, fp, fp]),
        "b200_step_enqueue": (ci, [vp, ci, ci, ci]),
        "b200_steps_enqueue": (ci, [vp, ci, ci, ci]),
        "b200_submit": (ci, [vp, ci, ci, fp]),
        "b200_collect": (ci, [vp, fp, ip]),
        "b200_sync": (ci, [vp]),
        "b200_join": (ci, [vp]),
        "b200_mimi_reset": (ci, [vp, ci, ci]),
        "b200_mimi_decode": (ci, [vp, ci, ci, fp, fp]),
        "b200_mimi_decode_enqueue": (ci, [vp, ci, ci]),
        "b200_set_seed": (None, [vp, ctypes.c_uint64]),
        "b200_slot_position": (ci, [vp, ci]),
        "b200_debug_set_position": (ci, [vp, ci, ci, ci, ci]),
        "b200_debug_set_latent": (ci, [vp, ci, ci, fp]),
        "b200_debug_gemm": (ci, [vp, ci, fp, ci, ci, ci, ci, ci, fp, ci, fp, ci, fp, fp]),
        "b200_profile": (ci, [vp, ci]),
        "b200_profile_read": (ci, [vp, fp, ip]),
        "b200_profiler_range": (None, [ci]),
        "b200_stream": (vp, [vp]),
        "b200_device_ptr": (vp, [vp, cp]),
        "b200_launch_count": (ctypes.c_longlong, [vp]),
        "b200_read_kv": (ci, [vp, ci, ci, ci, ci, fp]),
        "b200_debug_write_kv": (ci, [vp, ci, ci, ci, ci, ci, fp]),
        "b200_debug_set_prefix": (ci, [vp, ci, ci, ci]),
        "b200_debug_attention": (ci, [vp, ci, ci, ci, ci, ip, ip, fp, ctypes.POINTER(AttnOpts), fp]),
        "b200_debug_attn_plan": (ci, [ci, ci, ip, ip, ip, ip, ci, ci, ci, ip, ci, ip, ctypes.POINTER(ctypes.c_int)]),
        "b200_build_info": (cp, []),
        "b200_debug_taps": (ci, [vp, ci]),
        "b200_debug_tap": (ci, [vp, cp, ci, fp, ci]),
        "b200_debug_read_f32": (ci, [vp, cp, ctypes.c_longlong, fp, ci]),
        "ptts_c_set_seed": (None, [ctypes.c_uint]),
        "ptts_c_get_seed": (ctypes.c_uint, []),
        "ptts_c_init": (vp, [cp]),
        "ptts_c_init_ex": (vp, [cp, ctypes.POINTER(B200Config)]),
        "ptts_c_get_sample_rate": (ci, [vp]),
        "ptts_c_get_frame_size": (ci, [vp]),
        "ptts_c_stream_from_safetensors": (vp, [vp, cp, cf]),
        "ptts_c_stream_reset": (None, [vp]),
        "ptts_c_stream_flush": (None, [vp]),
        "ptts_c_stream_send": (None, [vp, cp]),
        "ptts_c_stream_receive": (ci, [vp, fp]),
        "ptts_c_engine": (vp, [vp]),
        "ptts_c_destroy": (None, [vp]),
        "ptts_c_voice": (ci, [vp]),
        "ptts_c_slot": (ci, [vp]),
        "ptts_c_tokenize": (ci, [vp, cp, ip, ci]),
        "ptts_c_count_words": (ci, [cp]),
        "ptts_c_stream_pending": (ci, [vp, ci, cp, ci]),
        "b200_begin_sentences_ex": (ci, [vp, ci, ip, ip, ip, ip, ip, ip, fp, ctypes.POINTER(ctypes.c_uint32)]),
        "b200_end_sentences": (ci, [vp, ci, ip]),
        "b200_voice_len": (ci, [vp, ci]),
        "b200_kv_capacity": (ci, [vp]),
        "b200_max_slots": (ci, [vp]),
        "ptts_c_batch_create": (vp, [vp, ci]),
        "ptts_c_batch_destroy": (None, [vp]),
        "ptts_c_batch_configure": (ci, [vp, ci, ci, ci, ci]),
        "ptts_c_batch_add": (ci, [vp, cp, cp, cf]),
        "ptts_c_batch_add_tokens": (ci, [vp, ci, ip, ci, ci, ci, cf, ctypes.c_uint32]),
        "ptts_c_batch_run": (ctypes.c_longlong, [vp]),
        "ptts_c_batch_frames": (ci, [vp, ci]),
        "ptts_c_batch_read": (ci, [vp, ci, fp, ci]),
        "ptts_c_batch_stats": (None, [vp, ctypes.POINTER(BatchStats)]),
        "ptts_c_batch_create_with_ops": (vp, [vp, BATCH_BEGIN_FN, BATCH_SUBMIT_FN, BATCH_COLLECT_FN, ci, ci]),
        "ptts_c_batch_create_with_ops_ex": (vp, [vp, BATCH_BEGIN_FN, BATCH_SUBMIT_FN, BATCH_COLLECT_FN, BATCH_END_FN, ci, ci]),
        "ptts_c_batch_append_tokens": (ci, [vp, ci, ci, ip, ci, ci, ci, cf, ctypes.c_uint32]),
        "ptts_c_batch_pump": (ctypes.c_longlong, [vp, ci]),
        "ptts_c_batch_pop": (ci, [vp, ci, fp, ci]),
        "ptts_c_batch_cancel": (ci, [vp, ci]),
        "ptts_c_batch_status": (ci, [vp, ci, ctypes.POINTER(ctypes.c_int)]),
        "ptts_c_text_create": (vp, [cp]),
        "ptts_c_text_destroy": (None, [vp]),
        "ptts_c_text_encode": (ci, [vp, cp, ip, ci]),
        "ptts_c_text_send": (None, [vp, cp]),
        "ptts_c_text_flush": (None, [vp]),
        "ptts_c_text_reset": (None, [vp]),
        "ptts_c_text_pop": (ci, [vp, cp, ci]),
        "b200_has_encoder": (ci, [vp]),
        "b200_debug_window_attention": (ci, [vp, ci, fp, fp, fp, fp]),
        "b200_voice_embed_audio": (ci, [vp, fp, ctypes.c_longlong, fp]),
        "b200_voice_create_from_audio": (ci, [vp, fp, ctypes.c_longlong]),
        "ptts_c_voice_add_audio": (ci, [vp, cp, fp, ctypes.c_longlong, ci]),
        "ptts_c_voice_export": (ci, [vp, cp, cp]),
        "ptts_c_wav_read": (ci, [cp, fp, ctypes.c_longlong, ctypes.POINTER(ctypes.c_int)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


C_ABI_SYMBOLS = None  # filled lazily by tests from include/ptts_b200.h


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def _ip(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def default_config(**kw) -> B200Config:
    cfg = B200Config()
    lib().b200_default_config(ctypes.byref(cfg))
    for k in ("pdl", "cuda_graphs", "gemm_path", "kv_f32", "overlap", "prefix_share"):          # environment overrides, like ptts_init (host_api.cpp)
        v = os.environ.get("PTTS_B200_" + k.upper())
        if v not in (None, ""):
            setattr(cfg, k, int(v))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, int(v))
    return cfg


class Engine:
    """Thin handle over b200_engine (device layer). Obtained from a Context."""

    def __init__(self, handle):
        self.h = handle
        self.L = lib()

    def voice_create(self, prompt: np.ndarray) -> int:
        prompt = np.ascontiguousarray(prompt.reshape(-1, 1024), np.float32)
        v = self.L.b200_voice_create(self.h, _fp(prompt), prompt.shape[0])
        if v < 0:
            raise RuntimeError(f"b200_voice_create failed: {v}")
        return v

    @property
    def has_encoder(self) -> bool:
        """True when the checkpoint carries the voice-cloning encoder."""
        return self.L.b200_has_encoder(self.h) == 1

    def embed_audio(self, pcm) -> np.ndarray:
        """Mono 24 kHz PCM -> audio_prompt rows [T, 1024] (T = ceil(n / 1920)), encoded on the device."""
        x = np.ascontiguousarray(np.asarray(pcm, np.float32).reshape(-1))
        T = -(-len(x) // FRAME)
        out = np.zeros((max(T, 1), 1024), np.float32)
        rc = self.L.b200_voice_embed_audio(self.h, _fp(x) if len(x) else None, len(x), _fp(out))
        if rc < 0:
            raise RuntimeError(f"b200_voice_embed_audio failed: {rc}")
        return out[:rc]

    def debug_window_attention(self, q, k, v) -> np.ndarray:
        """The encoder's window attention alone over q, k, v [R, 512] (rotated q / k); returns the bf16 output as f32 [R, 512]."""
        q, k, v = (np.ascontiguousarray(np.asarray(t, np.float32).reshape(-1, 512)) for t in (q, k, v))
        out = np.zeros_like(q)
        rc = self.L.b200_debug_window_attention(self.h, q.shape[0], _fp(q), _fp(k), _fp(v), _fp(out))
        if rc != 0:
            raise RuntimeError(f"b200_debug_window_attention failed: {rc}")
        return out

    def voice_from_audio(self, pcm) -> int:
        """Clones a voice from mono 24 kHz PCM: encode + prefill on the device; returns the voice id."""
        x = np.ascontiguousarray(np.asarray(pcm, np.float32).reshape(-1))
        v = self.L.b200_voice_create_from_audio(self.h, _fp(x) if len(x) else None, len(x))
        if v < 0:
            raise RuntimeError(f"b200_voice_create_from_audio failed: {v}")
        return v

    def begin_sentence(self, slot, voice, tokens, max_gen_len, frames_after_eos, temp=0.0):
        t = np.ascontiguousarray(tokens, np.int32)
        rc = self.L.b200_begin_sentence(self.h, slot, voice, _ip(t), len(t), max_gen_len, frames_after_eos, float(temp))
        if rc != 0:
            raise RuntimeError(f"b200_begin_sentence failed: {rc}")

    def begin_sentences(self, slots, voices, token_lists, max_gen_len, frames_after_eos, temps, rng_streams=None):
        n = len(slots)
        off = np.zeros(n + 1, np.int32)
        off[1:] = np.cumsum([len(t) for t in token_lists])
        toks = np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in token_lists]) if n else np.zeros(0, np.int32), np.int32)
        a = [np.ascontiguousarray(x, np.int32) for x in (slots, voices, max_gen_len, frames_after_eos)]
        tp = np.ascontiguousarray(temps, np.float32)
        if rng_streams is not None:
            rs = np.ascontiguousarray(rng_streams, np.uint32)
            rc = self.L.b200_begin_sentences_ex(self.h, n, _ip(a[0]), _ip(a[1]), _ip(toks), _ip(off), _ip(a[2]), _ip(a[3]), _fp(tp), rs.ctypes.data_as(_U32P))
        else:
            rc = self.L.b200_begin_sentences(self.h, n, _ip(a[0]), _ip(a[1]), _ip(toks), _ip(off), _ip(a[2]), _ip(a[3]), _fp(tp))
        if rc != 0:
            raise RuntimeError(f"b200_begin_sentences failed: {rc}")

    def step(self, slot0, n, noise=None, want_latents=True):
        pcm = np.zeros((n, FRAME), np.float32)
        produced = np.zeros(n, np.int32)
        lat = np.zeros((n, LDIM), np.float32) if want_latents else None
        eos = np.zeros(n, np.float32) if want_latents else None
        nz = None
        if noise is not None:
            nz = np.ascontiguousarray(noise, np.float32).reshape(n, LDIM)
        rc = self.L.b200_step(self.h, slot0, n, _fp(nz) if nz is not None else None, _fp(pcm), _ip(produced),
                              _fp(lat) if lat is not None else None, _fp(eos) if eos is not None else None)
        if rc != 0:
            raise RuntimeError(f"b200_step failed: {rc}")
        return pcm, produced, lat, eos

    def step_into(self, slot0, n, noise, pcm, produced):
        """Zero-allocation variant for the bench's end-to-end leg (host buffers supplied by the caller)."""
        return self.L.b200_step(self.h, slot0, n, _fp(noise) if noise is not None else None, _fp(pcm), _ip(produced), None, None)

    def submit(self, slot0, n, noise=None):
        """Pipelined b200_step: enqueue one frame for slots [slot0, slot0+n) and return at once (at most three frames in flight)."""
        rc = self.L.b200_submit(self.h, slot0, n, _fp(noise) if noise is not None else None)
        if rc != 0:
            raise RuntimeError(f"b200_submit failed: {rc}")

    def collect_into(self, pcm, produced):
        """Blocks until the oldest submitted frame is complete; fills pcm [n][1920] and produced [n]; returns n."""
        rc = self.L.b200_collect(self.h, _fp(pcm), _ip(produced))
        if rc < 0:
            raise RuntimeError(f"b200_collect failed: {rc}")
        return rc

    def steps_enqueue(self, slot0, n, count):
        rc = self.L.b200_steps_enqueue(self.h, slot0, n, count)
        if rc != 0:
            raise RuntimeError(f"b200_steps_enqueue failed: {rc}")

    def step_enqueue(self, slot0, n, injected=False):
        rc = self.L.b200_step_enqueue(self.h, slot0, n, 1 if injected else 0)
        if rc != 0:
            raise RuntimeError(f"b200_step_enqueue failed: {rc}")

    def sync(self):
        self.L.b200_sync(self.h)

    def join(self):
        """Main stream waits for the Mimi stream: an event recorded on stream_handle() afterwards covers every enqueued frame."""
        self.L.b200_join(self.h)

    def mimi_reset(self, slot0, n):
        assert self.L.b200_mimi_reset(self.h, slot0, n) == 0

    def mimi_decode(self, slot0, n, latents):
        lat = np.ascontiguousarray(latents, np.float32).reshape(n, LDIM)
        pcm = np.zeros((n, FRAME), np.float32)
        rc = self.L.b200_mimi_decode(self.h, slot0, n, _fp(lat), _fp(pcm))
        if rc != 0:
            raise RuntimeError(f"b200_mimi_decode failed: {rc}")
        return pcm

    def mimi_decode_enqueue(self, slot0, n):
        assert self.L.b200_mimi_decode_enqueue(self.h, slot0, n) == 0

    def set_seed(self, seed):
        self.L.b200_set_seed(self.h, seed)

    def end_sentences(self, slots):
        """b200_end_sentences: the slots' sentences end before the next enqueued step (stream-ordered)."""
        a = np.ascontiguousarray(slots, np.int32)
        rc = self.L.b200_end_sentences(self.h, len(a), _ip(a))
        if rc != 0:
            raise RuntimeError(f"b200_end_sentences failed: {rc}")

    def slot_position(self, slot):
        return self.L.b200_slot_position(self.h, slot)

    def debug_set_position(self, slot0, n, pos, max_gen_len):
        rc = self.L.b200_debug_set_position(self.h, slot0, n, pos, max_gen_len)
        if rc != 0:
            raise RuntimeError(f"b200_debug_set_position failed: {rc}")

    def debug_gemm(self, A, W, T, taps, f16=False, bias=None, path=0, want_out2=False):
        """A [n_slots][rows_buf][C], W [N][taps*C] -> (out [n_slots*T][N] f32, out2 or None, used_tensor_cores)."""
        A = np.ascontiguousarray(A, np.float32); W = np.ascontiguousarray(W, np.float32)
        n_slots, rows_buf, C = A.shape
        N = W.shape[0]
        assert W.shape[1] == taps * C
        out = np.zeros((n_slots * T, N), np.float32)
        out2 = np.zeros((n_slots * T, N), np.float32) if want_out2 else None
        b = None if bias is None else np.ascontiguousarray(bias, np.float32)
        rc = self.L.b200_debug_gemm(self.h, 1 if f16 else 0, _fp(A), n_slots, rows_buf, C, T, taps, _fp(W), N, _fp(b) if b is not None else None,
                                    path, _fp(out), _fp(out2) if out2 is not None else None)
        if rc < 0:
            raise RuntimeError(f"b200_debug_gemm failed: {rc}")
        return out, out2, bool(rc)

    def debug_set_latent(self, slot0, n, latents):
        lat = np.ascontiguousarray(latents, np.float32).reshape(n, LDIM)
        assert self.L.b200_debug_set_latent(self.h, slot0, n, _fp(lat)) == 0

    def profile(self, on=True):
        self.L.b200_profile(self.h, 1 if on else 0)

    def profile_read(self):
        ms = np.zeros(7, np.float32); cnt = np.zeros(7, np.int32)
        self.L.b200_profile_read(self.h, _fp(ms), _ip(cnt))
        names = ["attn_stream", "flow_backbone", "head", "mimi_transformer", "seanet", "step", "attn_prefix_tiles"]
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(names)}

    def stream_handle(self):
        return self.L.b200_stream(self.h)

    def launch_count(self):
        return self.L.b200_launch_count(self.h)

    def debug_taps(self, on=True):
        assert self.L.b200_debug_taps(self.h, 1 if on else 0) == 0

    def debug_tap(self, name, slot):
        n = self.L.b200_debug_tap(self.h, name.encode(), slot, None, 0)
        if n < 0:
            raise RuntimeError(f"b200_debug_tap({name}) failed: {n}")
        out = np.zeros(n, np.float32)
        assert self.L.b200_debug_tap(self.h, name.encode(), slot, _fp(out), n) == n
        return out

    def debug_read(self, name, offset, n):
        out = np.zeros(n, np.float32)
        rc = self.L.b200_debug_read_f32(self.h, name.encode(), offset, _fp(out), n)
        if rc != 0:
            raise RuntimeError(f"b200_debug_read_f32({name}) failed: {rc}")
        return out

    def read_kv(self, slot, layer, which, n_pos):
        out = np.zeros((n_pos, 1024), np.float32)
        assert self.L.b200_read_kv(self.h, slot, layer, which, n_pos, _fp(out)) == 0
        return out

    def debug_write_kv(self, slot, layer, which, pos0, rows):
        rows = np.ascontiguousarray(rows, np.float32).reshape(-1, 1024)
        rc = self.L.b200_debug_write_kv(self.h, slot, layer, which, pos0, rows.shape[0], _fp(rows))
        if rc != 0:
            raise RuntimeError(f"b200_debug_write_kv failed: {rc}")

    def debug_set_prefix(self, slot, pfx_slot, pfx_len):
        rc = self.L.b200_debug_set_prefix(self.h, slot, pfx_slot, pfx_len)
        if rc != 0:
            raise RuntimeError(f"b200_debug_set_prefix failed: {rc}")

    def debug_attention(self, layer, q, rows_pos, slot0=0, rows_slot=None, prefill=False, **opts):
        """One layer's attention dispatch over q [n][1024]; returns (out [n][1024] f32, tile work items)."""
        q = np.ascontiguousarray(q, np.float32).reshape(-1, 1024)
        n = q.shape[0]
        pos = np.ascontiguousarray(rows_pos, np.int32)
        rs = None if rows_slot is None else np.ascontiguousarray(rows_slot, np.int32)
        assert pos.shape == (n,) and (rs is None or rs.shape == (n,))
        out = np.zeros((n, 1024), np.float32)
        o = AttnOpts(**opts)
        rc = self.L.b200_debug_attention(self.h, layer, 1 if prefill else 0, slot0, n, _ip(rs) if rs is not None else None, _ip(pos), _fp(q),
                                         ctypes.byref(o), _fp(out))
        if rc < 0:
            raise RuntimeError(f"b200_debug_attention failed: {rc}")
        return out, rc


def attn_plan(prefill, pfx_slot, pfx_len, row_slot=None, row_pos=None, num_sms=148, chunk_rows=4096, max_voices=8):
    """Host-only work lists of the FlowLM attention (b200_debug_attn_plan): (return value, items [k][9], aux)."""
    ps = np.ascontiguousarray(pfx_slot, np.int32); pl = np.ascontiguousarray(pfx_len, np.int32)
    rs = None if row_slot is None else np.ascontiguousarray(row_slot, np.int32)
    rp = None if row_pos is None else np.ascontiguousarray(row_pos, np.int32)
    n = len(rs) if prefill else len(ps)
    nk = ctypes.c_int()
    cap = 64
    while True:
        items = np.zeros((cap, 9), np.int32)
        aux = np.zeros(n + 2, np.int32)
        rc = lib().b200_debug_attn_plan(1 if prefill else 0, n, _ip(rs) if rs is not None else None, _ip(rp) if rp is not None else None,
                                        _ip(ps), _ip(pl), num_sms, chunk_rows, max_voices, _ip(items), cap, _ip(aux), ctypes.byref(nk))
        if nk.value <= cap:
            break
        cap = nk.value
    return rc, items[:nk.value], (aux[:rc + 1] if prefill and rc >= 0 else aux[:n])


class Context:
    """ptts_context_t (reference ptts_init, src/pocket_tts.cpp:273-322)."""

    def __init__(self, model_path: str, **cfg):
        L = lib()
        if not model_path.endswith("/"):
            model_path += "/"
        self.model_path = model_path
        c = default_config(**cfg)
        self.cfg = c
        self.h = L.ptts_c_init_ex(model_path.encode(), ctypes.byref(c))
        if not self.h:
            raise RuntimeError("ptts_init failed")
        self.engine = Engine(L.ptts_c_engine(self.h))

    def close(self):
        """Frees the engine (device memory) and the context. Streams / batches of this context must not be used afterwards."""
        if self.h:
            lib().ptts_c_destroy(self.h)
            self.h = None; self.engine = None

    @property
    def sample_rate(self):
        return lib().ptts_c_get_sample_rate(self.h)

    @property
    def frame_size(self):
        return lib().ptts_c_get_frame_size(self.h)

    def tokenize(self, text: str):
        buf = (ctypes.c_int32 * 8192)()
        n = lib().ptts_c_tokenize(self.h, text.encode(), buf, 8192)
        return list(buf[:n])

    def stream(self, voice="cosette", temp=0.7) -> "Stream":
        return Stream(self, voice, temp)

    def add_voice(self, name: str, pcm, sample_rate: int = SAMPLE_RATE) -> int:
        """Clones a voice from mono PCM (24 kHz only) and registers it under `name`; returns the engine voice id."""
        x = np.ascontiguousarray(np.asarray(pcm, np.float32).reshape(-1))
        v = lib().ptts_c_voice_add_audio(self.h, name.encode(), _fp(x) if len(x) else None, len(x), int(sample_rate))
        if v < 0:
            raise RuntimeError(f"ptts_c_voice_add_audio failed: {v}")
        return v

    def export_voice(self, name: str, path: str):
        """Writes a cloned voice as an audio_prompt [1, T, 1024] F32 safetensors voice file."""
        rc = lib().ptts_c_voice_export(self.h, name.encode(), path.encode())
        if rc != 0:
            raise RuntimeError(f"ptts_c_voice_export failed: {rc}")


class Batch:
    """Continuous batching over the engine's slots (ptts_c_batch_*): queue utterances, run() generates all of them, finished slots are
    refilled with queued sentences. For online serving, add() at any time, pump() a few steps, pop() each utterance's ready frames in order
    and cancel() the ones nobody waits for. With `ops` = (begin, submit, collect[, end]) Python callables the scheduler runs over a mock
    engine (CPU tests)."""

    STATES = ("queued", "running", "done", "cancelled")

    def __init__(self, ctx: "Context" = None, n_slots: int = 0, ops=None, frame_size: int = FRAME):
        L = lib()
        self.frame_size, self.ctx = frame_size, ctx
        if ops is not None:
            end = BATCH_END_FN(ops[3]) if len(ops) > 3 and ops[3] is not None else BATCH_END_FN()
            self._cbs = (BATCH_BEGIN_FN(ops[0]), BATCH_SUBMIT_FN(ops[1]), BATCH_COLLECT_FN(ops[2]), end)   # keep the thunks alive
            self.h = L.ptts_c_batch_create_with_ops_ex(None, *self._cbs, n_slots, frame_size)
        else:
            self.h = L.ptts_c_batch_create(ctx.h, n_slots)
        if not self.h:
            raise RuntimeError("ptts_c_batch_create failed")

    def configure(self, refill_min=0, refill_every=0, range_quantum=0, keep_pcm=-1):
        assert lib().ptts_c_batch_configure(self.h, refill_min, refill_every, range_quantum, keep_pcm) == 0

    def add(self, voice: str, text: str, temp: float = 0.7) -> int:
        u = lib().ptts_c_batch_add(self.h, voice.encode(), text.encode(), float(temp))
        if u < 0:
            raise RuntimeError(f"ptts_c_batch_add failed: {u}")
        return u

    def add_tokens(self, voice_id, ids, max_gen_len, frames_after_eos, temp=0.7, rng_stream=0, utt=None) -> int:
        """One sentence given as token ids: a new utterance, or the next sentence of utterance `utt`."""
        a = np.ascontiguousarray(ids, np.int32)
        if utt is None:
            u = lib().ptts_c_batch_add_tokens(self.h, voice_id, _ip(a), len(a), max_gen_len, frames_after_eos, float(temp), rng_stream)
        else:
            u = lib().ptts_c_batch_append_tokens(self.h, utt, voice_id, _ip(a), len(a), max_gen_len, frames_after_eos, float(temp), rng_stream)
        if u < 0:
            raise RuntimeError(f"ptts_c_batch_add_tokens failed: {u}")
        return u

    def run(self) -> int:
        n = lib().ptts_c_batch_run(self.h)
        if n < 0:
            raise RuntimeError(f"ptts_c_batch_run failed: {n}")
        return n

    def pump(self, max_steps: int = 1) -> int:
        """Runs the scheduler for at least max_steps collected steps (and one produced frame); returns the frames produced, 0 when idle."""
        n = lib().ptts_c_batch_pump(self.h, max_steps)
        if n < 0:
            raise RuntimeError(f"ptts_c_batch_pump failed: {n}")
        return n

    def status(self, utt):
        """(state, ready frames): state is one of Batch.STATES."""
        ready = ctypes.c_int()
        st = lib().ptts_c_batch_status(self.h, utt, ctypes.byref(ready))
        if st < 0:
            raise RuntimeError(f"ptts_c_batch_status failed: {st}")
        return self.STATES[st], ready.value

    def pop(self, utt) -> np.ndarray:
        """The utterance's frames that are ready and were not popped before, [n, frame_size], in order."""
        n = self.status(utt)[1]
        out = np.zeros((max(n, 1), self.frame_size), np.float32)
        got = lib().ptts_c_batch_pop(self.h, utt, _fp(out), n)
        if got < 0:
            raise RuntimeError(f"ptts_c_batch_pop failed: {got}")
        return out[:got]

    def cancel(self, utt):
        rc = lib().ptts_c_batch_cancel(self.h, utt)
        if rc != 0:
            raise RuntimeError(f"ptts_c_batch_cancel failed: {rc}")

    def frames(self, utt) -> int:
        return lib().ptts_c_batch_frames(self.h, utt)

    def read(self, utt) -> np.ndarray:
        n = self.frames(utt)
        out = np.zeros((max(n, 1), self.frame_size), np.float32)
        got = lib().ptts_c_batch_read(self.h, utt, _fp(out), n)
        return out[:got]

    def stats(self) -> dict:
        st = BatchStats()
        lib().ptts_c_batch_stats(self.h, ctypes.byref(st))
        d = {k: getattr(st, k) for k, _ in BatchStats._fields_}
        d["idle_slot_fraction"] = 1.0 - d["frames"] / d["slot_steps"] if d["slot_steps"] else 0.0
        return d

    def __del__(self):
        try:
            # destroy collects the steps still in flight on the engine: not possible once the context (and its engine) was closed
            if self.ctx is None or self.ctx.h is not None:
                lib().ptts_c_batch_destroy(self.h)
        except Exception:
            pass


class Stream:
    """ptts_stream_t: send text in arbitrary chunks, receive 1920-sample frames (reference src/pocket_tts.cpp:351-519)."""

    def __init__(self, ctx: Context, voice: str, temp: float):
        self.ctx = ctx
        self.h = lib().ptts_c_stream_from_safetensors(ctx.h, voice.encode(), float(temp))
        self.slot = lib().ptts_c_slot(self.h)
        self.voice = lib().ptts_c_voice(self.h)

    def reset(self):
        lib().ptts_c_stream_reset(self.h)

    def send(self, chunk: str):
        lib().ptts_c_stream_send(self.h, chunk.encode() if isinstance(chunk, str) else chunk)

    def flush(self):
        lib().ptts_c_stream_flush(self.h)

    def receive(self):
        buf = np.zeros(FRAME, np.float32)
        ok = lib().ptts_c_stream_receive(self.h, _fp(buf))
        return buf if ok else None

    def pending(self):
        n = lib().ptts_c_stream_pending(self.h, -1, None, 0)
        out = []
        for i in range(n):
            b = ctypes.create_string_buffer(65536)
            lib().ptts_c_stream_pending(self.h, i, b, 65536)
            out.append(b.value)
        return out


def read_wav(path: str):
    """Host-only RIFF reader of the engine (PCM16 / float32, mixed down to mono): (samples float32 [n], sample_rate)."""
    rate = ctypes.c_int()
    n = lib().ptts_c_wav_read(path.encode(), None, 0, ctypes.byref(rate))
    if n < 0:
        raise ValueError(f"{path}: not a readable PCM16 / float32 WAV file")
    out = np.zeros(max(n, 1), np.float32)
    lib().ptts_c_wav_read(path.encode(), _fp(out), n, ctypes.byref(rate))
    return out[:n], rate.value


def set_seed(seed: int):
    lib().ptts_c_set_seed(seed)


def get_seed() -> int:
    return lib().ptts_c_get_seed()


class TextFrontEnd:
    """Host-only tokenizer + sentence splitter (no GPU): the C++ restatement of conditioners/text.h used by the engine."""

    def __init__(self, tokenizer_model: str):
        self.h = lib().ptts_c_text_create(tokenizer_model.encode())
        if not self.h:
            raise RuntimeError(f"cannot load {tokenizer_model}")

    def encode(self, text):
        buf = (ctypes.c_int32 * 16384)()
        n = lib().ptts_c_text_encode(self.h, text.encode() if isinstance(text, str) else text, buf, 16384)
        return list(buf[:n])

    def send(self, chunk):
        lib().ptts_c_text_send(self.h, chunk.encode() if isinstance(chunk, str) else chunk)

    def flush(self):
        lib().ptts_c_text_flush(self.h)

    def reset(self):
        lib().ptts_c_text_reset(self.h)

    def pop_all(self):
        out = []
        while True:
            b = ctypes.create_string_buffer(1 << 16)
            n = lib().ptts_c_text_pop(self.h, b, 1 << 16)
            if n < 0:
                return out
            out.append(b.raw[:n])
